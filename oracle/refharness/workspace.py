"""TEST-ONLY: build the working directory the reference needs in order to be imported unmodified
(SURVEY.md section 8c): ``Control_Toolkit -> $CTK_REFERENCE`` symlink, a ``Control_Toolkit_ASF`` with working
``config_*.yml`` (the reference reads them relative to CWD at import time) and the CartPole cost plugins,
with the SI_Toolkit / tensorflow / watchdog shims on ``sys.path``.  Only usable where CTK_REFERENCE names a checkout of the
original Control_Toolkit; the repository does not contain one, so the cross-checks against it skip without it."""
import os
import shutil
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REFERENCE = os.environ.get("CTK_REFERENCE", "")


def reference_has(*parts: str) -> bool:
    """True when CTK_REFERENCE is set and the checkout it names contains ``parts`` (a file or directory below its root)."""
    return bool(REFERENCE) and os.path.exists(os.path.join(REFERENCE, *parts))


def reference_available() -> bool:
    return reference_has("Optimizers")


def enter_workspace() -> str:
    """Create the workspace, chdir into it, extend sys.path.  Returns the workspace path."""
    if not reference_available():
        raise RuntimeError(f"reference not found at {REFERENCE}")
    ws = tempfile.mkdtemp(prefix="ctk_ref_ws_")
    os.symlink(REFERENCE, os.path.join(ws, "Control_Toolkit"))
    shutil.copytree(os.path.join(HERE, "asf", "Control_Toolkit_ASF"), os.path.join(ws, "Control_Toolkit_ASF"))
    os.chdir(ws)
    for p in (REPO, HERE, ws):
        if p not in sys.path:
            sys.path.insert(0, p)
    return ws
