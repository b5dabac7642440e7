"""CPU checks of the SHIPPED library's machine code (cuobjdump; no GPU): K1's two-rollouts-per-thread instantiations advance a thread's
rollouts as packed FP32 pairs (the f2 lanes of ctk_ode_scaled.cuh).  K1 is issue-bound, and FFMA2 / FMUL2 / FADD2 issue once for two
lanes, so the paired segment takes about 28 issue slots per rollout-step where the scalar one took 50 (DESIGN.md section 5.1).  A source
change that splits the pairs again loses that without changing a single result, which is why it is pinned here."""
import collections
import re

import pytest

from test_static_sass import _mnemonics, _sass, pytestmark  # noqa: F401  (same skip condition: the built library and cuobjdump)


def _kernel(kind, ilp):
    maxt = 896 if ilp == 2 else 1024
    return f"_ZN3ctk15mppi_ode_kernelILi{kind}ELb0ELi10ELi{ilp}ELi{maxt}ELb0EEEvNS_11MppiOdeArgsE"


def _unrolled_segment(sass):
    """Mnemonics of the largest basic block: the fully unrolled ten-step segment of the PERIOD = 10 instantiations."""
    lines = [(int(m.group(1), 16), ln) for m, ln in ((re.match(r"\s+/\*([0-9a-f]{4,})\*/", ln), ln) for ln in sass.splitlines()) if m]
    targets = {int(t, 16) for _, ln in lines for t in re.findall(r"\b(?:BRA|BSSY|CALL)\S*\s+(?:!?U?P\d+,\s*)?(?:B\d+,\s*)?0x([0-9a-f]+)", ln)}
    blocks, cur = [], []
    for addr, ln in lines:
        if addr in targets:
            blocks.append(cur)
            cur = []
        op = _mnemonics(ln)[0]
        cur.append(op)
        if op in ("BRA", "EXIT", "CALL", "RET", "BSSY", "BSYNC", "WARPSYNC"):
            blocks.append(cur)
            cur = []
    blocks.append(cur)
    return max(blocks, key=len)


@pytest.mark.parametrize("kind", [0, 1])
def test_k1_two_rollouts_per_thread_run_as_packed_pairs(kind):
    pair = collections.Counter(_unrolled_segment(_sass(_kernel(kind, 2))))
    single = collections.Counter(_unrolled_segment(_sass(_kernel(kind, 1))))
    assert pair["FRND"] == 20 and single["FRND"] == 10, (pair, single)  # (one wrap per step and lane: ten steps, two / one lanes)
    # Every FP32 add, multiply and fma of the step is paired: no scalar one is left in the segment.  What stays per lane has no
    # packed form: the clamps of u and the barrier's max(., 0) (FMNMX), the wrap's rint (FRND), 1/A (MUFU.RCP) and, for the
    # boundary-gradient cost, the border indicator (FSETP + FSEL).
    assert pair["FFMA"] + pair["FMUL"] + pair["FADD"] == 0, pair
    # The same operations as the one-rollout-per-thread segment, two lanes at a time: an fmul + fadd that ptxas contracted into one
    # FFMA in the scalar build (or the reverse) would show up here as a different mix -- and as different bits.
    assert (pair["FFMA2"], pair["FMUL2"], pair["FADD2"]) == (single["FFMA"], single["FMUL"], single["FADD"]), (pair, single)
    assert pair["FMNMX"] == 2 * single["FMNMX"] and pair["MUFU"] == 2 * single["MUFU"], (pair, single)
    # issue slots per rollout-step (two rollouts x ten steps); the scalar pair segment took 50.2
    assert sum(pair.values()) <= 20 * 33, sum(pair.values())
    assert pair["LDL"] + pair["STL"] + pair["MOV"] == 0, pair  # no spill, no moves that build pairs
