"""CPU test of the drop-in claim ("nothing in the reference has to be modified", INTEGRATION.md section 2): the reference's own
UNMODIFIED controller_mpc discovers, constructs and configures the B200 plugins through the shim files of integration/ and gets all
the way to ``ctk_create`` -- which, on a box without a GPU, is the first thing that can fail (BackendUnavailable: no CPU fallback).
Needs a checkout of the original Control_Toolkit named by CTK_REFERENCE and skips without one; tests/test_gpu_parity.py drives the
same plugins through the repo's controller_mpc mirror.  Reference: Controllers/controller_mpc.py:56-89, others/globals_and_utils.py:103-133."""
import json
import os
import subprocess
import sys

import pytest

from oracle.refharness.workspace import reference_available

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.skipif(not reference_available(), reason="needs a Control_Toolkit checkout: set CTK_REFERENCE to its path")
def test_reference_controller_mpc_reaches_ctk_create_through_the_shims():
    r = subprocess.run([sys.executable, os.path.join(HERE, "dropin", "drive_reference_controller.py")], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("DROPIN_RESULT ")]
    assert line, r.stdout[-2000:]
    res = json.loads(line[-1][len("DROPIN_RESULT "):])
    expect = {"mppi-b200": ("optimizer_mppi_b200", 2000, 50), "cem-tf-b200": ("optimizer_cem_tf_b200", 4096, 50), "rpgd-b200": ("optimizer_rpgd_b200", 32, 50),
              "random-action-tf-b200": ("optimizer_random_action_tf_b200", 512, None), "gradient-tf-b200": ("optimizer_gradient_tf_b200", 40, None),
              "cem-naive-grad-tf-b200": ("optimizer_cem_naive_grad_tf_b200", 200, None),
              "cem-grad-bharadhwaj-tf-b200": ("optimizer_cem_grad_bharadhwaj_tf_b200", 32, None)}
    assert [x["optimizer"] for x in res] == list(expect)  # every shim of integration/ (all seven optimizers served)
    for x in res:
        cls, n, h = expect[x["optimizer"]]
        assert x["class"] == cls and x["module_file"] == os.path.join("Control_Toolkit_ASF", "Optimizers", cls + ".py")
        assert x["bases"][0].startswith("control_toolkit_b200.Optimizers.")       # the plugin class of this repo ...
        assert x["predictor_is_reference_wrapper"] and x["cost_is_reference_wrapper"]  # ... fed the reference's OWN wrapper objects
        assert (x["num_rollouts"], x["mpc_horizon"]) == (x["yaml_num_rollouts"], x["yaml_mpc_horizon"])  # the YAML block arrived through **config_optimizer
        assert x["num_rollouts"] == n and (h is None or x["mpc_horizon"] == h)
        assert (x["num_states"], x["num_control_inputs"]) == (6, 1)                # from the reference's PredictorWrapper
        if x["outcome"] == "backend_unavailable":  # no GPU here: ctk_create itself refused -- every layer above it has run
            assert "CUDA" in x["error"] or "cuda" in x["error"], x["error"]
        else:
            assert x["outcome"] == "configured" and len(x["u"]) == 1 and -1.0 <= x["u"][0] <= 1.0
