"""-m gpu: K1 at both lane widths computes the same per-rollout costs, bit for bit.

With two rollouts per thread (CTK_K1_ILP=2) K1 advances them as one f2 roll: every add, multiply and fma of the step is one packed
FADD2 / FMUL2 / FFMA2 that computes per lane exactly what the scalar instruction computes (ctk_ode_scaled.cuh).  With one rollout per
thread (CTK_K1_ILP=1) the same source runs on float.  The Philox draws of a rollout depend on its global index only, so two handles
with the same configuration and state sample the same perturbations whatever their launch geometry: their per-rollout costs J must be
EQUAL element for element.  u and u_nom go through the per-thread online softmin, whose grouping of rollouts follows the geometry, so
they agree to rounding only (the usual 1e-5).
"""
import numpy as np
import pytest

from gpu_helpers import make_controller, max_rel
from helpers import load_golden

pytestmark = pytest.mark.gpu

N = 200_000  # above one wave of single-rollout threads (148 SMs x 1024), so ILP = 2 is a production choice here too


@pytest.mark.parametrize("cost,kind", [("default", 0), ("quadratic_boundary_grad", 1)])
def test_k1_float_and_pair_lanes_give_identical_costs(monkeypatch, cost, kind):
    from control_toolkit_b200 import _lib as L
    from oracle import spec
    _, meta = load_golden("mppi_h100_n256")
    meta = dict(meta, cost=cost, cfg=dict(meta["cfg"], num_rollouts=N, mpc_horizon=100, period_interpolation_inducing_points=10))
    ctrls = {}
    for ilp in (1, 2):
        monkeypatch.setenv("CTK_K1_ILP", str(ilp))
        ctrls[ilp] = make_controller(meta, rng=None, logging=False)
    s = spec.synthetic_states(1, seed=57)[0]
    out = {}
    for ilp, ctrl in ctrls.items():
        u = ctrl.step(s)
        opt = ctrl.optimizer
        out[ilp] = (float(np.ravel(u)[0]), np.array(opt._get_log(L.LOG_J, (N,))), np.array(opt.u_nom, np.float32), opt.last_kernel)
    assert out[1][3] == f"mppi_ode_kernel<{kind},0,10,1,1024,0>", out[1][3]
    assert out[2][3] == f"mppi_ode_kernel<{kind},0,10,2,896,0>", out[2][3]
    J1, J2 = out[1][1], out[2][1]
    assert np.isfinite(J1).all()
    np.testing.assert_array_equal(J2, J1)
    scale = max(float(np.abs(out[1][2]).max()), 1e-2)
    assert abs(out[2][0] - out[1][0]) <= 1e-5 * scale, (out[1][0], out[2][0])
    assert max_rel(out[2][2], out[1][2], floor=1e-2) <= 1e-5
