"""CPU test of K1's step source at both lane widths (tests/host_twin/lanes.cpp, compiled with g++): two rollouts advanced as one f2
roll -- the way K1 runs two rollouts per thread -- end with the same bits as the same rollouts advanced one float roll at a time,
for both cost kinds.  On the device each f2 operation is one packed instruction with the same per-lane rounding; here it is two
scalar operations, so this pins the other half of the contract: the generic step routes every lane through the same operations in
the same order, and lane q of a pair is rollout q."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import spec
from test_host_twin import _fp, _params

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def lanes(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("lanes") / "libctk_host_lanes.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", os.path.join(HERE, "host_twin", "lanes.cpp"), "-o", out],
                   check=True)
    return C.CDLL(out)


@pytest.mark.parametrize("cost_name", ["default", "quadratic_boundary_grad"])
def test_pair_lanes_equal_float_lanes_bit_for_bit(lanes, cost_name):
    N, H = 64, 100
    rng = np.random.default_rng(17)
    for s0 in spec.synthetic_states(4, seed=19):
        dU = (rng.standard_normal((N, H)) * 0.3).astype(np.float32)
        U = np.clip(rng.uniform(-0.5, 0.5, (1, H)).astype(np.float32) + dU, -1, 1).astype(np.float32)
        ode, cost = _params(cost_name)
        S = {w: np.full(N, np.nan, np.float32) for w in ("float", "pair")}
        st = {w: np.full((N, 7), np.nan, np.float32) for w in ("float", "pair")}
        lanes.twin_lanes(_fp(s0), _fp(U), _fp(dU), N, H, C.byref(ode), C.byref(cost), C.c_float(0.3), _fp(S["float"]), _fp(S["pair"]),
                         _fp(st["float"]), _fp(st["pair"]))
        assert np.isfinite(S["float"]).all() and np.isfinite(st["float"]).all()
        assert len(np.unique(S["float"])) == N  # every rollout (every lane) differs from every other
        np.testing.assert_array_equal(S["pair"], S["float"])
        np.testing.assert_array_equal(st["pair"], st["float"])
