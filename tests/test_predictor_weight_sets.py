"""Weight sets for the network-predictor tests (tests/test_gpu_predictors.py), and the CPU proof that they can catch what the
default weights cannot.

The default MLP (``random_init``) has zero biases and never saturates: every bias read of the five MLP engines is multiplied by
zero and layer-2 pre-activations stay below ~2.6.  The sets here are built once from a seed as numpy arrays; the SAME arrays
become the product's ``MLPSpec`` / ``GRUSpec`` and the oracle's ``MLPWeights`` / ``GRUWeights``.

* ``biased``: the fixture network (seed 2, width 128) plus per-unit biases b1, b2 ~ N(0, 0.3^2), b3 ~ N(0, 0.05^2); the position
  read-out (column 3 of W3 and b3[3]) is scaled by 0.08 as in ``GRUWeights.random_init``, so that rollouts stay on the track.
* ``saturating``: ``biased`` with W1 and W2 scaled by 4 (tanh saturates, the kernels' tanh clamps run).
* ``w16`` / ``w48`` / ``w112``: ``biased`` at the other hidden widths the FP32-pipe engine accepts.
* GRU widths 8 / 16 / 24 (32 is the fixtures' width): ``random_init``, which already draws non-zero biases.

This file checks, in float64 on the oracle only, that each bias mutation moves the one-step output by at least 100 x the bound the
GPU one-step test asserts (for the reduced-precision engines: their median bound), that the saturating set reaches saturation, and
that product and oracle weights are the same numbers.
"""
import functools
import math

import numpy as np
import pytest
import torch

from oracle import spec

MLP_SETS = {"biased": (128, 1.0), "saturating": (128, 4.0), "w16": (16, 1.0), "w48": (48, 1.0), "w112": (112, 1.0)}
GRU_WIDTHS = (8, 16, 24)
MLP_SEED, GRU_SEED = 2, 3

# One-step residual bounds of tests/test_gpu_predictors.py: max over rollouts, steps and outputs of |device - float64| / (1 + |y|),
# per engine for (the ordinary sets, the saturating set).  Each is >= 3 x the largest value measured on a B200 (power limit 1000 W)
# over every case of that file: simt 5.1e-6 / 5.0e-5, tcgen05 1.0e-5 / 1.4e-4 (saturated pre-activations reach |a| ~ 60, whose fp32
# rounding the outputs carry), tcgen05_bf16 2.9e-3 / 8.8e-3, tcgen05_fast 1.1e-2 / 2.1e-2, GRU 8.6e-6.  The reduced-precision
# engines' maxima are isolated rows where an fp32 ulp of h1 flips a bf16 rounding (bf16) or MUFU tanh errs (fast); their MEDIAN is
# bounded tightly as well (measured 1.4e-7 / 2.2e-6), and that is the bound a bias bug, which moves every row, runs into.
ONE_STEP_BOUND = {"simt": (2e-5, 1.5e-4), "tcgen05": (4e-5, 5e-4), "tcgen05_bf16": (1e-2, 3e-2), "tcgen05_fast": (4e-2, 7e-2)}
ONE_STEP_MEDIAN_BOUND = {"tcgen05_bf16": 5e-7, "tcgen05_fast": 7e-6}
GRU_ONE_STEP_BOUND = 3e-5
TEETH = 100.0  # every bias mutation moves the output by at least this many bounds


def one_step_bound(engine, set_name):
    return ONE_STEP_BOUND[engine][1 if set_name == "saturating" else 0]


@functools.lru_cache(maxsize=None)
def mlp_arrays(name):
    """{W1, b1, W2, b2, W3, b3} float32 of weight set ``name``."""
    hid, gain = MLP_SETS[name]
    base = spec.MLPWeights.random_init(MLP_SEED, hidden=hid)
    rng = np.random.default_rng(1000 + hid)
    b1 = (0.3 * rng.standard_normal(hid)).astype(np.float32)
    b2 = (0.3 * rng.standard_normal(hid)).astype(np.float32)
    b3 = (0.05 * rng.standard_normal(5)).astype(np.float32)
    W3 = base.W3.copy()
    W3[:, 3] *= np.float32(0.08)
    b3[3] *= np.float32(0.08)
    a = dict(W1=(base.W1 * np.float32(gain)).astype(np.float32), b1=b1, W2=(base.W2 * np.float32(gain)).astype(np.float32), b2=b2,
             W3=W3, b3=b3)
    for v in a.values():
        v.flags.writeable = False
    return a


@functools.lru_cache(maxsize=None)
def gru_arrays(hidden):
    g = spec.GRUWeights.random_init(GRU_SEED, hidden=hidden)
    return {k: getattr(g, k) for k in ("Wi1", "Wh1", "bi1", "bh1", "Wi2", "Wh2", "bi2", "bh2", "W3", "b3")}


def mlp_spec(name):
    import control_toolkit_b200 as ctk
    return ctk.MLPSpec(**{k: v.copy() for k, v in mlp_arrays(name).items()})


def mlp_weights(name, **over):
    a = {k: v.copy() for k, v in mlp_arrays(name).items()}
    a.update(over)
    return spec.MLPWeights(**a)


def gru_spec(hidden):
    import control_toolkit_b200 as ctk
    return ctk.GRUSpec(**{k: v.copy() for k, v in gru_arrays(hidden).items()})


def gru_weights(hidden):
    return spec.GRUWeights(**{k: v.copy() for k, v in gru_arrays(hidden).items()})


def predictor_name(name):
    """Registry name of a weight set: not 'Dense...' / 'GRU...', which gpu_helpers.make_controller reserves for the fixtures'
    random_init networks."""
    return f"TestNet-{name}"


def one_step_residual(y_dev, y_ref):
    """[..., 6] -> [...]: max over the six outputs of |dev - ref| / (1 + |ref|), the angle compared modulo 2 pi."""
    d = np.asarray(y_dev, np.float64) - np.asarray(y_ref, np.float64)
    d[..., 0] = np.remainder(d[..., 0] + math.pi, 2 * math.pi) - math.pi
    return np.max(np.abs(d) / (1.0 + np.abs(np.asarray(y_ref, np.float64))), axis=-1)


def sample_pairs(name, n=512, H=30, seed=7):
    """(s [n*H, 6], Q [n*H, 1]) float64: the GPU tests' initial states (synthetic_states(., seed=31)) rolled out through the float64
    network of set ``name`` under uniform controls in [-1, 1] -- the kind of (state, control) pairs the device logs."""
    pred = spec.MLPPredictor(mlp_weights(name), dtype=torch.float64)
    s0 = spec.synthetic_states(4, seed=31)
    rng = np.random.default_rng(seed)
    s = torch.from_numpy(np.repeat(s0, n // 4, axis=0)).double()
    Q = torch.from_numpy(rng.uniform(-1.0, 1.0, (s.shape[0], H, 1)))
    traj = pred.predict_core(s, Q)
    return traj[:, :-1].reshape(-1, 6), Q.reshape(-1, 1)


MUTANTS = {
    "drop_b1": lambda w: dict(b1=np.zeros_like(w["b1"])),
    "drop_b2": lambda w: dict(b2=np.zeros_like(w["b2"])),
    "drop_b3": lambda w: dict(b3=np.zeros_like(w["b3"])),
    "roll_b2": lambda w: dict(b2=np.roll(w["b2"], 1)),
}


@pytest.mark.parametrize("name", sorted(MLP_SETS))
@pytest.mark.parametrize("mutant", sorted(MUTANTS))
def test_every_bias_mutation_moves_the_one_step_output(name, mutant):
    """A kernel that dropped a bias or read b2 one unit off must fail the GPU one-step test: the mutation moves the float64 one-step
    output by >= 100 x the max bound asserted there for the FP32-level engines, its median by >= 100 x the median bound of the
    reduced-precision engines, and its max by >= 10 x their loose max bound."""
    s, Q = sample_pairs(name)
    ref = spec.MLPPredictor(mlp_weights(name), dtype=torch.float64).step(s, Q).numpy()
    mut = spec.MLPPredictor(mlp_weights(name, **MUTANTS[mutant](mlp_arrays(name))), dtype=torch.float64).step(s, Q).numpy()
    d = one_step_residual(mut, ref)
    dist, med = float(d.max()), float(np.median(d))
    engines = ("simt",) if MLP_SETS[name][0] != 128 else ("simt", "tcgen05")
    for e in engines:
        assert dist >= TEETH * one_step_bound(e, name), (name, mutant, e, dist)
    if MLP_SETS[name][0] == 128:
        for e in ONE_STEP_MEDIAN_BOUND:
            assert med >= TEETH * ONE_STEP_MEDIAN_BOUND[e], (name, mutant, e, med)
            assert dist >= 10 * one_step_bound(e, name), (name, mutant, e, dist)


def _preactivations(name, s, Q):
    w = {k: torch.from_numpy(np.array(v, np.float64)) for k, v in mlp_arrays(name).items()}
    x = torch.cat([Q, s[:, 1:]], dim=1)
    a1 = x @ w["W1"] + w["b1"]
    a2 = torch.tanh(a1) @ w["W2"] + w["b2"]
    return a1.numpy(), a2.numpy()


def test_saturating_set_reaches_saturation():
    """At least 30 % of the layer-2 pre-activations beyond |a| = 3 (tanh within 5e-3 of +-1) and some layer-1 pre-activations beyond
    15 (the kernels' tanh clamp); the biased set stays in the linear-ish range of the default weights."""
    a1, a2 = _preactivations("saturating", *sample_pairs("saturating"))
    assert np.mean(np.abs(a2) > 3.0) >= 0.30, float(np.mean(np.abs(a2) > 3.0))
    assert np.any(np.abs(a1) > 15.0), float(np.abs(a1).max())
    b1, b2 = _preactivations("biased", *sample_pairs("biased"))
    assert np.mean(np.abs(b2) > 3.0) < 0.05


@pytest.mark.parametrize("name", sorted(MLP_SETS))
def test_product_and_oracle_mlp_weights_are_the_same_numbers(name):
    s, w = mlp_spec(name), mlp_weights(name)
    assert s.hidden == MLP_SETS[name][0]
    for k in ("W1", "b1", "W2", "b2", "W3", "b3"):
        a, b = getattr(s, k), getattr(w, k)
        assert a.dtype == b.dtype == np.float32 and a.shape == b.shape
        np.testing.assert_array_equal(a, b)
    assert np.all(s.b1 != 0) and np.all(s.b2 != 0) and np.all(s.b3 != 0)
    assert len(np.unique(s.b2)) == s.hidden  # per-unit distinct: a bias read one unit off changes the value


@pytest.mark.parametrize("hidden", GRU_WIDTHS + (32,))
def test_product_and_oracle_gru_weights_are_the_same_numbers(hidden):
    import control_toolkit_b200 as ctk
    s, w = gru_spec(hidden), gru_weights(hidden)
    assert s.hidden == w.hidden == hidden
    for k in s._KEYS:
        np.testing.assert_array_equal(getattr(s, k), getattr(w, k))
    if hidden == 32:  # the fixtures' network: the product's own random_init draws the same numbers
        r = ctk.GRUSpec.random_init(GRU_SEED)
        for k in s._KEYS:
            np.testing.assert_array_equal(getattr(s, k), getattr(r, k))


def test_specs_accept_every_advertised_width_and_nothing_else():
    import control_toolkit_b200 as ctk
    for hid in range(16, 129, 16):
        assert ctk.MLPSpec.random_init(1, hidden=hid).hidden == hid
    for hid in (8, 16, 24, 32):
        assert ctk.GRUSpec.random_init(1, hidden=hid).hidden == hid
    for hid in (8, 24, 144):
        with pytest.raises(ValueError):
            ctk.MLPSpec.random_init(1, hidden=hid)
    for hid in (4, 12, 40):
        with pytest.raises(ValueError):
            ctk.GRUSpec.random_init(1, hidden=hid)
