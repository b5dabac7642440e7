"""CPU tests: the standalone oracle restatements (oracle/mppi.py, cem.py, rpgd.py) against the golden vectors
produced by the reference's UNMODIFIED files (oracle/gen_golden.py).  Both run torch-CPU fp32 with the same op
order, so agreement is expected at rounding level; tolerance 2e-6 relative (fixtures were generated
single-threaded, the test may run with several threads -> different reduction order)."""
import os
import sys

import numpy as np
import pytest

from helpers import golden_names, load_golden, make_oracle, maybe_reset_oracle, rel_err, replay
from oracle.refharness.workspace import reference_available, reference_has

TOL = 2e-6


def test_noise_stream_checksum():
    from oracle.replay_rng import ReplayRNG
    for name in golden_names():
        z, meta = load_golden(name)
        import json
        r = ReplayRNG(meta["noise_seed"], as_torch=False)
        acc = 0.0
        for kind, shape in json.loads(str(z["noise_blocks"])):
            acc += float(np.sum(r.standard_draws(kind, shape).astype(np.float64)))
        assert abs(acc - float(z["noise_checksum"][0])) < 1e-6, name


@pytest.mark.parametrize("name", golden_names("mppi_"))
def test_mppi_oracle_matches_reference(name):
    z, meta = load_golden(name)
    o = make_oracle(meta)
    rng = replay(meta)
    for t in range(meta["ticks"]):
        maybe_reset_oracle(o, meta, t, rng)
        u = o.step(z["states"][t], rng)
        assert rel_err(u, z[f"u_{t}"]) < TOL
        assert rel_err(o.u_nom.numpy(), z[f"u_nom_{t}"]) < TOL
        assert rel_err(o.last["J"], z[f"J_{t}"]) < TOL
        if t == 0 and "rollouts_0" in z:
            assert rel_err(o.last["rollouts"], z["rollouts_0"]) < TOL
            assert rel_err(o.last["Q"], z["Q_logged_0"]) < TOL


@pytest.mark.parametrize("name", golden_names("cem_"))
def test_cem_oracle_matches_reference(name):
    z, meta = load_golden(name)
    o = make_oracle(meta)
    rng = replay(meta)
    for t in range(meta["ticks"]):
        maybe_reset_oracle(o, meta, t, rng)
        u = o.step(z["states"][t], rng)
        np.testing.assert_array_equal(o.last["elite_idx"], z[f"elite_idx_{t}"])
        assert rel_err(u, z[f"u_{t}"]) < TOL
        assert rel_err(o.dist_mue.numpy(), z[f"dist_mue_{t}"]) < TOL
        assert rel_err(o.stdev.numpy(), z[f"stdev_{t}"]) < TOL
        assert rel_err(o.last["J"], z[f"J_{t}"]) < TOL


@pytest.mark.parametrize("name", golden_names("rpgd_"))
def test_rpgd_oracle_matches_reference(name):
    z, meta = load_golden(name)
    o = make_oracle(meta)
    rng = replay(meta)
    o.reset(rng)
    assert rel_err(o.Q.numpy(), z["Q_init"]) == 0.0
    for t in range(meta["ticks"]):
        maybe_reset_oracle(o, meta, t, rng)
        u = o.step(z["states"][t], rng)
        assert rel_err(u, z[f"u_{t}"]) < TOL, (t, u, z[f"u_{t}"])
        assert rel_err(o.Q.numpy(), z[f"Q_{t}"]) < TOL
        assert rel_err(o.m.numpy(), z[f"adam_m_{t}"]) < 1e-5
        assert rel_err(o.v.numpy(), z[f"adam_v_{t}"]) < 1e-5
        assert o.adam_step == int(z[f"adam_step_{t}"][0])
        np.testing.assert_array_equal(o.ages.numpy(), z[f"ages_{t}"])
        assert rel_err(o.last["J"], z[f"J_{t}"]) < TOL
        assert rel_err(o.last["u_nom"], z[f"u_nom_{t}"]) < TOL


def test_rpgd_keras_vs_torch_adam_form():
    """SURVEY.md 8a row a10 expected the Keras-form and torch-form Adam (eps placement: eps vs eps*sqrt(1-b2^t))
    to agree within 1e-5.  Measured here: they do NOT where |g| ~ 1e-6 (late-horizon controls), the population
    differs by up to ~3e-3 relative after one tick.  Both forms are therefore implemented and parity-tested
    separately (torch form vs the unmodified reference file, Keras form vs this oracle); this test only pins the
    size of the gap so a change in either form is noticed."""
    z, meta = load_golden("rpgd_c3")
    o = make_oracle(meta, adam_form="keras")
    rng = replay(meta)
    o.reset(rng)
    for t in range(3):
        u = o.step(z["states"][t], rng)
        assert rel_err(u, z[f"u_{t}"]) < 5e-2
        assert rel_err(o.Q.numpy(), z[f"Q_{t}"]) < 5e-2


@pytest.mark.parametrize("name", golden_names("random_action_"))
def test_random_action_oracle_matches_reference(name):
    """oracle/random_action.py vs the unmodified reference Optimizers/optimizer_random_action_tf.py (SURVEY 8f.1)."""
    z, meta = load_golden(name)
    o = make_oracle(meta)
    rng = replay(meta)
    o.reset(rng)  # the reference draws (and discards) one population in optimizer_reset
    for t in range(meta["ticks"]):
        u = o.step(z["states"][t], rng)
        assert o.last["best_idx"] == int(z[f"best_idx_{t}"][0])
        assert rel_err(u, z[f"u_{t}"]) == 0.0  # u is one of the sampled controls: bit-exact
        assert rel_err(o.last["J"], z[f"J_{t}"]) < TOL
        if t == 0 and "rollouts_0" in z:
            assert rel_err(o.last["rollouts"], z["rollouts_0"]) < TOL
            assert rel_err(o.last["Q"], z["Q_logged_0"]) == 0.0


@pytest.mark.parametrize("name", golden_names("gradient_"))
def test_gradient_oracle_matches_reference(name):
    """oracle/gradient.py vs the unmodified reference Optimizers/optimizer_gradient_tf.py (SURVEY 8f.1)."""
    z, meta = load_golden(name)
    o = make_oracle(meta)
    rng = replay(meta)
    o.reset(rng)
    assert rel_err(o.Q.numpy(), z["Q_init"]) == 0.0
    for t in range(meta["ticks"]):
        u = o.step(z["states"][t], rng)
        assert o.last["best_idx"] == int(z[f"best_idx_{t}"][0])
        assert rel_err(u, z[f"u_{t}"]) < 5e-6
        assert rel_err(o.Q.numpy(), z[f"Q_{t}"]) < 5e-6
        assert rel_err(o.m.numpy(), z[f"adam_m_{t}"]) < 2e-5
        assert rel_err(o.v.numpy(), z[f"adam_v_{t}"]) < 2e-5
        assert o.adam_step == int(z[f"adam_step_{t}"][0])
        assert rel_err(o.last["J"], z[f"J_{t}"]) < 5e-6


@pytest.mark.parametrize("name", golden_names("gradcem_"))
def test_cem_grad_oracles_match_reference(name):
    """oracle/cem_grad.py vs the unmodified reference Optimizers/optimizer_cem_naive_grad_tf.py and
    optimizer_cem_grad_bharadhwaj_tf.py (SURVEY 8f.1): identical elite index lists in every outer iteration."""
    z, meta = load_golden(name)
    o = make_oracle(meta)
    rng = replay(meta)
    o.reset(rng)
    for t in range(meta["ticks"]):
        maybe_reset_oracle(o, meta, t, rng)
        u = o.step(z["states"][t], rng)
        np.testing.assert_array_equal(o.last["elite_idx"], z[f"elite_idx_{t}"])
        assert rel_err(u, z[f"u_{t}"]) < 5e-6
        assert rel_err(o.dist_mue.numpy(), z[f"dist_mue_{t}"]) < 5e-6
        assert rel_err(o.stdev.numpy(), z[f"stdev_{t}"]) < 5e-6
        assert rel_err(o.last["Q"], z[f"Qn_{t}"]) < 5e-6
        assert rel_err(o.last["J"], z[f"J_{t}"]) < 5e-6
        if f"adam_m_{t}" in z:
            assert rel_err(o.m.numpy(), z[f"adam_m_{t}"]) < 2e-5
            assert rel_err(o.v.numpy(), z[f"adam_v_{t}"]) < 2e-5
            assert o.adam_step == int(z[f"adam_step_{t}"][0])


@pytest.mark.parametrize("name", ["mppi_c1_n2000", "mppi_mlp_h50_n64"])
def test_mppi_oracle_chunked_equals_monolithic(name):
    """oracle.mppi.MPPIOracle.step_chunked (used for the full-size C4 / C5 parity tests) against step() and the fixture."""
    z, meta = load_golden(name)
    o, oc = make_oracle(meta), make_oracle(meta)
    rng, rngc = replay(meta), replay(meta)
    for t in range(min(meta["ticks"], 3)):
        u = o.step(z["states"][t], rng)
        uc = oc.step_chunked(z["states"][t], rngc, chunk=37)
        assert rel_err(uc, u) < TOL
        assert rel_err(oc.u_nom.numpy(), o.u_nom.numpy()) < TOL
        assert rel_err(oc.u_nom.numpy(), z[f"u_nom_{t}"]) < 2 * TOL
        # per-rollout costs: identical arithmetic, but torch's vectorised sin / cos round differently in the SIMD body and the scalar
        # remainder of a batch, and the unstable pendulum amplifies that ulp (the fp32 noise floor of DESIGN.md section 3)
        eJ = np.abs(oc.last["J"].astype(np.float64) - o.last["J"]) / (np.abs(o.last["J"]) + 1e-3)
        assert np.median(eJ) < 1e-6 and eJ.max() < 1e-3


def test_queue_rng_replays_given_blocks():
    from oracle.replay_rng import QueueRNG
    a, b = np.arange(6, dtype=np.float32), np.arange(4, dtype=np.float32) + 10
    r = QueueRNG([a, b])
    x = r.normal([2, 3, 1], mean=1.0, stddev=2.0)
    np.testing.assert_allclose(x.numpy().ravel(), a * 2 + 1)
    y = r.uniform([4], minval=-1.0, maxval=1.0)
    np.testing.assert_allclose(y.numpy().ravel(), b * 2 - 1)
    with pytest.raises(RuntimeError):
        r.normal([1])


def test_philox4x32_10_known_answers():
    """oracle/philox.py (the CPU restatement of the generator behind the reference's rng, others/globals_and_utils.py:95-97, and
    of the device generator K0) against the known-answer vectors Random123 1.09 ships for philox4x32-10 (examples/kat_vectors:
    counter, key -> output), plus the structural properties the kernels rely on."""
    from oracle import philox as P
    kat = [
        ([0x00000000] * 4, [0x00000000] * 2, [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
        ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
        ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0], [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]),
    ]
    for ctr, key, out in kat:
        np.testing.assert_array_equal(P.philox4x32_10(np.array(ctr, np.uint32), np.array(key, np.uint32)), np.array(out, np.uint32))
    # vectorised evaluation == one counter at a time
    ctr = np.random.default_rng(0).integers(0, 2**32, (7, 4), dtype=np.uint64).astype(np.uint32)
    key = np.array([123, 456], np.uint32)
    batch = P.philox4x32_10(ctr, key)
    for i in range(7):
        np.testing.assert_array_equal(batch[i], P.philox4x32_10(ctr[i], key))
    # counter layout of a noise block: draw i of rollout n is word i % 4 of counter (i // 4, n, tick, stream)
    w = P.draw_words(seed=(7 << 32) | 42, stream=1, tick=5, rows=[3, 1000000], per_rollout=10)
    assert w.shape == (2, 10)
    one = P.philox4x32_10(np.array([2, 1000000, 5, 1], np.uint32), np.array([42, 7], np.uint32))
    np.testing.assert_array_equal(w[1, 8:10], one[:2])
    # word -> uniform: 24 bits, [0, 1), exact in fp32
    u = P.uniform24(np.array([0, 0xFF, 0x100, 0xFFFFFFFF], np.uint32))
    np.testing.assert_array_equal(u, np.array([0.0, 0.0, 2.0 ** -24, 1.0 - 2.0 ** -24], np.float32))
    # word -> normal: the mapping covers (0, 1] x [-pi, pi) and gives standard normals
    z, u1 = P.box_muller(P.draw_words(seed=42, stream=0, tick=1, rows=np.arange(4096), per_rollout=16))
    assert u1.min() > 0.0 and u1.max() <= 1.0 and np.isfinite(z).all()
    assert abs(z.mean()) < 0.02 and abs(z.std() - 1.0) < 0.02


REGEN_CASES = ["mppi_c1_n64", "mppi_h43_p10_n64", "mppi_gru_n256", "mppi_dubins_h23_p5_n96", "cem_warmup_n128", "cem_reset_mid_n128", "rpgd_c3",
               "gradient_warmup_n33", "gradcem_bharadhwaj_n32", "random_action_n512"]


@pytest.mark.skipif(not reference_available(), reason="needs a Control_Toolkit checkout: set CTK_REFERENCE to its path")
def test_committed_fixtures_are_what_the_unmodified_reference_produces(tmp_path):
    """Pinning of the fixtures themselves: re-run the reference's UNMODIFIED optimizer files (oracle/gen_golden.py, in a process of
    its own because the harness changes the working directory and the module table) and compare every array of a committed fixture
    with the regenerated one -- bit for bit on the host the fixtures were made on (the build container: no warning is raised), to 1e-5
    of the array's scale on a host whose torch-CPU kernels round differently; the json config on the keys both hold (later fixtures carry more metadata keys)."""
    import json
    import subprocess
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "oracle.gen_golden", "--out", str(tmp_path)] + REGEN_CASES, cwd=repo, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    not_bitwise = []
    for name in REGEN_CASES:
        new = np.load(os.path.join(str(tmp_path), name + ".npz"), allow_pickle=False)
        old = np.load(os.path.join(repo, "tests", "golden", name + ".npz"), allow_pickle=False)
        assert sorted(new.files) == sorted(old.files), name
        for k in old.files:
            if k == "config":
                a, b = json.loads(str(new[k])), json.loads(str(old[k]))
                assert all(a[q] == b[q] for q in b), (name, a, b)
                continue
            assert new[k].dtype == old[k].dtype and new[k].shape == old[k].shape, (name, k)
            if new[k].tobytes() == old[k].tobytes():
                continue
            # Not bit-identical: torch-CPU picks its kernels by the host's instruction set, so on another CPU model than the one the
            # fixtures were generated on the last bit may differ.  Then the fixture must still be the reference's output to the
            # tolerance every oracle test in this file uses; index arrays (elite lists) may differ only where costs tie to an ulp.
            not_bitwise.append((name, k))
            if np.issubdtype(old[k].dtype, np.floating):
                scale = max(float(np.max(np.abs(old[k]))), 1e-6)
                assert float(np.max(np.abs(new[k].astype(np.float64) - old[k].astype(np.float64)))) / scale < 1e-5, (name, k)
            else:
                assert np.mean(new[k] == old[k]) > 0.98, (name, k)
    if not_bitwise:
        import warnings
        warnings.warn(f"regenerated fixtures equal the committed ones to tolerance, not bit for bit (other host CPU?): {not_bitwise[:5]}")


def test_interpolation_matrix_equals_the_unmodified_reference_interpolator():
    """a2 (others/Interpolator.py:53-84,97-106) pinned directly: oracle.mppi.interpolation_matrix against the reference class's weights
    over 1152 geometries (H = 1 .. 101, period = 1 .. 12, one and two control inputs; includes H < period, period 1, and H - 1 a multiple
    of the period, where the last-point quirk shows), bit for bit.  The weights do not depend on the number of control inputs, so
    tests/golden/interpolator/weights_sweep.npz stores them once per (H, period).  They were written from oracle.mppi.interpolation_matrix
    as it stands since the live check below found it equal to the reference Interpolator bit for bit over this sweep;
    ``drive_reference_interpolator.py --write`` rewrites them from the reference itself.  With CTK_REFERENCE naming a checkout, the
    reference class is also run live: its weights against the stored ones and the oracle's, its applied interpolation to one ulp."""
    from helpers import load_interpolation_weights
    from oracle.mppi import interpolation_matrix
    stored = load_interpolation_weights()
    assert len(stored) == 576  # 48 horizons x 12 periods
    for (H, period), W in stored.items():
        np.testing.assert_array_equal(interpolation_matrix(H, period), W, err_msg=f"H={H} period={period}")
    if not reference_has("others"):
        return
    import json
    import subprocess
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(repo, "tests", "dropin", "drive_reference_interpolator.py")], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("INTERP_RESULT ")]
    assert line, r.stdout[-2000:]
    res = json.loads(line[-1][len("INTERP_RESULT "):])
    assert res["checked"] == 1152 and res["n_bad"] == 0, res
