"""TEST-ONLY driver (subprocess of tests/test_oracle_golden.py; needs the Control_Toolkit checkout named by CTK_REFERENCE): the reference's UNMODIFIED others/Interpolator.py
(through the refharness workspace, which provides the SI_Toolkit computation-library shim it imports) against the oracle's restatement
oracle.mppi.interpolation_matrix over a sweep of (horizon, period, num_control_inputs) -- the weights bit for bit, an applied interpolation to one ulp --
and against the stored weights tests/golden/interpolator/weights_sweep.npz (bit for bit).  ``--write PATH`` stores the reference's weights
of the sweep to PATH instead of comparing with the stored ones."""
import json
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))

HORIZONS = list(range(1, 45)) + [50, 97, 100, 101]
PERIODS = range(1, 13)


def main(write=None):
    import numpy as np
    import torch
    from helpers import load_interpolation_weights
    from oracle.mppi import interpolation_matrix
    from oracle.refharness.workspace import enter_workspace
    enter_workspace()
    import logging
    logging.disable(logging.INFO)
    from Control_Toolkit.others.Interpolator import Interpolator  # the reference module, unmodified
    from SI_Toolkit.computation_library import PyTorchLibrary
    lib = PyTorchLibrary() if isinstance(PyTorchLibrary, type) else PyTorchLibrary
    stored = None if write else load_interpolation_weights()
    geometry, weights = [], []
    rng = np.random.default_rng(0)
    checked, bad = 0, []
    import contextlib
    import io
    for H in HORIZONS:
        for period in PERIODS:
            for nu in (1, 2):
                with contextlib.redirect_stdout(io.StringIO()):  # the reference prints a notice when H < period
                    ref = Interpolator(H, period, nu, lib)
                W = interpolation_matrix(H, period)  # [n_ind, H]
                n_ind = ref.number_of_interpolation_inducing_points
                mat = np.asarray(ref.interp_mat if not torch.is_tensor(ref.interp_mat) else ref.interp_mat.numpy())  # [n_ind, H, nu] (Interpolator.py:75-77)
                ok = (W.shape == (n_ind, H)) and mat.shape == (n_ind, H, nu) and all(np.array_equal(mat[..., c], W) for c in range(nu))
                if stored is not None:
                    ok = ok and all(np.array_equal(mat[..., c], stored[(H, period)]) for c in range(nu))
                elif nu == 1:
                    geometry.append((H, period, n_ind))
                    weights.append(mat[..., 0].astype(np.float32).ravel())
                y = rng.standard_normal((5, n_ind, nu)).astype(np.float32)
                out = ref.interpolate(torch.from_numpy(y)).numpy()  # [5, H, nu]
                mine = np.stack([(torch.from_numpy(y[..., c]) @ torch.from_numpy(W)).numpy() for c in range(nu)], -1)
                # the weights are compared bit for bit above; the product goes through another matmul entry point of torch (batched vs 2-D),
                # which may contract the two non-zero terms of a row with or without an FMA: one ulp
                ok = ok and out.shape == (5, H, nu) and np.allclose(out, mine, rtol=3e-7, atol=1e-7)
                checked += 1
                if not ok:
                    bad.append([H, period, nu])
    if write:
        np.savez_compressed(write, geometry=np.array(geometry, np.int32), weights=np.concatenate(weights))
    print("INTERP_RESULT " + json.dumps({"checked": checked, "n_bad": len(bad), "bad": bad[:10]}))


if __name__ == "__main__":
    main(sys.argv[sys.argv.index("--write") + 1] if "--write" in sys.argv else None)
