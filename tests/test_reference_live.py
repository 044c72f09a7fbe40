"""The UNMODIFIED reference classes (with oracle/kaolin_shim) were run on seeded `make_case` cases by
oracle/make_golden.py::make_live; what they returned is frozen in tests/golden/ref_live_*.npz.  The oracle restatement
must reproduce it on the same cases."""
import os

import numpy as np
import pytest

from tests.parity_utils import GOLDEN_DIR, live_golden_name, make_case, run_oracle_step


@pytest.mark.parametrize("levels,frames,poly", [(2, 1, True), (4, 2, True), (3, 2, False)])
def test_oracle_equals_live_reference(levels, frames, poly):
    ref = np.load(os.path.join(GOLDEN_DIR, live_golden_name(levels, frames, poly) + ".npz"))
    case = make_case(n_points=1200, n_batch=1000, feat_levels=levels, seed=77 + levels, n_frames=frames, poly=poly)
    assert [t.shape[0] for t in case["tables"]] == ref["table_rows"].tolist()
    want = run_oracle_step(case)
    for i, b in enumerate(want["indices"]):
        assert np.array_equal(ref[f"exp_indices_{i}"].astype(np.int64), b)
    assert np.abs(ref["exp_pred"] - want["pred"]).max() < 1e-6
    assert abs(float(ref["exp_loss"]) - want["loss"]) < 1e-6
    for k, g in enumerate(want["table_grads"]):
        # the golden keeps which rows have a gradient, a weighted sum of each such row (weights in [0.5, 1.5], held to
        # the bound of a single element), and a seeded sample of whole rows
        touched = np.abs(g).sum(1) > 0
        assert np.array_equal(np.packbits(touched), ref[f"exp_tgrad_touched_{k}"])
        tol = 1e-5 * np.abs(g).max() + 1e-12
        rowsum = g[touched].astype(np.float64) @ ref["tgrad_row_weights"]
        assert np.abs(ref[f"exp_tgrad_rowsum_{k}"] - rowsum).max() <= tol
        assert np.abs(ref[f"exp_tgrad_{k}"] - g[ref[f"exp_tgrad_rows_{k}"]]).max() <= tol
