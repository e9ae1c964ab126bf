"""Host-side pieces of per-shot priors (no GPU): the column order a WindowPlan records, and the C-ABI declarations."""
import os

import numpy as np

from conftest import ROOT


def test_window_plan_records_column_order():
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, detector_error_model, dem_to_check_matrices
    from slidingwindowdecoder_b200.windows import build_windows, reshuffle_by_round
    code, A, B = bb_code(72)
    chk, obs, pri = dem_to_check_matrices(detector_error_model(bb_memory_circuit(code, A, B, 0.003, 6)))
    plan = build_windows(chk, obs, pri, code.N, W=3, F=1, method=1)
    order = plan.col_order
    assert sorted(order.tolist()) == list(range(chk.shape[1]))
    assert (plan.chk != chk.tocsc()[:, order]).nnz == 0
    assert (plan.obs != obs.tocsc()[:, order]).nnz == 0
    assert np.array_equal(plan.priors, np.asarray(pri)[order])
    assert len(reshuffle_by_round(chk, obs, pri, n=code.N)) == 4          # public return value unchanged
    # window i's genuine DEM columns are plan columns [col0, col0 + ncols_dem)
    for w in plan.windows:
        assert np.array_equal(w.prior[:w.ncols_dem], plan.priors[w.col0:w.col0 + w.ncols_dem])


def test_per_shot_entry_points_declared():
    header = open(os.path.join(ROOT, "include", "swd_b200.h")).read()
    for sym in ("swd_decode_batch_host_llr", "swd_decode_batch_device_llr", "swd_decode_batch_host_packed_llr",
                "swd_decode_batch_device_packed_llr"):
        assert sym + "(" in header
