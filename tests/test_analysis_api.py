"""The Analysis surface without a GPU: it fails loudly (no CPU fallback), and its host-side
checks run before the library is asked for anything."""
import numpy as np
import pytest

import corintho_ai_b200 as cb


def test_analysis_raises_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(cb.Corintho200Error):
        cb.Analysis(16, 64, 16, 1.0, 0.25)


def test_invalid_parameters_are_rejected_before_the_device_is_touched():
    for args in [(0, 64, 16), (16, 0, 16), (16, 64, 0), (16, 64, 65)]:
        with pytest.raises(cb.Corintho200Error, match="invalid argument"):
            cb.Analysis(*args)
    with pytest.raises(cb.Corintho200Error, match="invalid argument"):
        cb.Analysis(16, 64, 16, c_puct=0.0)
    with pytest.raises(cb.Corintho200Error, match="invalid argument"):
        cb.Analysis(16, 64, 16, epsilon=1.5)


def test_output_buffers_are_checked_like_the_trainers():
    ok = np.zeros(8, np.int32)
    assert cb._out_buf(ok, np.int32, 8, "x") is ok
    for bad in (np.zeros(8, np.int64), np.zeros(16, np.int32)[::2], np.zeros(7, np.int32), [0] * 8):
        with pytest.raises(cb.Corintho200Error):
            cb._out_buf(bad, np.int32, 8, "x")


def test_check_states_needs_no_gpu():
    from oracle.pyoracle import OracleLib
    start = cb.planes_from_reference_order(OracleLib().start()[None])
    bad = start.copy()
    bad[0, 1] |= np.uint64(2) << np.uint64(48)  # side to move 2
    assert cb.check_states(np.concatenate([start, bad])).tolist() == [True, False]
