"""The analysis' external-evaluator protocol (cb200_analysis_begin .. _results) without a GPU: argument
errors come back as CB200_ERR_ARG before anything else is looked at, no session can be opened without
a device, and the Python wrappers reject bad buffers before the library is called."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest

import corintho_ai_b200 as cb

ERR_ARG = -1


def test_entry_points_reject_null_and_negative_arguments_first():
    L = cb.lib()
    buf = np.zeros(16 * 96, np.float32)
    st = np.zeros((4, 2), np.uint64)
    i32 = np.zeros(16 * 96, np.int32)
    p, s = cb._ptr(buf), cb._ptr(st)
    calls = {
        "begin": lambda: L.cb200_analysis_begin(None, 4, s, 0),
        "num_requests": lambda: L.cb200_analysis_num_requests(None),
        "write_requests": lambda: L.cb200_analysis_write_requests(None, p),
        "do_iteration": lambda: L.cb200_analysis_do_iteration(None, p, p, 1),
        "results": lambda: L.cb200_analysis_results(None, cb._ptr(i32), cb._ptr(i32), p, cb._ptr(i32), p),
        "write_requests_device": lambda: L.cb200_analysis_write_requests_device(None, C.c_void_p(4096)),
        "do_iteration_device": lambda: L.cb200_analysis_do_iteration_device(None, C.c_void_p(4096),
                                                                            C.c_void_p(4096), 1),
    }
    for name, call in calls.items():
        assert call() == ERR_ARG, name
        assert b"null analysis" in L.cb200_last_error(), name
    # negative sizes and null buffers are argument errors too, whatever the handle
    assert L.cb200_analysis_do_iteration(None, p, p, -1) == ERR_ARG
    assert L.cb200_analysis_do_iteration_device(None, None, None, 3) == ERR_ARG


def test_no_session_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    # the object that a session lives in needs the device: creating it is the CUDA error
    assert not cb.lib().cb200_analysis_create(16, 64, 16, 1.0, 0.25)
    assert cb.lib().cb200_last_error()
    with pytest.raises(cb.Corintho200Error):
        cb.Analysis(16, 64, 16)


class FakeCudaTensor:
    """What the device forms read from a torch CUDA tensor, without needing a GPU."""

    def __init__(self, numel, dtype="torch.float32", contiguous=True, device="cuda"):
        self.dtype, self.device = dtype, SimpleNamespace(type=device, index=0)
        self._numel, self._contiguous = numel, contiguous

    def is_contiguous(self):
        return self._contiguous

    def numel(self):
        return self._numel

    def data_ptr(self):
        return 0x7F0000000000


def test_device_buffers_are_checked():
    import torch
    assert cb._dev_f32(FakeCudaTensor(70), 70, "x") == 0x7F0000000000
    for bad in (FakeCudaTensor(69), FakeCudaTensor(70, dtype="torch.float64"),
                FakeCudaTensor(70, contiguous=False), FakeCudaTensor(70, device="cpu"),
                torch.zeros(70), np.zeros(70, np.float32), None):
        with pytest.raises(cb.Corintho200Error):
            cb._dev_f32(bad, 70, "x")


def test_python_wrappers_reject_bad_buffers_before_the_library():
    a = object.__new__(cb.Analysis)  # no device: stand in for an open session with 3 requests
    a._h = None
    a.num_requests = lambda: 3
    ok_rows = np.zeros((3, 70), np.float32)
    for bad in (np.zeros((3, 70), np.float64), np.zeros((2, 70), np.float32), np.zeros((6, 70), np.float32)[::2],
                [[0.0] * 70] * 3):
        with pytest.raises(cb.Corintho200Error, match="write_requests"):
            a.write_requests(bad)
    with pytest.raises(cb.Corintho200Error, match="do_iteration: eval"):
        a.do_iteration(np.zeros(2, np.float32), np.zeros((3, 96), np.float32))
    with pytest.raises(cb.Corintho200Error, match="do_iteration: probs"):
        a.do_iteration(np.zeros(3, np.float32), np.zeros((3, 95), np.float32))
    with pytest.raises(cb.Corintho200Error, match="None"):
        a.do_iteration()  # 3 requests pending
    with pytest.raises(cb.Corintho200Error, match="write_requests_device"):
        a.write_requests_device(ok_rows)
    with pytest.raises(cb.Corintho200Error, match="write_requests_device"):
        a.write_requests_device(FakeCudaTensor(3 * 70 - 1))
    with pytest.raises(cb.Corintho200Error, match="do_iteration_device: eval"):
        a.do_iteration_device(FakeCudaTensor(2), FakeCudaTensor(3 * 96))
    with pytest.raises(cb.Corintho200Error, match="do_iteration_device: probs"):
        a.do_iteration_device(FakeCudaTensor(3), FakeCudaTensor(3 * 96, dtype="torch.bfloat16"))
    for bad in (np.zeros((4, 3), np.uint64), np.zeros(8, np.uint64)):
        with pytest.raises(cb.Corintho200Error, match="begin: states"):
            a.begin(bad)
