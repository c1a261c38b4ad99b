"""Analysis.run_device's argument checks, which run before the library is called (no GPU needed):
the states and output buffers must be contiguous CUDA tensors of the right dtype, shape and size."""
from types import SimpleNamespace

import pytest

import corintho_ai_b200 as cb


class FakeCudaTensor:
    """What run_device reads from a torch CUDA tensor, without needing a GPU."""

    def __init__(self, shape, dtype="torch.int64", contiguous=True, device="cuda"):
        self.shape = tuple(shape)
        self.dtype, self.device = dtype, SimpleNamespace(type=device, index=0)
        self._contiguous = contiguous

    def is_contiguous(self):
        return self._contiguous

    def numel(self):
        n = 1
        for d in self.shape:
            n *= d
        return n

    def data_ptr(self):
        return 0x7F0000000000


def outputs(n, **over):
    out = {"moves": FakeCudaTensor((n,), "torch.int32"), "results": FakeCudaTensor((n,), "torch.int32"),
           "values": FakeCudaTensor((n,), "torch.float32"), "visits": FakeCudaTensor((n, 96), "torch.int32"),
           "evals": FakeCudaTensor((n, 96), "torch.float32"), "status": FakeCudaTensor((2,), "torch.int32")}
    out.update(over)
    return out


def analysis():
    a = object.__new__(cb.Analysis)  # no device: the checks come first
    a._h = None
    return a


@pytest.mark.parametrize("states", [
    FakeCudaTensor((8, 2), device="cpu"),
    FakeCudaTensor((8, 2), dtype="torch.float32"),
    FakeCudaTensor((8, 2), dtype="torch.int32"),
    FakeCudaTensor((8, 2), contiguous=False),
    FakeCudaTensor((8, 3)),
    FakeCudaTensor((16,)),
    FakeCudaTensor((0, 2)),
    [[0, 0]] * 8,
    None,
])
def test_run_device_rejects_bad_states(states):
    with pytest.raises(cb.Corintho200Error, match="run_device: states"):
        analysis().run_device(states, out=outputs(8))


@pytest.mark.parametrize("key,bad", [
    ("moves", FakeCudaTensor((8,), "torch.int64")),
    ("results", FakeCudaTensor((7,), "torch.int32")),
    ("values", FakeCudaTensor((8,), "torch.float64")),
    ("visits", FakeCudaTensor((8, 96), "torch.int32", contiguous=False)),
    ("evals", FakeCudaTensor((8, 96), "torch.float32", device="cpu")),
    ("status", FakeCudaTensor((1,), "torch.int32")),
])
def test_run_device_rejects_bad_outputs(key, bad):
    with pytest.raises(cb.Corintho200Error, match=f"run_device: {key}"):
        analysis().run_device(FakeCudaTensor((8, 2), dtype="torch.uint64"), out=outputs(8, **{key: bad}))


def test_device_buffer_check_takes_a_dtype():
    t = FakeCudaTensor((4, 2), dtype="torch.uint64")
    assert cb._dev_buf(t, 8, "x", ("torch.int64", "torch.uint64")) == 0x7F0000000000
    with pytest.raises(cb.Corintho200Error, match="int64 or uint64"):
        cb._dev_buf(FakeCudaTensor((4, 2), dtype="torch.float32"), 8, "x", ("torch.int64", "torch.uint64"))
    with pytest.raises(cb.Corintho200Error, match="float32"):
        cb._dev_buf(t, 8, "x")


def test_the_entry_point_is_bound():
    assert cb.lib().cb200_analysis_run_device.argtypes is not None
