"""The answer buffers of a new trainer start as zeros whatever the device memory held before. A fused
two-model tourney reads answer rows that no evaluation of the run has written yet (the answer offsets
of tourney.cpp:54-62), and the reference loop's fresh buffers hold zeros there. Device memory that
the process used and freed earlier comes back with its old contents, so the engine has to clear its
buffers itself, in every layout the network writes."""
import numpy as np
import pytest

import corintho_ai_b200 as cb
from test_gpu_tourney import _Engine
from util import make_tourney, run_tourney

pytestmark = pytest.mark.gpu


def recycle_poisoned_memory(gib=16):
    """Fill device memory with NaNs and hand it back to the driver, so that the next allocations
    of this process are likely to reuse it."""
    import torch
    blocks = [torch.full((1 << 28,), float("nan"), device="cuda") for _ in range(gib)]  # 1 GiB each
    torch.cuda.synchronize()
    del blocks
    torch.cuda.empty_cache()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_fused_two_model_tourney_after_device_memory_was_reused(oracle, precision):
    recycle_poisoned_memory()
    weights = {m: cb.fold_batchnorm(cb.random_weights(100 + m)) for m in (0, 1)}
    eng = make_tourney(_Engine(), "two_models")
    for m, w in weights.items():
        eng.set_weights(m, w, precision)
    assert eng.run(0)
    helpers = {}
    for m, w in weights.items():
        helpers[m] = cb.Trainer(64, "", 1, 64, 16)
        helpers[m].set_weights(w, 0, precision)
    ref = run_tourney(make_tourney(oracle, "two_models"),
                      {m: (lambda req, h=helpers[m]: h.evaluate(req)) for m in weights})
    got = np.array(eng.scores(), np.float64).reshape(-1, 3)
    assert (got == ref["scores"]).all()
