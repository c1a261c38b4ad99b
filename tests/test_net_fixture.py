"""Network parity, pinned (SURVEY 8c / VERDICT r1 item 4): tests/golden/net_fixture.npz holds the
outputs of one of the reference's own shipped TFLite graphs, executed by hand operator by
operator (tests/golden/make_net_fixture.py). The CPU restatement of the network (tests/netref.py,
the oracle of the GPU kernels) and the weight importer are checked against it here; the CUDA
kernels in tests/test_gpu_net.py."""
import os

import numpy as np

from netref import forward_folded
from util import NO_REFERENCE, reference_file

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_fixture():
    z = np.load(os.path.join(GOLD, "net_fixture.npz"))
    x = z["positions"].astype(np.float32) / np.float32(4)
    return z, x


def test_fixture_shape_and_output_order():
    z, x = load_fixture()
    assert x.shape == (512, 70) and z["value"].shape == (512,) and z["policy"].shape == (512, 96)
    # TFLite conversions return the policy first, the value second (rating/tourney.pyx:153-154)
    assert list(z["output_order"]) == ["policy", "value"]
    assert np.allclose(z["policy"].sum(1), 1.0, atol=1e-5) and np.all(np.abs(z["value"]) <= 1.0)
    # float32 execution of the graph vs float64 execution: the error budget of fp32 itself
    assert np.abs(z["value"] - z["value64"]).max() < 5e-5
    assert np.abs(z["policy"] - z["policy64"]).max() < 5e-5


def test_network_restatement_and_importer_match_the_hand_evaluated_graph():
    """netref.forward_folded (Keras semantics restated, BatchNorm folded by the importer's own
    algebra) on the imported weights == the graph walked operator by operator."""
    z, x = load_fixture()
    flat = np.load(os.path.join(GOLD, "trained_net.npz"))["flat"]
    v, p = forward_folded(flat, x, np.float64)
    assert np.abs(v - z["value64"]).max() < 5e-6      # folded weights are stored in fp32
    assert np.abs(p - z["policy64"]).max() < 5e-6
    assert (p.argmax(1) == z["policy64"].argmax(1)).all()


def test_importer_reproduces_the_committed_weights():
    src = reference_file("corintho_ai/docker/tflite_model.tflite")
    if src is None:
        import pytest
        pytest.skip(NO_REFERENCE)
    from corintho_ai_b200.tflite_import import load_tflite_weights
    flat = np.load(os.path.join(GOLD, "trained_net.npz"))["flat"]
    assert load_tflite_weights(src).tobytes() == flat.tobytes()
