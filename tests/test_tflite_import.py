"""TFLite checkpoint import (SURVEY.md 8f-4): container parsing and folding, checked on CPU with
the numpy network; the trained network must put its policy mass on legal moves."""
import os

import numpy as np
import pytest

from netref import forward_folded
from util import NO_REFERENCE, REFERENCE, reference_file

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLAT = np.load(os.path.join(ROOT, "tests", "golden", "trained_net.npz"))["flat"]
REF_TFLITE = reference_file("corintho_ai/docker/tflite_model.tflite")


def _positions(oracle, n, seed=0):
    rng = np.random.default_rng(seed)
    rows, masks = [], []
    st = oracle.start()
    while len(rows) < n:
        mask, _ = oracle.legal(st)
        ids = [m for m in range(96) if (mask[m >> 5] >> (m & 31)) & 1]
        if not ids:
            st = oracle.start()
            continue
        rows.append(oracle.encode(st))
        masks.append(np.array([(mask[m >> 5] >> (m & 31)) & 1 for m in range(96)], bool))
        st = oracle.do_move(st, int(rng.choice(ids)))
    return np.stack(rows), np.stack(masks)


def test_trained_network_prefers_legal_moves(oracle):
    x, legal = _positions(oracle, 400)
    v, p = forward_folded(FLAT, x, np.float64)
    assert ((v > -1) & (v < 1)).all() and np.allclose(p.sum(1), 1, atol=1e-5)
    mass = (p * legal).sum(1)
    # positions come from uniformly random play (off-distribution for the trained net); a
    # random-init network puts ~ n_legal/96 = 0.28 of its mass on legal moves here
    import corintho_ai_b200 as cb
    _, pr = forward_folded(cb.fold_batchnorm(cb.random_weights(3)), x, np.float64)
    assert mass.mean() > 0.6 and mass.mean() > 2.0 * (pr * legal).sum(1).mean()
    assert mass[0] > 0.999  # the start position


@pytest.mark.skipif(REF_TFLITE is None, reason=NO_REFERENCE)
def test_fixture_equals_fresh_import_and_all_checkpoints_load():
    import glob
    from corintho_ai_b200.tflite_import import load_tflite_weights, parse_tflite
    assert load_tflite_weights(REF_TFLITE).tobytes() == FLAT.tobytes()
    tensors, ops, inputs, outputs = parse_tflite(REF_TFLITE)
    assert tensors[inputs[0]]["shape"] == [1, 70]
    # rating/tourney.pyx:153-154: TFLite outputs are (policy, value), the reverse of Keras
    assert tensors[outputs[0]]["shape"] == [1, 96] and tensors[outputs[1]]["shape"] == [1, 1]
    files = glob.glob(os.path.join(REFERENCE, "corintho_ai", "rating", "tflite_models", "*.tflite"))
    assert len(files) == 95
    for f in files[::12]:
        assert load_tflite_weights(f).size == 127997
