"""The reference restatement used by test_gpu_tree_kernels.py can tell right from wrong: each
deliberate error below, applied to tests/treeref.py, changes at least one expected output on the
constructed cases of tests/tree_cases.py. And treeref's slot value agrees with the independent
vectorised expression of test_puct_interval.py."""
import math

import numpy as np
import pytest

import tree_cases as TC
import treeref as T
from test_puct_interval import reference, samples


@pytest.fixture(scope="module")
def gamma(oracle):
    return [float(oracle.gamma_sample(i)) for i in range(1024)]


def selection_outputs():
    out = []
    for c in TC.selection_cases():
        choice, us = TC.ref_choice(c)
        out.append((choice, [T.bits(u) for u in us]))
    return out


def ingest_outputs(gamma):
    out = []
    for c in TC.ingest_cases():
        a, re, ring, idx = T.receive_eval(c["arena"], c["pending"], c["evals"], c["probs"], c["ring"], c["mt_idx"],
                                          c["root_eval"], c["eps"], gamma)
        out.append((a.tobytes(), T.bits(re), ring.tobytes(), idx))
    return out


def _fmaxf(w, m):
    return m if w != w else (w if m != m or w > m else m)


def _round_half_even(x):
    if x != x or abs(x) >= 2.0 ** 63:
        return 0
    return int(round(x))


def _pairwise_sum(values):
    v = list(values)
    if not v:
        return 0.0
    while len(v) > 1:
        v = [T.f32(v[i] + v[i + 1]) if i + 1 < len(v) else v[i] for i in range(0, len(v), 2)]
    return v[0]


def _float_quotients(ne, pv, cv):
    fcv = T.f32(cv)
    return T.f32(T.f32(T.ddiv(ne, fcv)) + T.f32(T.ddiv(pv, fcv + 1.0)))


def _mt_state_wrap_off_by_one(ring, idx):
    mt = [int(x) for x in ring]
    if idx >= 624 or idx == 0:
        return mt, 624
    for i in range(idx, 624):
        y = (mt[i] & 0x80000000) | (mt[(i + 1) % 623] & 0x7FFFFFFF)
        mt[i] = mt[(i + 397) % 624] ^ (y >> 1) ^ (0x9908B0DF if y & 1 else 0)
    return mt, idx


MUTATIONS = {
    "divide_by_N_not_float_N": ("selection", "_quot_divisor", float),
    "last_maximum_wins": ("selection", "_better", lambda u, best: u >= best and u != -math.inf),
    "float_quotients": ("selection", "_puct_sum", _float_quotients),
    "fmaxf_not_std_max": ("ingest", "_fmax", _fmaxf),
    "round_half_to_even": ("ingest", "_lround", _round_half_even),
    "pairwise_prior_sum": ("ingest", "_prior_sum", _pairwise_sum),
    "mt_ring_wrap_off_by_one": ("ingest", "_mt_state", _mt_state_wrap_off_by_one),
}


@pytest.fixture(scope="module")
def expected(gamma):
    return {"selection": selection_outputs(), "ingest": ingest_outputs(gamma)}


@pytest.mark.parametrize("name", sorted(MUTATIONS))
def test_constructed_cases_catch_the_mutation(monkeypatch, expected, gamma, name):
    part, attr, wrong = MUTATIONS[name]
    monkeypatch.setattr(T, attr, wrong)
    got = selection_outputs() if part == "selection" else ingest_outputs(gamma)
    changed = sum(a != b for a, b in zip(got, expected[part]))
    assert changed > 0, name


def test_slot_value_agrees_with_the_interval_reference():
    """slot_value with prior 1, denominator pv and v_sqrt 1 (so pvf = pv) equals the vectorised
    reference expression of test_puct_interval.py, including N above 2^24."""
    N, E, pv = samples()
    ref = reference(N, E, pv)
    idx = np.random.default_rng(3).choice(len(N), 20000, replace=False)
    for i in idx:
        s = [T.bits(E[i]), int(N[i]), 0, (1 << 7) | T.HAS]
        assert T.bits(T.slot_value(s, float(pv[i]), 1.0)) == T.bits(ref[i]), (int(N[i]), E[i], pv[i])
