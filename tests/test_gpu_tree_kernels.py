"""The tree search's arithmetic against tests/treeref.py, launched directly through
tests/tree_kernels.cu on constructed cases: PUCT selection (select_slot: screening pass, exact pass,
n > 64 slots, the c_puct * sqrt table and its absence), puct_u bit for bit, the screening interval
of puct_bounds with the hardware rcp.approx, fast_rcp's error bound, and receive_eval (priors,
Dirichlet noise, MT19937 ring, backup) on degenerate evaluator outputs."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import tree_cases as TC
import treeref as T

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PEND_WORDS = 66


@pytest.fixture(scope="session")
def tk(tmp_path_factory):
    """The harness, built with the library's flags into a temporary directory."""
    out = str(tmp_path_factory.mktemp("tree_kernels") / "libtree_kernels.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false",
                    "-Xcompiler", "-fPIC", "-shared", "-ccbin", "/usr/bin/g++", "-o", out,
                    os.path.join(ROOT, "tests", "tree_kernels.cu")], check=True, capture_output=True)
    L = C.CDLL(out)
    L.tk_last_error.restype = C.c_char_p
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_long
    L.tk_puct.argtypes = [i32] + [vp] * 8
    L.tk_rcp.argtypes = [i64, vp, C.c_double, vp]
    L.tk_select.argtypes = [i32, vp, i64, vp, vp, vp, vp, vp, vp]
    L.tk_ingest.argtypes = [vp, i64, vp, i32, vp, vp, i64, i64, i64, vp, vp, vp, C.c_float]
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def sel_cases():
    return TC.selection_cases()


def run_select(L, cases):
    words, offs = [], []
    pos = 0
    for c in cases:
        w = TC.record_words(c)
        offs.append(pos)
        words.append(w)
        pos += len(w)
    words = np.ascontiguousarray(np.concatenate(words), np.uint32)
    offs = np.array(offs, np.int32)
    vis = np.array([c["visits"] for c in cases], np.int32)
    cp = np.array([c["c_puct"] for c in cases], np.float32)
    tab = np.array([c["table"] for c in cases], np.int32)
    ch = np.full(len(cases), -7, np.int32)
    ex = np.full(len(cases), -7, np.int32)
    rc = L.tk_select(len(cases), _p(words), len(words), _p(offs), _p(vis), _p(cp), _p(tab), _p(ch), _p(ex))
    assert rc == 0, L.tk_last_error()
    return ch, ex


def run_puct(L, slots, den, vs):
    n = len(slots)
    slots = np.ascontiguousarray(slots, np.uint32)
    den, vs = np.ascontiguousarray(den, np.float32), np.ascontiguousarray(vs, np.float32)
    u, lo, hi = (np.full(n, np.nan, np.float32) for _ in range(3))
    inx, div = np.full(n, -1, np.int32), np.full(n, -1, np.int32)
    rc = L.tk_puct(n, _p(slots), _p(den), _p(vs), _p(u), _p(lo), _p(hi), _p(inx), _p(div))
    assert rc == 0, L.tk_last_error()
    return u, lo, hi, inx, div


@pytest.fixture(scope="module")
def per_slot(tk, sel_cases):
    """puct_u / puct_bounds on every slot of every constructed node, with the reference's float and
    the case each slot belongs to."""
    slots, den, vs, ref, case = [], [], [], [], []
    for k, c in enumerate(sel_cases):
        v = T.v_sqrt(c["c_puct"], c["visits"])
        for s in c["slots"]:
            slots.append(s)
            den.append(c["den"])
            vs.append(v)
            ref.append(T.f32(T.slot_value(s, c["den"], v) + 0.0))
            case.append(k)
    slots = np.array(slots, np.uint32)
    u, lo, hi, inx, div = run_puct(tk, slots, den, vs)
    return dict(slots=slots, ref=np.array(ref, np.float32), case=np.array(case), u=u, lo=lo, hi=hi, inx=inx, div=div)


def test_selection_equals_reference(tk, sel_cases, per_slot):
    """The chosen slot equals chooseNext's first maximum for every constructed node, and the cases
    reach the branches they were built for."""
    ch, ex = run_select(tk, sel_cases)
    bad = []
    n_exact = n_big = n_none = 0
    for k, c in enumerate(sel_cases):
        want, us = TC.ref_choice(c)
        if ch[k] != want:
            bad.append((k, len(c["slots"]), c["visits"], int(ch[k]), want))
        n = len(c["slots"])
        n_exact += int(ex[k] == 1)
        n_big += int(n > 64 and want >= 0)
        n_none += int(want < 0)
    # slots whose puct_u took the two divisions (ulo != uhi) in levels that went to the exact pass
    n_div = int(per_slot["div"][ex[per_slot["case"]] == 1].sum())
    assert not bad, f"{len(bad)} of {len(sel_cases)} cases differ, first {bad[:10]}"
    # coverage of the constructed suite (the counts are fixed by the seed)
    assert n_exact >= 300, n_exact
    assert n_div >= 100, n_div
    assert n_big >= 100, n_big
    assert n_none >= 10, n_none
    # a level with more than 64 slots always goes to the exact pass
    assert all(ex[k] == 1 for k, c in enumerate(sel_cases) if len(c["slots"]) > 64 and TC.ref_choice(c)[0] >= 0)
    print(f"selection: {len(sel_cases)} cases, exact pass {n_exact}, divided slots {n_div}, n > 64 {n_big}")


def test_puct_value_and_interval_per_slot(per_slot, sel_cases):
    """puct_u is bit-equal to the reference's float (up to -0.0 -> +0.0, which operator> cannot
    tell apart) and puct_bounds' [lo, hi] contains it, with the real rcp.approx.f32. A slot whose
    reference double lies within 2^-48 of a float rounding midpoint takes the divisions (the fast
    path's 2^-46 window straddles the midpoint)."""
    slots, ref, u, lo, hi = (per_slot[k] for k in ("slots", "ref", "u", "lo", "hi"))
    diff = np.nonzero(u.view(np.uint32) != ref.view(np.uint32))[0]
    assert len(diff) == 0, [(int(slots[i][1]), float(u[i]), float(ref[i])) for i in diff[:10]]
    assert np.all(lo <= ref) and np.all(ref <= hi)
    exact = per_slot["inx"] == 0
    assert np.all(lo[exact] == hi[exact])
    div = per_slot["div"] == 1
    n_mid = 0
    for i in np.nonzero(~exact)[0]:
        s = slots[i]
        if (int(s[3]) & T.ALLV) or ((int(s[3]) >> 16) & 7) != 0:
            continue
        c = sel_cases[per_slot["case"][i]]
        if T.near_midpoint(float(T.exact_value(s, c["den"], T.v_sqrt(c["c_puct"], c["visits"]))), 2.0 ** -48):
            n_mid += 1
            assert div[i], i
    assert n_mid >= 100 and int(div.sum()) >= n_mid, (n_mid, int(div.sum()))
    print(f"puct: {len(slots)} slots, {int((~exact).sum())} inexact intervals, {int(div.sum())} divided, "
          f"{n_mid} on a midpoint")


def test_interval_holds_with_hardware_rcp(tk):
    """The host proof of the screening bound (test_puct_interval.py) emulates rcp.approx; here the
    instruction itself, over N up to 2^31 - 1 and evaluations of every size and sign."""
    rng = np.random.default_rng(11)
    n = 1 << 20
    N = np.concatenate([rng.integers(1, 64, n // 4), rng.integers(1, 1 << 20, n // 4),
                        rng.integers(1 << 24, 1 << 31, n // 2)]).astype(np.int64)
    E = (rng.uniform(-1, 1, n) * N * rng.choice([1.0, 1e-3, 1e-7], n)).astype(np.float32)
    prior = rng.integers(1, 512, n)
    slots = np.zeros((n, 4), np.uint32)
    slots[:, 0] = E.view(np.uint32)
    slots[:, 1] = N.astype(np.uint32)
    slots[:, 3] = (prior << 7).astype(np.uint32) | T.HAS
    den = (1.0 / rng.integers(1, 5000, n)).astype(np.float32)
    vs = (rng.uniform(0, 1, n) ** 2 * rng.choice([1.0, 40.0, 1e-4], n)).astype(np.float32)
    u, lo, hi, inx, _ = run_puct(tk, slots, den, vs)
    assert inx.all()
    # the reference's float, vectorised: pvf = f32(f32(prior * den) * vs), double quotients by float(N)
    pvf = ((prior.astype(np.float32) * den).astype(np.float32) * vs).astype(np.float32).astype(np.float64)
    fn = N.astype(np.float32).astype(np.float64)
    ref = ((-E.astype(np.float64)) / fn + pvf / (fn + 1.0)).astype(np.float32)
    ref = (ref + np.float32(0.0)).astype(np.float32)
    assert np.all(lo <= ref) and np.all(ref <= hi)
    assert (u.view(np.uint32) == ref.view(np.uint32)).all()


@pytest.mark.parametrize("what", ["integers", "random"])
def test_fast_rcp_within_2_pow_minus_50(tk, what):
    """|fast_rcp(x) * x - 1| <= 2^-50: for every integer in [1, 2^24 + 2^20] in one launch and for
    random normal doubles. fl(r * x) is within 2^-52 of r * x and the subtraction is exact, so
    |fl(r * x) - 1| <= 2^-50 - 2^-52 proves the bound."""
    if what == "integers":
        n = (1 << 24) + (1 << 20)
        r = np.empty(n, np.float64)
        assert tk.tk_rcp(n, None, 1.0, _p(r)) == 0, tk.tk_last_error()
        x = np.arange(1, n + 1, dtype=np.float64)
    else:
        rng = np.random.default_rng(5)
        n = 1 << 22
        x = np.ldexp(rng.uniform(1.0, 2.0, n), rng.integers(-1000, 1000, n))
        r = np.empty(n, np.float64)
        assert tk.tk_rcp(n, _p(x), 0.0, _p(r)) == 0, tk.tk_last_error()
    err = np.abs(r * x - 1.0)
    assert err.max() <= 2.0 ** -50 - 2.0 ** -52, float(err.max())


@pytest.fixture(scope="module")
def gamma(oracle):
    return [float(oracle.gamma_sample(i)) for i in range(1024)]


def run_ingest(L, c, move_major):
    arena = np.ascontiguousarray(c["arena"].copy(), np.uint32)
    k = len(c["pending"])
    pend = np.zeros((max(k, 1), PEND_WORDS), np.uint32)
    for i, (leaf, path) in enumerate(c["pending"]):
        pend[i, 0] = leaf
        pend[i, 1] = len(path) | ((int(arena[leaf + 4]) & 0xFF) << 8)
        pend[i, 2:2 + len(path)] = path
    if move_major:
        probs = np.ascontiguousarray(c["probs"].T, np.float32)
        prs, pcs = 1, k
    else:
        probs = np.ascontiguousarray(c["probs"], np.float32)
        prs, pcs = 96, 1
    ring = np.ascontiguousarray(c["ring"].copy(), np.uint32)
    state = np.array([c["mt_idx"], 0], np.int32)
    root = np.array([c["root_eval"]], np.float32)
    ev = np.ascontiguousarray(c["evals"], np.float32)
    rc = L.tk_ingest(_p(arena), len(arena), _p(pend), k, _p(ev), _p(probs), probs.size, prs, pcs, _p(ring),
                     _p(state), _p(root), C.c_float(c["eps"]))
    assert rc == 0, L.tk_last_error()
    assert state[1] == 0
    return arena, float(root[0]), ring, int(state[0])


def test_ingest_equals_reference(tk, gamma):
    """Every arena word, the root evaluation, the MT ring and its index bit-equal to receiveEval's
    for every constructed game, with the row-major and the move-major probability layouts."""
    cases = TC.ingest_cases()
    bad = []
    for k, c in enumerate(cases):
        want = T.receive_eval(c["arena"], c["pending"], c["evals"], c["probs"], c["ring"], c["mt_idx"],
                              c["root_eval"], c["eps"], gamma)
        got = run_ingest(tk, c, move_major=bool(k % 2))
        if not ((got[0] == want[0]).all() and T.bits(got[1]) == T.bits(want[1]) and (got[2] == want[2]).all()
                and got[3] == want[3]):
            w = np.nonzero(got[0] != want[0])[0]
            bad.append((k, [len(p) for _, p in c["pending"]][:3], c["eps"], c["mt_idx"], w[:5].tolist(),
                        got[1], want[1], int((got[2] != want[2]).sum()), got[3], want[3]))
    assert not bad, f"{len(bad)} of {len(cases)} games differ, first {bad[:5]}"
