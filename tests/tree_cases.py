"""Constructed, seeded inputs for the tree search's selection and prior ingest, shared by the GPU
comparison (test_gpu_tree_kernels.py) and the CPU check that the reference restatement tells right
from wrong on them (test_treeref.py)."""
import math

import numpy as np

import treeref as T

HAS, ALLV = T.HAS, T.ALLV
NS = (1, 2, 31, 32, 33, 63, 64, 65, 95, 96)
VISITS = (1, 2047, 2048, 2049, 2 ** 24 - 1, 2 ** 24, 2 ** 24 + 1, 2 ** 30)
BIG_N = (1, 2 ** 20, 2 ** 24 - 1, 2 ** 24, 2 ** 24 + 1, 2 ** 24 + 3, 2 ** 27 + 5, 2 ** 31 - 1)
C_PUCT = (1.0, 3.0, 0.7)
WINNER_SLOTS = (0, 31, 32, 63, 64, 95)


def w3(move, prior=0, result=0, allv=False, has=False, cn=0):
    return (move & 0x7F) | (prior << 7) | (result << 16) | (ALLV if allv else 0) | (HAS if has else 0) | (cn << 21)


def slot(move, prior, E=0.0, N=0, result=0, allv=False, has=None):
    has = N > 0 if has is None else has
    return [T.bits(E), N, 0, w3(move, prior, result, allv, has, 20 if has else 0)]


def node_case(slots, den, visits=1, c_puct=1.0, table=True):
    return dict(slots=np.array(slots, np.uint32).reshape(-1, 4), den=T.f32(den), visits=visits,
                c_puct=T.f32(c_puct), table=bool(table))


def record_words(case):
    s = case["slots"]
    head = np.array([0, 0, 0, 0, len(s), T.bits(case["den"]), 0, 0], np.uint32)
    return np.concatenate([head, s.reshape(-1)])


def ref_choice(case):
    return T.choose_next(case["slots"], case["den"], case["c_puct"], case["visits"])


def solve_E(target, N, pvf):
    """A float E whose slot value f32(-E / float(N) + pvf / (float(N) + 1)) equals target, or the
    closest one found (searching float neighbours of the real-number solution)."""
    fn = T.f32(N)
    e0 = np.float32((pvf / (fn + 1.0) - target) * fn)
    best = None
    for d in range(-64, 65):
        E = float(e0)
        step = np.float32(math.inf if d > 0 else -math.inf)
        x = e0
        for _ in range(abs(d)):
            x = np.nextafter(x, step)
        E = float(x)
        u = T.f32(T.ddiv(-E, fn) + T.ddiv(pvf, fn + 1.0))
        err = abs(u - target)
        if best is None or err < best[0]:
            best = (err, E)
        if err == 0.0:
            break
    return best[1]


def _ulp_step(x, k):
    y = np.float32(x)
    for _ in range(abs(k)):
        y = np.nextafter(y, np.float32(math.inf if k > 0 else -math.inf))
    return float(y)


def selection_cases(seed=2024):
    rng = np.random.default_rng(seed)
    cases = []

    def rnd_slot(m, N_choices, den):
        kind = rng.integers(0, 8)
        prior = int(rng.integers(1, 512))
        if kind <= 2:
            return slot(m, prior)
        if kind == 3:  # decided or pending children
            return slot(m, prior, 0.5, 3, result=int(rng.choice([1, 3, 4, 6])), allv=bool(rng.integers(0, 2)))
        if kind == 4:  # drawn, with or without visits
            return slot(m, prior, 0.0, int(rng.integers(0, 3)), result=int(rng.choice([2, 5])), has=True)
        N = int(rng.choice(N_choices))
        E = float(np.float32(rng.uniform(-1, 1) * N * rng.choice([1.0, 0.3, 1e-3])))
        return slot(m, prior, E, N)

    # grid: n x visits x c_puct x table, random slot classes, N from BIG_N
    for n in NS:
        for visits in VISITS:
            for cp in C_PUCT:
                for table in (True, False):
                    den = 1.0 / float(rng.integers(n, 512 * n))
                    cases.append(node_case([rnd_slot(m, BIG_N, den) for m in range(n)], den, visits, cp, table))
    # equal priors; the winner at a chosen slot: earlier slots unselectable or worse, later ones tie
    for win in WINNER_SLOTS:
        for n in (win + 1, 96):
            for variant in range(3):
                den, vis, cp = 1.0 / 96, int(rng.choice([1, 100, 5000])), float(rng.choice(C_PUCT))
                pvf = T.f32(T.f32(7.0 * den) * T.v_sqrt(cp, vis))
                sl = []
                for m in range(n):
                    if m < win:
                        sl.append(slot(m, 7, 0.25, 4, result=1) if m % 3 == 0 else
                                  slot(m, 7, 2.0, 3, allv=True) if m % 3 == 1 else
                                  slot(m, 7, solve_E(_ulp_step(pvf, -1 - variant), 9, pvf), 9))
                    elif m == win or variant == 0:
                        sl.append(slot(m, 7))
                    else:  # a visited slot whose value equals the unvisited pvf exactly
                        N = int(rng.choice([3, 40, 2 ** 20, 2 ** 24 + 1, 2 ** 27 + 5]))
                        sl.append(slot(m, 7, solve_E(pvf, N, pvf), N) if m % 2 else slot(m, 7))
                cases.append(node_case(sl, den, vis, cp, bool(rng.integers(0, 2))))
    # ties and near-ties between visited (inexact) and unvisited or drawn (exact) slots
    for n in NS:
        for rep in range(12):
            den = 1.0 / float(rng.integers(50, 5000))
            vis = int(rng.choice(VISITS + (3, 77)))
            cp = float(rng.choice(C_PUCT))
            vs = T.v_sqrt(cp, vis)
            sl = [slot(m, int(rng.integers(1, 200))) for m in range(n)]
            pb = int(rng.integers(200, 512))
            target = T.f32(T.f32(pb * den) * vs)
            pos = sorted(rng.choice(n, size=min(n, 4), replace=False).tolist())
            sl[pos[-1]] = slot(pos[-1], pb, result=int(rng.choice([0, 2, 5])), N=0, has=bool(rep % 2))
            if sl[pos[-1]][3] & HAS and ((sl[pos[-1]][3] >> 16) & 7) == 0:
                sl[pos[-1]] = slot(pos[-1], pb)
            for q, p in enumerate(pos[:-1]):
                N = int(rng.choice(BIG_N[1:] + (2, 5, 1000)))
                pr = int(rng.integers(1, 512))
                pvf = T.f32(T.f32(pr * den) * vs)
                t = _ulp_step(target, (0, 1, -1)[(rep + q) % 3])
                sl[p] = slot(p, pr, solve_E(t, N, pvf), N)
            cases.append(node_case(sl, den, vis, cp, bool(rep % 3)))
    # values on a float rounding midpoint: N = 2^k - 1 (float(N) + 1 = 2^k), E = -q * N, pvf =
    # (2j + 1) * 2^(k - 24) with v_sqrt = 1, so -E/N + pvf/(N+1) = q + (2j + 1) * 2^-24 exactly
    for k in (2, 5, 11, 17, 23):
        N = 2 ** k - 1
        for q in (1.0, 1.5, -2.0):
            for n in (3, 40, 70, 96):
                den = 2.0 ** (k - 24)
                sl = []
                for m in range(n):
                    j = int(rng.integers(0, 3))
                    if m % 5 == 4:
                        sl.append(slot(m, 2 * j + 1))
                    else:
                        sl.append(slot(m, 2 * j + 1, -q * N, N))
                        # a neighbour a hair above or below the midpoint (E one ulp away)
                        if m % 7 == 3:
                            sl[-1] = slot(m, 2 * j + 1, _ulp_step(-q * N, 1 if m % 2 else -1), N)
                cases.append(node_case(sl, den, 1, 1.0, bool(m % 2)))
    # E = +-0 and +-N, cur_visits = 0 (every pvf is +0), a node with no selectable slot
    for n in (1, 33, 65, 96):
        for E in (0.0, -0.0, 1.0, -1.0):
            for vis in (0, 1, 2048):
                sl = []
                for m in range(n):
                    N = int(rng.choice([1, 7, 2 ** 24 + 1]))
                    sl.append(slot(m, int(rng.integers(1, 512)), E * N if E != 0.0 else E, N) if m % 2 else
                              slot(m, int(rng.integers(1, 512))))
                cases.append(node_case(sl, 1.0 / 300, vis, 1.0, vis != 2048))
        cases.append(node_case([slot(m, 5, 1.0, 2, result=int(rng.choice([1, 3, 4, 6])), allv=bool(m % 2))
                                for m in range(n)], 0.01, 10, 1.0, True))
    # every class of {has, allv, result}
    for has in (False, True):
        for allv in (False, True):
            for res in range(7):
                for n in (1, 40, 96):
                    sl = [slot(m, 9, 0.5, 2 if has else 0, result=res, allv=allv, has=has) for m in range(n)]
                    cases.append(node_case(sl, 1.0 / 64, 5, 1.0, True))
    return cases


# ---- prior ingest -----------------------------------------------------------------------------
def _leaf_record(moves):
    n = len(moves)
    head = [0, 0, 0, 0, n | (3 << 8), 0, 0, 0]
    body = []
    for m in moves:
        body += [0, 0, 0, int(m)]
    return head + body


def ingest_case(rng, leaf_sizes, prob_kind, eps, mt_idx, plens, evals=None, shared=True):
    """One game: a chain of interior records (the paths), then one fresh record per leaf."""
    words = []
    # interior nodes: depth up to 64, 3 slots each, slot e of level L: leaves share prefixes
    depth = max(plens) if plens else 0
    chain = []  # chain[L][b] = slot offset of branch b at level L
    for L in range(depth):
        off = len(words)
        rec = [0, 0, 0, 0, 3 | (L << 8), T.bits(1.0 / 3), 0, 0]
        for b in range(3):
            E = float(np.float32(rng.choice([1e8, -1e8, 1.0, 0.5, -3.0])))
            rec += [T.bits(E), int(rng.integers(1, 100)), 0, w3(b, 100, has=True, allv=True)]
        words += rec
        chain.append([off + 8 + 4 * b for b in range(3)])
    pending = []
    for i, n in enumerate(leaf_sizes):
        moves = np.sort(rng.choice(96, size=n, replace=False))
        off = len(words)
        words += _leaf_record(moves)
        pl = plens[i % len(plens)] if plens else 0
        path = [chain[L][(0 if shared and (L < pl // 2) else int(rng.integers(0, 3)))] for L in range(pl)]
        pending.append((off, path))
    k = len(leaf_sizes)
    probs = np.zeros((k, 96), np.float32)
    for i, (off, _) in enumerate(pending):
        n = words[off + 4] & 0xFF
        mv = [words[off + 8 + 4 * j + 3] & 0x7F for j in range(n)]
        kind = prob_kind if prob_kind != "mixed" else ("equal", "some_zero", "all_zero", "subnormal", "huge",
                                                        "inf", "random", "halves")[i % 8]
        if kind == "equal":
            v = np.full(n, 1.0 / 96)
        elif kind == "some_zero":
            v = rng.uniform(0, 1, n) * (rng.uniform(0, 1, n) < 0.5)
        elif kind == "all_zero":
            v = np.zeros(n)
            probs[i, [m for m in range(96) if m not in set(mv)][:1]] = 1.0  # one-hot on an illegal move
        elif kind == "subnormal":
            v = rng.integers(0, 50, n) * 2.0 ** -149
        elif kind == "huge":
            v = rng.uniform(0.5, 1.0, n) * 3e38
        elif kind == "halves":
            v = halves_probs(rng, n)
            if n > 16:  # tails that an edge-order sum drops and a pairwise sum keeps
                v[-8:] = 2.0 ** -26
        elif kind == "inf":  # an infinite probability: NaN among finite weights after scaling by 0
            v = rng.uniform(0, 1, n)
            v[rng.integers(0, n)] = np.inf
        else:
            v = rng.uniform(0, 1, n) ** 3
        probs[i, mv] = v.astype(np.float32)
    ev = evals if evals is not None else rng.choice([1.0, -1.0, 0.0, -0.0, 0.3, -0.7], k)
    ring = rng.integers(0, 2 ** 32, 624, dtype=np.uint64).astype(np.uint32)
    return dict(arena=np.array(words, np.uint32), pending=pending, evals=np.array(ev, np.float32), probs=probs,
                ring=ring, mt_idx=mt_idx, root_eval=T.f32(rng.choice([0.0, 5.0, -1e8])), eps=T.f32(eps))


def halves_probs(rng, n):
    """Probabilities whose quantisation value w * (511 / max) is an exact half for most slots when
    epsilon is 0: numerators 511 and j + 0.5 that add up to a power of two 2^K, over 2^K, so that
    the normalisation, the maximum and 511 / max are all exact."""
    nums = np.concatenate([[511.0], rng.integers(0, 300, n - 1) + 0.5])
    if (n - 1) % 2:
        nums[-1] -= 0.5
    D = 2.0 ** math.ceil(math.log2(nums.sum())) - nums.sum()
    for j in range(1, n):
        add = min(D, math.floor(510.5 - nums[j]))
        nums[j] += add
        D -= add
    return nums / nums.sum()


def ingest_cases(seed=77):
    rng = np.random.default_rng(seed)
    cases = []
    for sizes in ([5], [31] * 31, [1] * 32, [3] * 33, [7] * 64, [2] * 96, [96], [48] * 9 + [40] * 3,
                  [20] * 22 + [30] * 2, [10] * 44 + [96]):
        for kind in ("equal", "some_zero", "all_zero", "subnormal", "huge", "inf", "halves", "random", "mixed"):
            for eps in (0.0, 0.25, 1.0):
                mt = int(rng.choice([0, 600, 623, 624]))
                plens = [int(x) for x in rng.choice([1, 2, 5, 17, 40, 64], 3)]
                cases.append(ingest_case(rng, sizes, kind, eps, mt, plens))
    # path lengths 0 .. 64 with deltas of very different size, so the order of additions shows
    for mt in (0, 600, 623, 624):
        for pl in (0, 1, 2, 3, 4, 5, 8, 31, 63, 64):
            cases.append(ingest_case(rng, [4] * 40, "random", 0.25, mt, [pl, max(pl - 1, 0), pl],
                                     evals=rng.choice([1.0, -1.0, 0.0, -0.0, 1e8, -1e8], 40)))
    return cases
