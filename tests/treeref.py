"""Plain restatement of the reference's tree arithmetic (corintho_ai/cpp/src/trainmc.cpp), written
from the source and sharing no code with the CUDA kernels or the oracle:

  choose_next   TrainMC::chooseNext   trainmc.cpp:540-600  (PUCT selection at one node)
  receive_eval  TrainMC::receiveEval  trainmc.cpp:212-296  (prior ingest, Dirichlet noise, backup)

Doubles are Python floats; every float operation of the reference is done in double and rounded
once to float32 (exact for +, -, *, / of two floats). The record layout is the engine's
(tree.cuh): header[8] {cstate[4], n_legal | depth << 8, denominator bits, 0, 0}, then one slot
{evaluation bits, visits, child offset, move | prior << 7 | result << 16 | allv << 19 | has << 20
| child_n << 21} per legal move.

The small helpers (_quot_divisor, _puct_sum, _better, _fmax, _lround, _prior_sum, _mt_state) are
the places where a kernel could plausibly deviate; tests/test_treeref.py replaces each with a wrong
version and checks that the constructed cases notice.
"""
import math
import random
from fractions import Fraction

import numpy as np

NONE, LOSS, DRAW, WIN, DLOSS, DDRAW, DWIN = range(7)
ALLV, HAS = 1 << 19, 1 << 20


def f32(x):
    """double -> float, round to nearest even, overflow to inf."""
    with np.errstate(all="ignore"):
        return float(np.float32(x))


def bits(x):
    return int(np.array([x], np.float32).view(np.uint32)[0])


def from_bits(w):
    return float(np.array([w], np.uint32).view(np.float32)[0])


def ddiv(a, b):
    """IEEE double division (Python raises on a zero divisor)."""
    if b == 0.0:
        if a != a or a == 0.0:
            return math.nan
        return math.copysign(math.inf, a) * math.copysign(1.0, b)
    return a / b


# ---- chooseNext ---------------------------------------------------------------------------------
def v_sqrt(c_puct, visits):
    """float v_sqrt = c_puct * sqrt(visits): unqualified sqrt(float) is double sqrt(double)."""
    return f32(float(f32(c_puct)) * math.sqrt(float(f32(visits))))


def _quot_divisor(cv):
    """static_cast<float>(cv), the divisor of -E / N and (N + 1)."""
    return f32(cv)


def _puct_sum(ne, pv, cv):
    """-1.0 * E / float(cv) + pv / (float(cv) + 1.0): both quotients and the sum in double."""
    fcv = _quot_divisor(cv)
    return ddiv(ne, fcv) + ddiv(pv, fcv + 1.0)


def _better(u, best):
    """if (u > max_eval): the first maximum wins."""
    return u > best


def slot_value(slot, denominator, vs):
    """The float u of one slot (-inf = not selectable)."""
    e_bits, cv, _, w = (int(x) for x in slot)
    prob = f32(float((w >> 7) & 0x1FF) * denominator)
    pvf = f32(prob * vs)
    if not (w & HAS):
        return pvf
    cr = (w >> 16) & 7
    drawn = cr in (DRAW, DDRAW)
    if (cr != NONE and not drawn) or (w & ALLV):
        return -math.inf
    if drawn:
        return pvf
    cv = cv - (1 << 32) if cv >= 1 << 31 else cv
    return f32(_puct_sum(-1.0 * from_bits(e_bits), pvf, cv))


def choose_next(slots, denominator, c_puct, visits):
    """(chosen slot or -1, [u per slot]) for slots [n][4] of uint32 words."""
    vs = v_sqrt(c_puct, visits)
    best, choice, us = -math.inf, -1, []
    for e, s in enumerate(slots):
        u = slot_value(s, denominator, vs)
        us.append(u)
        if _better(u, best):
            best, choice = u, e
    return choice, us


def exact_value(slot, denominator, vs):
    """The real-number value of a visited slot's expression, for classifying cases."""
    e_bits, cv, _, w = (int(x) for x in slot)
    pvf = f32(f32(float((w >> 7) & 0x1FF) * denominator) * vs)
    fcv = Fraction(f32(cv))
    return -Fraction(from_bits(e_bits)) / fcv + Fraction(pvf) / (fcv + 1)


def near_midpoint(d, rel=2.0 ** -40):
    """True when the double d lies within rel * |d| of a point halfway between two floats."""
    if d == 0.0 or not math.isfinite(d) or not math.isfinite(f32(d)):
        return False
    x = np.float32(d)
    y = np.nextafter(x, np.float32(math.inf if Fraction(float(x)) <= Fraction(d) else -math.inf))
    mid = (Fraction(float(x)) + Fraction(float(y))) / 2
    return abs(Fraction(d) - mid) <= Fraction(rel) * abs(Fraction(d))


# ---- receiveEval --------------------------------------------------------------------------------
def _fmax(w, m):
    """std::max(w, max_prob) as the reference writes it: (w < m) ? m : w, so a NaN w is kept."""
    return m if w < m else w


def _lround(x):
    """(int)lround(x) on x86-64: half away from zero; NaN and out-of-range give LONG_MIN, and the
    cast to int keeps the low 32 bits."""
    if x != x or abs(x) >= 2.0 ** 63:
        q = -(1 << 63)
    else:
        q = int(math.floor(abs(x) + 0.5)) * (1 if x >= 0 else -1)
    q &= 0xFFFFFFFF
    return q - (1 << 32) if q >= 1 << 31 else q


def _prior_sum(values):
    """float sum += v in edge order."""
    s = 0.0
    for v in values:
        s = f32(s + v)
    return s


def _mt_state(ring, idx):
    """The engine keeps std::mt19937's state as a ring regenerated word by word as it is drawn
    (tree.cuh): words below idx are the current generation, the others the previous one. The
    equivalent std::mt19937 state finishes the block twist from idx on."""
    mt = [int(x) for x in ring]
    if idx >= 624 or idx == 0:
        return mt, 624
    for i in range(idx, 624):
        y = (mt[i] & 0x80000000) | (mt[(i + 1) % 624] & 0x7FFFFFFF)
        mt[i] = mt[(i + 397) % 624] ^ (y >> 1) ^ (0x9908B0DF if y & 1 else 0)
    return mt, idx


def _untemper(z):
    z ^= z >> 18
    z ^= (z << 15) & 0xEFC60000
    y = z
    for _ in range(5):
        y = z ^ ((y << 7) & 0x9D2C5680)
    y &= 0xFFFFFFFF
    x = y
    for _ in range(3):
        x = y ^ (x >> 11)
    return x & 0xFFFFFFFF


class MTRing:
    """std::mt19937 from Python's random module, reporting the state in the engine's ring form."""

    def __init__(self, ring, idx):
        mt, pos = _mt_state(ring, idx)
        self.ring = [int(x) for x in ring]
        self.idx = idx
        self.rng = random.Random()
        self.rng.setstate((3, tuple(mt) + (pos,), None))

    def next(self):
        z = self.rng.getrandbits(32)
        if self.idx >= 624:
            self.idx = 0
        self.ring[self.idx] = _untemper(z)
        self.idx += 1
        return z


def receive_eval(arena, pending, evals, probs, ring, mt_idx, root_eval, epsilon, gamma):
    """Returns (arena, root_eval, ring, mt_idx) after TrainMC::receiveEval.

    arena: uint32 words; pending: [(leaf_off, [path slot offsets, level 1 .. leaf])];
    evals [k]; probs [k][96] float32; gamma: the 1024 gamma samples of the Dirichlet draw."""
    a = [int(x) for x in arena]
    rng = MTRing(ring, mt_idx)
    eps = f32(epsilon)
    for i, (leaf, path) in enumerate(pending):
        n = a[leaf + 4] & 0xFF
        sl = [leaf + 8 + 4 * j for j in range(n)]
        filtered = [float(probs[i][a[s + 3] & 0x7F]) for s in sl]
        scalar = f32(ddiv(1.0, _prior_sum(filtered)) * f32(1.0 - eps))
        filtered = [f32(x * scalar) for x in filtered]
        dirichlet = [float(gamma[rng.next() % 1024]) for _ in sl]
        scalar = f32(ddiv(1.0, _prior_sum(dirichlet)) * eps)
        dirichlet = [f32(x * scalar) for x in dirichlet]
        weighted, max_prob = [], 0.0
        for x, y in zip(filtered, dirichlet):
            w = f32(x + y)
            weighted.append(w)
            max_prob = _fmax(w, max_prob)
        denom = f32(ddiv(511.0, max_prob))
        final_sum = 0
        for s, w in zip(sl, weighted):
            p = _lround(f32(w * denom))
            p = 1 if p < 1 else p
            a[s + 3] = (a[s + 3] & ~(0x1FF << 7)) | ((p & 0x1FF) << 7)
            final_sum = (final_sum + p + (1 << 31)) % (1 << 32) - (1 << 31)  # int, wraps on x86-64
        a[leaf + 5] = bits(f32(ddiv(1.0, f32(final_sum))))
        cur = float(evals[i])
        for s in reversed(path):
            a[s] = bits(f32(from_bits(a[s]) + f32(cur - 1.0)))
            a[s + 3] &= ~ALLV
            cur = cur * -1.0
        root_eval = f32(root_eval + f32(cur - 1.0))
    return np.array(a, np.uint32), root_eval, np.array(rng.ring, np.uint32), rng.idx
