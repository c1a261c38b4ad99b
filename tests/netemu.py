"""Emulation of the tensor-core network (corintho_ai_b200/csrc/mlp_tc.cuh) in its own arithmetic.

`upload` restates net_tc_upload: weights rounded to nearest-even bf16 or fp16 (bf16x3: plus a lo
image bf16(w - bf16(w))), the bias split into hi = r(b) and lo = r(b - hi) on the two constant-one
activation columns 100 / 101 (bf16x3: a third part bf16(b - hi - lo) in the lo image), and unit
weights that keep the ones columns alive. `forward` restates tc_forward: 16-bit operands, the
hidden epilogue ReLU + 16-bit round (bf16x3: activation lo = bf16(relu(x) - hi), products
a_hi*w_hi + a_hi*w_lo + a_lo*w_hi), tanh of column 0 and a softmax over columns 1..96.

Sums are taken in float64. Where every product term is a multiple of 2^g and the terms add up to
less than 2^(24+g) in magnitude, every partial sum is an fp32 number, so the tensor core's fp32
accumulator holds the exact sum whatever its order: those outputs are exact. Elsewhere the
accumulator may differ from the exact sum by a few fp32 ulps of sum|terms|; a row is flagged
ambiguous when such a difference could change a hidden 16-bit rounding.

`mutant` switches on one deliberate error (MUTANTS), so that tests can show the probe networks
would catch it."""
import numpy as np

MODES = {"bf16": 0, "fp16": 1, "bf16x3": 2}
MUTANTS = ("no_bias_lo", "no_bias_lo2", "no_alo_whi", "no_ahi_wlo", "fp16_as_bf16", "ones_dead",
           "policy_shift")
DIMS = [70] + [100] * 12 + [97]
ONES = 100      # activation columns 100 and 101 are constant 1
WIDTH = 102     # activation columns the emulation keeps: 100 hidden + the two ones columns
HEAD = 98       # head columns emulated: value, 96 logits and one padding column (zero)
FP16_MAX = 65504.0


def bf16(x):
    """float32 -> nearest-even bf16, returned as float32 (x finite)."""
    b = np.ascontiguousarray(x, np.float32).view(np.uint32)
    b = (b + np.uint32(0x7FFF) + ((b >> np.uint32(16)) & np.uint32(1))) & np.uint32(0xFFFF0000)
    return b.view(np.float32)


def fp16(x, saturate=False):
    """float32 -> nearest-even fp16 (subnormals included), returned as float32. Out of range
    rounds to inf, or to +-65504 with saturate (cvt.rn.satfinite)."""
    with np.errstate(over="ignore"):
        h = np.asarray(x, np.float32).astype(np.float16).astype(np.float32)
    if saturate:
        h = np.where(np.isinf(h) & np.isfinite(x), np.copysign(np.float32(FP16_MAX), h), h)
    return h


def _rounder(mode, mutant, saturate=False):
    if mode == 1 and mutant != "fp16_as_bf16":
        return lambda x: fp16(x, saturate)
    return bf16


def upload(flat, mode, mutant=None):
    """Per layer (hi, lo) operand matrices [WIDTH, out] in float64, as net_tc_upload builds them
    (lo is None outside bf16x3). Rows 0..99 multiply the activations, rows 100/101 the ones."""
    mode = MODES.get(mode, mode)
    r = _rounder(mode, mutant)
    flat = np.asarray(flat, np.float32)
    layers, off = [], 0
    for l in range(13):
        K, N = DIMS[l], DIMS[l + 1]
        ncol = WIDTH if l < 12 else HEAD
        w = flat[off:off + K * N].reshape(K, N)
        off += K * N
        b = flat[off:off + N]
        off += N
        hi = np.zeros((WIDTH, ncol), np.float32)
        lo = np.zeros((WIDTH, ncol), np.float32) if mode == 2 else None
        hi[:K, :N] = r(w)
        if mode == 2:
            lo[:K, :N] = bf16(w - hi[:K, :N])  # w - bf16(w) is exact in fp32
        bh = r(b)
        bl = r(b - bh)
        hi[ONES, :N] = bh
        if mutant != "no_bias_lo":
            hi[ONES + 1, :N] = bl
        if mode == 2 and mutant != "no_bias_lo2":
            lo[ONES, :N] = bf16((b - bh) - bl)
        if l < 12 and mutant != "ones_dead":
            hi[ONES, ONES] = hi[ONES, ONES + 1] = 1.0
        layers.append((hi.astype(np.float64), None if lo is None else lo.astype(np.float64)))
    return layers


def _lowbit(x):
    """Exponent of the lowest set bit of each float64 (a large number for zeros, a very negative one
    for inf / NaN, which no sum holds exactly)."""
    x = np.asarray(x, np.float64)
    fin = np.isfinite(x)
    m, e = np.frexp(np.where(fin, np.abs(x), 1.0))
    mi = (m * 2.0 ** 53).astype(np.int64)
    low = mi & -mi
    lb = e - 53 + np.log2(np.maximum(low, 1)).astype(np.int64)
    return np.where(x == 0, 10 ** 6, np.where(fin, lb, -10 ** 6))


def _terms(a_parts, w_parts, mode, mutant):
    """(operand a, operand w) pairs of the MMAs of one layer."""
    (ah, al), (wh, wl) = a_parts, w_parts
    pairs = [(ah, wh)]
    if mode == 2:
        if mutant != "no_ahi_wlo":
            pairs.append((ah, wl))
        if mutant != "no_alo_whi":
            pairs.append((al, wh))
    return pairs


def _epilogue(x32, mode, r):
    """Hidden epilogue on fp32 accumulators: (hi, lo) activation operands."""
    h = r(np.maximum(x32, np.float32(0)))
    lo = bf16(np.maximum(x32, np.float32(0)) - h) if mode == 2 else np.zeros_like(h)
    return h, lo


def forward(layers, x, mode, mutant=None, saturate=True, ulps=16):
    """Emulated outputs for encoded positions x [rows, 70].

    Returns (value, probs, logits, ambiguous): value = tanh(column 0) and probs = softmax of
    columns 1..96 in float64 from the fp32 head accumulators `logits` [rows, HEAD]; ambiguous[row]
    is True where some hidden pre-activation is not provably exact in fp32 and lies within
    `ulps` fp32 ulps of sum|terms| of a point where its 16-bit rounding changes."""
    mode = MODES.get(mode, mode)
    r = _rounder(mode, mutant, saturate)
    x = np.asarray(x, np.float32)
    rows = x.shape[0]
    ah = np.zeros((rows, WIDTH), np.float32)
    ah[:, :70] = x   # 0/1 and k/4: exact in every 16-bit format
    ah[:, ONES:ONES + 2] = 1.0
    al = np.zeros_like(ah)
    ambiguous = np.zeros(rows, bool)
    for l, (wh, wl) in enumerate(layers):
        pairs = _terms((ah.astype(np.float64), al.astype(np.float64)), (wh, wl), mode, mutant)
        with np.errstate(invalid="ignore", over="ignore"):
            acc = sum(a @ w for a, w in pairs)
            mag = sum(np.abs(a) @ np.abs(w) for a, w in pairs)
        # lowest bit any term can have: activations x weights, and the ones columns x bias parts
        g = np.full(acc.shape, 10 ** 6, np.int64)
        for a, w in pairs:
            la = _lowbit(a[:, :ONES]).min(1)
            lw = _lowbit(w[:ONES]).min(0)
            lb = _lowbit(w[ONES:]).min(0)
            g = np.minimum(g, np.minimum(la[:, None] + lw[None, :], lb[None, :]))
        exact = (mag < np.ldexp(1.0, np.minimum(24 + g, 1000))) | (mag == 0)
        err = np.where(exact, 0.0, mag * (ulps * 2.0 ** -24))
        with np.errstate(over="ignore", invalid="ignore"):
            x32 = acc.astype(np.float32)
        if l == len(layers) - 1:
            logits = x32
            break
        ah, al = _epilogue(x32, mode, r)
        with np.errstate(over="ignore", invalid="ignore"):
            dn = _epilogue((acc - err).astype(np.float32), mode, r)
            up = _epilogue((acc + err).astype(np.float32), mode, r)
        flip = (dn[0] != up[0]) | (dn[1] != up[1])
        ambiguous |= (flip & ~exact).any(1)
    z = logits.astype(np.float64)
    value = np.tanh(z[:, 0])
    pol = z[:, 2:98] if mutant == "policy_shift" else z[:, 1:97]
    with np.errstate(invalid="ignore", over="ignore"):
        e = np.exp(pol - pol.max(1, keepdims=True))
        probs = e / e.sum(1, keepdims=True)
    return value, probs, logits, ambiguous


def recovered(value, probs, ref=None):
    """Layer outputs recovered from what the network returns: atanh(value) and, per row,
    log p_j - log p_ref (ref = the most likely move unless given). Returns (values [rows, 97], ref)."""
    value = np.asarray(value, np.float64)
    probs = np.asarray(probs, np.float64)
    if ref is None:
        ref = probs.argmax(1)
    with np.errstate(divide="ignore", invalid="ignore"):
        lp = np.log(probs)
        out = np.empty((probs.shape[0], 97))
        out[:, 0] = np.arctanh(np.clip(value, -1.0, 1.0))
        out[:, 1:] = lp - lp[np.arange(len(ref)), ref][:, None]
    return out, ref
