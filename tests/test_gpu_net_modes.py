"""Every tensor-core operand mode (bf16, fp16, bf16x3) against an emulation of its own arithmetic
(netemu.py), one layer slot at a time.

A probe network for slot L has random layers at L and, when L > 0, at L - 1 (so that layer L
receives activations that are not 16-bit numbers and their lo parts take part); every other layer
is an exact identity (unit diagonal, zero bias, head column j = hidden column j), which passes
values unchanged in every mode. The random operands lie on coarse binary grids and their terms
sum to less than 2^24 grid steps, so the tensor core's fp32 accumulator holds exact sums in any
order and the kernel must equal the emulation up to the head's __expf / tanhf / normalisation.
The layer outputs are recovered from the probabilities as log p_j - log p_ref and from the value
as atanh(v).

Operand parts the probes make visible: weights with 9 significant bits (bf16 rounding, bf16x3 lo
image), activations into layer L with up to 10 (bf16 rounding, bf16x3 activation lo), biases of
full fp32 precision built as hi + lo + third part with |lo| near a quarter and |third| near
2^-11, so that the bias lo part and the bf16x3 third part each move the recovered logits far
more than the tolerance (test_probes_catch_every_mutant, CPU only)."""
import numpy as np
import pytest

import corintho_ai_b200 as cb
import netemu
from netemu import DIMS, MUTANTS, recovered

TOL = 4e-6          # on recovered logits (|spread| <= 16) and atanh(value) (|value| <= tanh(1.5))
SLOTS = range(13)
MODES = ("bf16", "fp16", "bf16x3")


def sample_positions(oracle, n, seed=1):
    rng = np.random.default_rng(seed)
    rows = []
    while len(rows) < n:
        st = oracle.start()
        for _ in range(40):
            rows.append(oracle.encode(st))
            mask, _ = oracle.legal(st)
            ids = [m for m in range(96) if (mask[m >> 5] >> (m & 31)) & 1]
            if not ids:
                break
            st = oracle.do_move(st, int(rng.choice(ids)))
    return np.stack(rows[:n]).astype(np.float32)


def _layers_identity():
    out = []
    for l in range(13):
        K, N = DIMS[l], DIMS[l + 1]
        w = np.zeros((K, N), np.float64)
        d = min(K, N)
        w[np.arange(d), np.arange(d)] = 1.0
        out.append([w, np.zeros(N, np.float64)])
    return out


def _probe_bias(rng, n):
    """Biases hi + lo + third with hi in [64.5, 68) (bf16), |lo| in [1/8, 1/4) (8 bits), |third|
    in [48, 64) * 2^-17: each part survives the split and moves the output."""
    hi = 64.0 + rng.integers(1, 8, n) / 2.0
    lo = rng.choice([-1.0, 1.0], n) * rng.integers(128, 256, n) * 2.0 ** -10
    t = rng.choice([-1.0, 1.0], n) * rng.integers(48, 64, n) * 2.0 ** -17
    return hi + lo + t


def probe_flat(slot, seed=0):
    """C-ABI weight vector of the probe network for `slot` (0..12)."""
    rng = np.random.default_rng(1000 * seed + slot)
    L = _layers_identity()
    if slot > 0:  # layer slot-1: quarter-step weights on the 0 / 1 / k/4 inputs, outputs on 1/16
        K, N = DIMS[slot - 1], DIMS[slot]
        L[slot - 1] = [rng.integers(-12, 13, (K, N)) / 4.0, rng.integers(64, 385, N) / 16.0]
    K, N = DIMS[slot], DIMS[slot + 1]
    w = rng.integers(-383, 384, (K, N)) * 2.0 ** -13 * (rng.random((K, N)) < 0.125)
    w[:, 0] = rng.integers(-63, 64, K) * 2.0 ** -13 * (rng.random(K) < 0.25)  # the value column stays small
    b = _probe_bias(rng, N)
    b[0] = rng.integers(2 ** 15, 3 * 2 ** 15) * 2.0 ** -17  # in [0.25, 0.75), 17 bits
    L[slot] = [w, b]
    flat = np.concatenate([np.concatenate([w.ravel(), b]) for w, b in L]).astype(np.float32)
    assert flat.size == cb.WEIGHT_FLOATS
    assert np.array_equal(flat.astype(np.float64), np.concatenate([np.concatenate([w.ravel(), b]) for w, b in L]))
    return flat


def range_probe_flat():
    """fp16 range probe: layer 0 column 3 = 60000 + 30000 * (sum of the six piece-count inputs),
    which exceeds 65504 on any position with a piece in hand; layer 1 scales column 3 by 2^-12."""
    L = _layers_identity()
    L[0][0][64:70, 3] = 30000.0
    L[0][1][3] = 60000.0
    L[1][0][3, 3] = 2.0 ** -12
    return np.concatenate([np.concatenate([w.ravel(), b]) for w, b in L]).astype(np.float32)


def emulate(flat, x, mode, mutant=None, saturate=True):
    return netemu.forward(netemu.upload(flat, mode, mutant), x, mode, mutant, saturate)


# ---- CPU: the emulation, the probes and their power ---------------------------------------------

@pytest.fixture(scope="module")
def positions(oracle):
    return sample_positions(oracle, 2000, seed=5)


def test_emulation_matches_the_plain_network_on_identity_layers(positions):
    """An all-identity network passes the encoded input through unchanged in every mode."""
    flat = np.concatenate([np.concatenate([w.ravel(), b]) for w, b in _layers_identity()]).astype(np.float32)
    x = positions[:300]
    for mode in MODES:
        v, p, z, amb = emulate(flat, x, mode)
        assert not amb.any()
        assert np.array_equal(z[:, :70], x) and not z[:, 70:97].any()


def test_probes_are_exact_and_well_conditioned(positions):
    """No probe row is ambiguous, recovered values stay where the tolerance applies, and every
    hidden value stays in fp16 range."""
    x = positions[:500]
    for slot in SLOTS:
        flat = probe_flat(slot)
        for mode in MODES:
            v, p, z, amb = emulate(flat, x, mode)
            assert not amb.any(), (slot, mode)
            pol = z[:, 1:97].astype(np.float64)
            assert (pol.max(1) - pol.min(1)).max() <= 16.0, (slot, mode)
            assert np.abs(z[:, 0]).max() <= 1.5, (slot, mode)
            assert np.isfinite(p).all()


def test_ambiguity_flag_marks_only_inexact_sums(positions):
    """Deep random networks (Glorot, not on a grid) do have sums that fp32 may round either way;
    with no accumulation error allowed nothing is flagged, so the flag comes from inexact sums."""
    flat = cb.fold_batchnorm(cb.random_weights(3))
    for mode in MODES:
        layers = netemu.upload(flat, mode)
        assert netemu.forward(layers, positions[:300], mode)[3].any(), mode
        assert not netemu.forward(layers, positions[:300], mode, ulps=0)[3].any(), mode


def test_probes_catch_every_mutant(positions):
    """Each deliberate error in the emulation moves the recovered outputs of some probe by more
    than 100 times the GPU tolerance: a kernel with that error would fail the GPU test."""
    x = positions[:200]
    worst = {m: 0.0 for m in MUTANTS}
    for slot in SLOTS:
        flat = probe_flat(slot)
        for mode in MODES:
            v, p, _, _ = emulate(flat, x, mode)
            ref_vals, ref = recovered(v, p)
            for m in MUTANTS:
                if m in ("no_bias_lo2", "no_alo_whi", "no_ahi_wlo") and mode != "bf16x3":
                    continue
                if m == "fp16_as_bf16" and mode != "fp16":
                    continue
                vm, pm, _, _ = emulate(flat, x, mode, m)
                got, _ = recovered(vm, pm, ref)
                with np.errstate(invalid="ignore"):
                    d = np.abs(got - ref_vals)
                d = np.where(np.isnan(d), np.inf, d)
                worst[m] = max(worst[m], float(d.max()))
    print("largest change of a recovered output per mutant:", worst)
    for m in MUTANTS:
        assert worst[m] > 100 * TOL, (m, worst[m])


def test_fp16_range_probe_needs_saturation(positions):
    """Past 65504 a plain fp16 round gives +inf and the next layer turns it into NaN on every
    output; with satfinite conversions the value stops at 65504."""
    x = positions[:200]
    flat = range_probe_flat()
    assert (x[:, 64:70].sum(1) > 0).all()
    v, p, z, _ = emulate(flat, x, "fp16", saturate=False)
    assert np.isnan(z).all()
    v, p, z, _ = emulate(flat, x, "fp16")
    assert np.isfinite(z).all() and (z[:, 3] == np.float32(FP16_SCALED)).all()


FP16_SCALED = 65504.0 * 2.0 ** -12


# ---- GPU: the kernels against the emulation -----------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_every_layer_slot_equals_the_emulation(positions, mode):
    """All 13 slots: on every row not flagged ambiguous the kernel's recovered layer outputs equal
    the emulation's to TOL; fewer than 1 % of rows are flagged."""
    t = cb.Trainer(128, "", 1, 32, 16)
    x = positions
    for slot in SLOTS:
        flat = probe_flat(slot)
        t.set_weights(flat, 0, mode)
        ev, pr = t.evaluate(x)
        v, p, _, amb = emulate(flat, x, mode)
        assert amb.mean() < 0.01, (slot, amb.mean())
        want, ref = recovered(v, p)
        got, _ = recovered(ev, pr, ref)
        d = np.abs(got - want)[~amb]
        assert np.isfinite(d).all() and d.max() <= TOL, (slot, float(np.nanmax(d)))


@pytest.mark.gpu
def test_fp16_saturates_instead_of_spreading_nan(positions):
    x = positions[:500]
    flat = range_probe_flat()
    t = cb.Trainer(64, "", 1, 32, 16)
    t.set_weights(flat, 0, "fp16")
    ev, pr = t.evaluate(x)
    assert np.isfinite(ev).all() and np.isfinite(pr).all()
    v, p, _, amb = emulate(flat, x, "fp16")
    want, ref = recovered(v, p)
    got, _ = recovered(ev, pr, ref)
    assert not amb.any() and np.abs(got - want).max() <= TOL


@pytest.mark.gpu
@pytest.mark.parametrize("precision,rows", [("bf16", 80000), ("fp16", 80000), ("bf16x3", 40000), ("fp32", 20000)])
def test_evaluate_past_one_pass_of_the_grid(oracle, precision, rows):
    """More rows than one pass of the network grid covers (75 776 for the two-tile bf16 / fp16
    kernel, 37 888 for bf16x3, 18 944 for the fp32 kernel): every CTA runs a second tile pair,
    and each row must be what it is in a batch of 1 000."""
    base = sample_positions(oracle, 4000, seed=9)
    x = base[np.random.default_rng(2).integers(0, len(base), rows)]
    flat = cb.fold_batchnorm(cb.random_weights(17))
    t = cb.Trainer(rows // 16, "", 1, 32, 16)
    t.set_weights(flat, 0, precision)
    ev, pr = t.evaluate(x)
    for r0 in range(0, rows, 1000):
        e, p = t.evaluate(x[r0:r0 + 1000])
        assert e.tobytes() == ev[r0:r0 + 1000].tobytes() and p.tobytes() == pr[r0:r0 + 1000].tobytes(), r0
