"""Host check of the interval screening used by the game step's PUCT selection
(corintho_ai_b200/csrc/tree.cuh, puct_bounds): for visited children the float expression
-E*rcp(N) + pv*rcp(N+1) with a 1-ulp reciprocal must stay within 2^-20*(|a|+|b|) of the reference's
float(-E/float(N) + pv/(float(N) + 1.0)) in double (trainmc.cpp:540-600). The reciprocal of the hardware
(rcp.approx.f32, <= 1 ulp) is emulated by the correctly rounded one and both of its neighbours, so
every value it may return is covered."""
import numpy as np


def samples():
    """visits up to 2^20 and from 2^24 to 2^31 - 1 (where float(N) != N), evaluation sums of any sign
    up to the visit count, small and large priors"""
    rng = np.random.default_rng(7)
    n = 400_000
    N = np.concatenate([rng.integers(1, 64, n // 2), rng.integers(1, 1 << 20, n // 2),
                        rng.integers(1 << 24, 1 << 31, n // 2)]).astype(np.int64)
    n = len(N)
    E = (rng.uniform(-1, 1, n) * N * rng.choice([1.0, 1e-3, 1e-7], n)).astype(np.float32)
    pv = (rng.uniform(0, 1, n) ** 3 * rng.choice([1.0, 40.0, 1e-4], n)).astype(np.float32)
    return N, E, pv


def reference(N, E, pv):
    """float(-E / float(N) + pv / (float(N) + 1.0)), quotients and sum in double"""
    fn = N.astype(np.float32).astype(np.float64)
    return ((-E.astype(np.float64)) / fn + pv.astype(np.float64) / (fn + 1.0)).astype(np.float32)


def test_interval_contains_reference_value():
    N, E, pv = samples()
    ref = reference(N, E, pv)
    fn = N.astype(np.float32)
    fn1 = (fn + np.float32(1.0)).astype(np.float32)
    worst = 0.0
    for da in (-1, 0, 1):
        ra = (np.float32(1.0) / fn).astype(np.float32)
        ra = np.nextafter(ra, np.float32(np.inf) * da) if da else ra
        for db in (-1, 0, 1):
            rb = (np.float32(1.0) / fn1).astype(np.float32)
            rb = np.nextafter(rb, np.float32(np.inf) * db) if db else rb
            a = ((-E) * ra).astype(np.float32)
            b = (pv * rb).astype(np.float32)
            u = (a + b).astype(np.float32)
            d = ((np.abs(a) + np.abs(b)).astype(np.float32) * np.float32(2.0 ** -20)).astype(np.float32)
            lo, hi = (u - d).astype(np.float32), (u + d).astype(np.float32)
            assert np.all(lo <= ref) and np.all(ref <= hi)
            s = (np.abs(a) + np.abs(b)).astype(np.float64)
            ok = s > 0
            worst = max(worst, float(np.max(np.abs(u.astype(np.float64) - ref.astype(np.float64))[ok] / s[ok])))
    # the bound has the margin claimed in DESIGN.md (worst observed error well under 2^-20)
    assert worst < 2.0 ** -21.5
