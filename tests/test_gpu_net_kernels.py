"""Every network kernel form (k_mlp_tc two-tile, k_mlp_tc1 single-tile, k_mlp_f32) in every
operand mode, launched directly through tests/net_kernels.cu: forced grids of 1, 2 and 3 CTAs and
the natural grid, tail sizes around the 128-row tile and the 256-row pair, a device-side row count
below n_max, a leading dimension larger than the batch, and the zero2 counter reset."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import corintho_ai_b200 as cb
from test_gpu_net_modes import sample_positions

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRECISION = {"fp32": 0, "bf16": 1, "fp16": 2, "bf16x3": 3}
FORMS = {"tc": 0, "tc1": 1, "f32": 2}
CASES = [("tc", p) for p in ("bf16", "fp16", "bf16x3")] + [("tc1", p) for p in ("bf16", "fp16", "bf16x3")] \
    + [("f32", "fp32")]
SIZES = (1, 127, 128, 129, 255, 256, 257, 3 * 256 + 1, 7 * 128 + 5)
SENTINEL = np.array([0x7FC0DEAD], np.uint32).view(np.float32)[0]   # a NaN no kernel writes


@pytest.fixture(scope="session")
def nk(tmp_path_factory):
    """The harness, built with the library's flags into a temporary directory."""
    out = str(tmp_path_factory.mktemp("net_kernels") / "libnet_kernels.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false",
                    "-Xcompiler", "-fPIC", "-shared", "-ccbin", "/usr/bin/g++", "-o", out,
                    os.path.join(ROOT, "tests", "net_kernels.cu")], check=True, capture_output=True)
    L = C.CDLL(out)
    L.nk_last_error.restype = C.c_char_p
    L.nk_upload.argtypes = [C.c_void_p, C.c_int]
    L.nk_run.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                         C.c_void_p, C.c_void_p, C.c_void_p]
    return L


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def upload(L, flat, precision):
    w = np.ascontiguousarray(flat, np.float32)
    assert L.nk_upload(_ptr(w), PRECISION[precision]) == 0, L.nk_last_error()


def run(L, form, x, n_max=None, count=-1, grid=0, ld=None):
    """eval [n_max], probs (move-major [96][ld] or row-major [n_max][96]) and zero2 after one launch,
    every buffer pre-filled with SENTINEL / 7."""
    x = np.ascontiguousarray(x, np.float32)
    n = x.shape[0]
    n_max = n if n_max is None else n_max
    ld = n_max if ld is None else ld
    ev = np.full(n_max, SENTINEL, np.float32)
    pr = np.full(n_max * 96 if form == "f32" else 96 * ld, SENTINEL, np.float32)
    z2 = np.full(4, 7, np.int32)
    rc = L.nk_run(FORMS[form], _ptr(x), n, n_max, n, count, grid, ld, _ptr(ev), _ptr(pr), _ptr(z2))
    assert rc == 0, L.nk_last_error()
    return ev, pr, z2


def row_major(form, pr, rows, ld):
    return pr.reshape(-1, 96)[:rows] if form == "f32" else pr.reshape(96, ld)[:, :rows].T


def _trained_flat():
    return np.load(os.path.join(ROOT, "tests", "golden", "trained_net.npz"))["flat"]


@pytest.fixture(scope="module")
def rows(oracle):
    return sample_positions(oracle, 1024, seed=13)


@pytest.mark.parametrize("form,precision", CASES)
def test_every_grid_and_tail_equals_evaluate(nk, rows, form, precision):
    """Byte-identical to Trainer.evaluate for every batch size and grid: single- and two-tile
    forms agree, a CTA that loops over several tiles or pairs computes what one CTA per tile does,
    and a row's result does not depend on the batch around it."""
    flat = _trained_flat()
    t = cb.Trainer(64, "", 1, 32, 16)
    t.set_weights(flat, 0, precision)
    ref_e, ref_p = t.evaluate(rows)
    upload(nk, flat, precision)
    for n in SIZES:
        for grid in (1, 2, 3, 0):
            ev, pr, z2 = run(nk, form, rows[:n], grid=grid)
            p = row_major(form, pr, n, n)
            assert ev.tobytes() == ref_e[:n].tobytes(), (n, grid)
            assert np.ascontiguousarray(p).tobytes() == ref_p[:n].tobytes(), (n, grid)
            assert list(z2) == [0, 7, 0, 7]


@pytest.mark.parametrize("form,precision", CASES)
def test_device_count_below_n_max_leaves_the_rest_untouched(nk, rows, form, precision):
    """The row count read on the device (as the fused loop launches) below n_max, and ld > n_max:
    rows from n to n_max and the gaps of the [96][ld] layout keep their sentinel."""
    flat = _trained_flat()
    t = cb.Trainer(64, "", 1, 32, 16)
    t.set_weights(flat, 0, precision)
    ref_e, ref_p = t.evaluate(rows)
    upload(nk, flat, precision)
    n_max, ld = 700, 901
    for n in (0, 1, 129, 300, 513, 700):
        for grid in (1, 3, 0):
            ev, pr, z2 = run(nk, form, rows[:n], n_max=n_max, count=n, grid=grid, ld=ld)
            assert list(z2) == [0, 7, 0, 7]
            assert ev[:n].tobytes() == ref_e[:n].tobytes()
            assert ev[n:].view(np.uint32).tolist() == [SENTINEL.view(np.uint32)] * (n_max - n)
            if form == "f32":
                full = pr.reshape(n_max, 96)
                live, rest = full[:n], full[n:]
            else:
                full = pr.reshape(96, ld)
                live, rest = full[:, :n].T, full[:, n:]
            assert np.ascontiguousarray(live).tobytes() == ref_p[:n].tobytes(), (n, grid)
            assert (rest.view(np.uint32) == SENTINEL.view(np.uint32)).all(), (n, grid)
