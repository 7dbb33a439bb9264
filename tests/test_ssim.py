"""SSIM on the device (csrc/hevce_ssim.h, run by hevce_ssim_kernel and hevce_ssim_mean_kernel) on the CPU:
tests/sim/hevce_simssim.cpp runs the kernels' own functions in their order, and the result must equal the host SSIM of
tools/hevc_eval.py (scikit-image's defaults, data_range 256) between the coded picture and the measured plane."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import simutil as S
import test_decode as TD

sys.path.insert(0, os.path.join(S.ROOT, "tools"))
import hevc_eval  # noqa: E402

_u8p = ctypes.POINTER(ctypes.c_ubyte)
SHAPES = [(32, 32), (45, 70), (64, 1000), (333, 222), (100, 33)]
KINDS = ("smooth", "noise", "flat", "checker")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("simssim") / "libhevce_simssim.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", *S.variant_flags("g7"), "-I", S.CSRC, "-o", so,
                    os.path.join(S.SIM_DIR, "hevce_simssim.cpp")], check=True)
    L = ctypes.CDLL(so)
    L.hevce_simssim.restype = ctypes.c_int
    return L


def padded(v, max_dim=8192):
    return (min(v, max_dim) + 31) // 32 * 32


def coded(src, max_dim=8192):
    """The sample the encoder reads at each padded position: src[min(y, src_h - 1)][min(x, src_w - 1)]."""
    h, w = src.shape
    ys = np.minimum(np.arange(padded(h, max_dim)), h - 1)
    xs = np.minimum(np.arange(padded(w, max_dim)), w - 1)
    return src[np.ix_(ys, xs)]


def run(L, srcs, planes, order=0):
    n = len(srcs)
    srcs = [np.ascontiguousarray(s, dtype=np.uint8) for s in srcs]
    planes = [np.ascontiguousarray(p, dtype=np.uint8) for p in planes]
    arr = lambda xs: (_u8p * n)(*[x.ctypes.data_as(_u8p) for x in xs])
    ints = lambda xs: (ctypes.c_int * n)(*[int(x) for x in xs])
    out = np.zeros(n, np.float64)
    rc = L.hevce_simssim(n, arr(srcs), ints([s.shape[0] for s in srcs]), ints([s.shape[1] for s in srcs]), arr(planes),
                         ints([p.shape[0] for p in planes]), ints([p.shape[1] for p in planes]),
                         out.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), int(order))
    assert rc == 0
    return out


def perturb(rng, plane, q):
    """A plane with qpd6-like damage: coarser quantisation of 8x8 block means and more noise at higher q."""
    p = plane.astype(np.int64)
    if q >= 2:
        h, w = p.shape
        step = 2 << q
        b = p.reshape(h // 8, 8, w // 8, 8)
        m = b.mean(axis=(1, 3), keepdims=True)
        p = (np.round(m / step) * step + (b - m) * (1.0 - 0.15 * q)).reshape(h, w)
    p = p + rng.normal(0, 0.5 + q, p.shape)
    return np.clip(np.round(p), 0, 255).astype(np.uint8)


def batch(seed):
    rng = np.random.default_rng(seed)
    srcs, planes = [], []
    for k, (h, w) in enumerate(SHAPES * 2):
        src = TD.random_picture(rng, h, w, KINDS[(k + seed) % 4])
        srcs.append(src)
        planes.append(perturb(rng, coded(src), (k + seed) % 5))
    return srcs, planes


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_matches_host_ssim(harness, seed):
    srcs, planes = batch(seed)
    got = run(harness, srcs, planes)
    for i, (s, p) in enumerate(zip(srcs, planes)):
        assert coded(s).shape == p.shape
        if s.shape == p.shape:
            assert np.array_equal(coded(s), s)
        else:
            assert np.array_equal(coded(s), hevc_eval.image_pad(s))
        want = hevc_eval.ssim(coded(s), p)
        assert abs(got[i] - want) <= 1e-10, (i, s.shape, got[i], want)


def test_identical_planes_give_one(harness):
    rng = np.random.default_rng(5)
    srcs = [TD.random_picture(rng, h, w, KINDS[k % 4]) for k, (h, w) in enumerate(SHAPES)]
    got = run(harness, srcs, [coded(s) for s in srcs])
    assert got.tolist() == [1.0] * len(srcs)


def test_block_order_is_bit_identical(harness):
    srcs, planes = batch(7)
    a, b = run(harness, srcs, planes, 0), run(harness, srcs, planes, 1)
    assert a.tobytes() == b.tobytes()
    one = [run(harness, [s], [p])[0] for s, p in zip(srcs, planes)]     # a picture's value does not depend on its batch
    assert np.array(one).tobytes() == a.tobytes()


def test_picture_above_a_lowered_size_limit(harness):
    """A picture larger than max_dim: the coded picture is the clamped crop, padded at the right / bottom only where the
    crop is not a multiple of 32."""
    rng = np.random.default_rng(9)
    src = TD.random_picture(rng, 300, 170, "smooth")
    max_dim = 200
    c = coded(src, max_dim)
    assert c.shape == (224, 192)
    assert np.array_equal(c[:224, :170], src[:224, :170]) and np.array_equal(c[:, 170:], np.repeat(src[:224, 169:170], 22, axis=1))
    plane = perturb(rng, c, 3)
    (got,) = run(harness, [src], [plane])
    assert abs(got - hevc_eval.ssim(c, plane)) <= 1e-10
