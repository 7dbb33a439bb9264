"""The device deblocking filter (csrc/hevce_deblock.h, run by hevce_deblock_kernel) on the CPU: tests/sim/hevce_simdeblock.cpp
runs the kernel's own functions over whole pictures in the kernel's phase order, and the result must equal the numpy
model of the filter (tests/deblock_model.py) exactly, and libavcodec's decoding of simulator-encoded streams."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import decode_util as U
import deblock_model as D
import simutil as S
import test_conformance as TC

_u8p = ctypes.POINTER(ctypes.c_ubyte)


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("simdeblock") / "libhevce_simdeblock.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", *S.variant_flags("g7"), "-I", S.CSRC, "-o", so,
                    os.path.join(S.SIM_DIR, "hevce_simdeblock.cpp")], check=True)
    L = ctypes.CDLL(so)
    L.hevce_simdeblock.restype = ctypes.c_int
    return L


def run(L, rcons, parts, qs, order=0):
    """Decoded pictures of padded reconstructions rcons with partitions [(cu_size, kind)] at qpd6 qs."""
    n = len(rcons)
    rcons = [np.ascontiguousarray(r, dtype=np.uint8) for r in rcons]
    cus = [np.ascontiguousarray(c, dtype=np.uint8) for c, _ in parts]
    kinds = [np.ascontiguousarray(k, dtype=np.uint8) for _, k in parts]
    decs = [np.full(r.shape, 0xEE, np.uint8) for r in rcons]
    arr = lambda xs: (_u8p * n)(*[x.ctypes.data_as(_u8p) for x in xs])
    ints = lambda xs: (ctypes.c_int * n)(*[int(x) for x in xs])
    rc = L.hevce_simdeblock(n, arr(rcons), arr(cus), arr(kinds), ints([r.shape[0] for r in rcons]), ints([r.shape[1] for r in rcons]),
                            ints(qs), arr(decs), int(order))
    assert rc == 0
    return decs


def random_partition(rng, h, w):
    """A valid partition: per CTU a random 32/16/8 quadtree; kind 0 or 1 per CU, and NxN (2) only at 8x8."""
    cu, kind = np.zeros((h // 4, w // 4), np.uint8), np.zeros((h // 8, w // 8), np.uint8)

    def node(y, x, s):
        if s > 8 and rng.random() < 0.6:
            for dy in (0, s // 2):
                for dx in (0, s // 2):
                    node(y + dy, x + dx, s // 2)
            return
        cu[y // 4:(y + s) // 4, x // 4:(x + s) // 4] = s
        kind[y // 8:(y + s) // 8, x // 8:(x + s) // 8] = rng.integers(0, 3 if s == 8 else 2)

    for y in range(0, h, 32):
        for x in range(0, w, 32):
            node(y, x, 32)
    return cu, kind


def random_picture(rng, h, w, smooth):
    if not smooth:
        return rng.integers(0, 256, (h, w)).astype(np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    base = 110 + 50 * np.sin(xx / 11.0 + rng.random() * 6) + 40 * np.cos(yy / 9.0)
    blocks = rng.integers(-6, 7, (h // 8 + 1, w // 8 + 1)).repeat(8, 0).repeat(8, 1)[:h, :w]   # steps on the 8x8 grid
    return np.clip(base + blocks + rng.integers(-1, 2, (h, w)), 0, 255).astype(np.uint8)


SIZES = [(32, 32), (64, 32), (32, 96), (64, 96), (128, 160), (160, 224)]   # 64x96 = a 45x70 source after padding


@pytest.mark.parametrize("q", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("size", SIZES, ids=[f"{h}x{w}" for h, w in SIZES])
def test_equals_model_on_random_partitions(harness, size, q):
    h, w = size
    rng = np.random.default_rng(1000 * q + h + w)
    rcons, parts = [], []
    for k in range(6):
        rcons.append(random_picture(rng, h, w, smooth=k % 2 == 1))
        parts.append(random_partition(rng, h, w))
    decs = run(harness, rcons, parts, [q] * len(rcons))
    for k, (r, (cu, kind), d) in enumerate(zip(rcons, parts, decs)):
        assert np.array_equal(d, D.deblock(r, cu, kind, q)), (size, q, k)
        if q <= 1:
            assert np.array_equal(d, r)                  # beta = tc = 0: the decoded picture is the reconstruction


def test_filter_changes_pictures():
    """The model comparison above is not vacuous: at qpd6 2-4 the filter moves samples of smooth pictures."""
    rng = np.random.default_rng(4)
    r = random_picture(rng, 128, 160, smooth=True)
    cu, kind = random_partition(rng, 128, 160)
    assert all((D.deblock(r, cu, kind, q) != r).mean() > 0.01 for q in (2, 3, 4))


def test_mixed_batch_and_item_order(harness):
    """One launch with pictures of different sizes and qpd6, run with every phase's items in both orders."""
    rng = np.random.default_rng(77)
    shapes = [(64, 96), (32, 32), (128, 160), (32, 96), (96, 64), (64, 32), (160, 224), (64, 96)]
    qs = [4, 2, 0, 3, 1, 4, 2, 3]
    rcons = [random_picture(rng, h, w, smooth=i % 3 != 0) for i, (h, w) in enumerate(shapes)]
    parts = [random_partition(rng, h, w) for h, w in shapes]
    fwd = run(harness, rcons, parts, qs)
    rev = run(harness, rcons, parts, qs, order=1)
    for i, (r, (cu, kind), q) in enumerate(zip(rcons, parts, qs)):
        want = D.deblock(r, cu, kind, q)
        assert np.array_equal(fwd[i], want), i
        assert np.array_equal(rev[i], want), i


@pytest.mark.parametrize("q", [0, 1, 2, 3, 4])
def test_equals_decoder_on_simulator_streams(harness, q):
    """The five pictures of test_conformance.py, encoded by the simulator: the harness output is what libavcodec decodes."""
    n = 0
    for name, img in TC.pictures().items():
        s, r, err = S.sim_encode(img, q)
        assert err == 0
        luma = U.decode_luma(s, r.shape)
        if luma is None:
            pytest.skip("no HEVC decoder in this OpenCV build")
        cu, _, kind = S.sim_last_partition(r.shape)
        (dec,) = run(harness, [r], [(cu, kind)], [q])
        assert np.array_equal(dec, luma), (name, q)
        if q <= 1:
            assert np.array_equal(dec, r), name
        n += 1
    assert n == 5
