"""How HEVCImageEncoderBatch splits a batch, on the CPU: csrc/hevce_api.c, unmodified, linked with a stand-in for the CUDA
layer (tests/sim/hevce_apistub.c) that logs every hevce_session_configure call.  No kernel, CUDA runtime or GPU is
involved.  The tables pin today's shards and chunks: a change of the planner shows up as an edit of this file."""
import ctypes
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hevc-image-encoder-lite_b200", "csrc")
STUB = os.path.join(ROOT, "tests", "sim", "hevce_apistub.c")
ERR_CUDA, ERR_STATE = -2, -3
CALLER_DEVICE = 5   # the caller's current device; no call below runs on it, so its restoration is visible


@pytest.fixture(scope="module")
def api(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("apistub") / "libhevce_apistub.so")
    subprocess.run(["gcc", "-O2", "-Wall", "-fPIC", "-shared", "-pthread", "-I", CSRC, "-o", so,
                    os.path.join(CSRC, "hevce_api.c"), STUB], check=True)
    return ctypes.CDLL(so)


def run(L, sizes, ndev=1, max_dim=8192, fail_configure=0, fail_download=0, fail_code=0):
    """One HEVCImageEncoderBatch call over `ndev` stub devices.  Returns the return code, the sorted configure calls
    (device, first picture, count, variant, max_ctas, max_dim), the sizes written back and the stream lengths."""
    n = len(sizes)
    L.apistub_reset(ndev, fail_configure, fail_download, fail_code)
    assert L.hevce_set_devices(ndev, (ctypes.c_int * ndev)(*range(ndev))) == 0
    L.hevce_set_max_dim(max_dim)
    ys = (ctypes.c_int * n)(*[h for h, _ in sizes])
    xs = (ctypes.c_int * n)(*[w for _, w in sizes])
    qs = (ctypes.c_int * n)(*[2] * n)
    lens = (ctypes.c_int * n)(*[-1] * n)
    dummy = (ctypes.c_void_p * n)(*[1] * n)   # never dereferenced by the stub
    L.apistub_set_base(ys)
    L.hevce_internal_set_device(CALLER_DEVICE)
    rc = L.HEVCImageEncoderBatch(n, dummy, dummy, dummy, ys, xs, qs, lens)
    assert L.hevce_internal_get_device() == CALLER_DEVICE
    rows = (ctypes.c_longlong * (6 * 4096))()
    m = L.apistub_calls(rows, 4096)
    assert m <= 4096
    calls = sorted(tuple(rows[6 * i:6 * i + 6]) for i in range(m))
    return rc, calls, list(zip(ys, xs)), list(lens)


P = (512, 768)   # the default bench picture, 768x512
CASES = {
    # same-size shards below 8 x 7 pictures run as one chunk
    "55_same": ([P] * 55, 1, 8192, [(0, 0, 55, 1, 0, 8192)]),
    # same-size shards: four chunks of a multiple of 7 pictures; max_ctas = a quarter of the SMs above one g7 wave
    "56_same": ([P] * 56, 1, 8192, [(0, 0, 14, 2, 0, 8192), (0, 14, 14, 2, 0, 8192), (0, 28, 14, 2, 0, 8192), (0, 42, 14, 2, 0, 8192)]),
    "1036_same": ([P] * 1036, 1, 8192, [(0, 0, 259, 4, 0, 8192), (0, 259, 259, 4, 0, 8192), (0, 518, 259, 4, 0, 8192),
                                        (0, 777, 259, 4, 0, 8192)]),
    "1037_same": ([P] * 1037, 1, 8192, [(0, 0, 266, 5, 37, 8192), (0, 266, 266, 5, 37, 8192), (0, 532, 266, 5, 37, 8192),
                                        (0, 798, 239, 5, 37, 8192)]),
    "8192_same": ([P] * 8192, 1, 8192, [(0, 0, 2051, 2, 37, 8192), (0, 2051, 2051, 2, 37, 8192), (0, 4102, 2051, 2, 37, 8192),
                                        (0, 6153, 2039, 2, 37, 8192)]),
    "64_4k": ([(2160, 3840)] * 64, 1, 8192, [(0, 0, 21, 4, 0, 8192), (0, 21, 21, 4, 0, 8192), (0, 42, 21, 4, 0, 8192),
                                             (0, 63, 1, 4, 0, 8192)]),
    "70000_tiny": ([(32, 32)] * 70000, 1, 8192, [(0, 0, 17500, 4, 37, 8192), (0, 17500, 17500, 4, 37, 8192),
                                                 (0, 35000, 17500, 4, 37, 8192), (0, 52500, 17500, 4, 37, 8192)]),
    # ragged shards: chunks of at most 768 Mpixel and 32768 pictures
    "5000_alternating": ([P if i % 2 else P[::-1] for i in range(5000)], 1, 8192,
                         [(0, 0, 2048, 2, 0, 8192), (0, 2048, 2048, 2, 0, 8192), (0, 4096, 904, 2, 0, 8192)]),
    "85_ragged": ([s for s in [(32, 32), (64, 64), (45, 70), (33, 97), (96, 64), (64, 128)] for _ in range(14)] + [(8, 8)], 1, 8192,
                  [(0, 0, 85, 1, 0, 8192)]),
    # a picture over the size limit is clamped
    "xl_limit_8192": ([(11993, 15991)], 1, 8192, [(0, 0, 1, 1, 0, 8192)]),
    "xl_limit_16384": ([(11993, 15991)], 1, 16384, [(0, 0, 1, 1, 0, 16384)]),
    # several devices: contiguous shards of equal padded pixels, each with its own variant
    "2072_same_2dev": ([P] * 2072, 2, 8192, [(0, 0, 259, 4, 0, 8192), (0, 259, 259, 4, 0, 8192), (0, 518, 259, 4, 0, 8192),
                                             (0, 777, 259, 4, 0, 8192), (1, 1036, 259, 5, 0, 8192), (1, 1295, 259, 5, 0, 8192),
                                             (1, 1554, 259, 5, 0, 8192), (1, 1813, 259, 5, 0, 8192)]),
    "10_ragged_3dev": ([(32 * (1 + i % 5), 64) for i in range(10)], 3, 8192,
                       [(0, 0, 4, 4, 0, 8192), (1, 4, 4, 5, 0, 8192), (2, 8, 2, 4, 0, 8192)]),
}


@pytest.mark.parametrize("case", list(CASES))
def test_chunk_plan(api, case):
    sizes, ndev, max_dim, want = CASES[case]
    rc, calls, sizes_out, lens = run(api, sizes, ndev, max_dim)
    assert rc == 0
    assert calls == want
    pad = lambda v: (min(v, max_dim) + 31) // 32 * 32
    assert sizes_out == [(pad(h), pad(w)) for h, w in sizes]
    assert lens == list(range(len(sizes)))   # every picture downloaded once, by the chunk that holds it


def test_size_write_back_of_clamped_pictures(api):
    assert run(api, [(11993, 15991)], max_dim=8192)[2] == [(8192, 8192)]
    assert run(api, [(11993, 15991)], max_dim=16384)[2] == [(12000, 16000)]


@pytest.mark.parametrize("ndev,where,code", [(1, "configure", ERR_CUDA), (1, "download", ERR_STATE), (2, "configure", ERR_STATE)])
def test_injected_failure(api, ndev, where, code):
    """A failed chunk fails the call with its code and leaves the caller's sizes as they were."""
    sizes = [P] * 2072
    rc, calls, sizes_out, _ = run(api, sizes, ndev, **{f"fail_{where}": 2, "fail_code": code})
    assert rc == code
    assert sizes_out == sizes
    assert 2 <= len(calls) <= 8
