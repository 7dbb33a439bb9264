"""HEVCImageEncoderBatchDecoded on the CPU: csrc/hevce_api.c, unmodified, linked with the stand-in for the CUDA layer
(tests/sim/hevce_apistub.c) and a stand-in for the two decoded-picture calls (tests/sim/hevce_apistub_decoded.c).
The decoded entry point must split a batch exactly as HEVCImageEncoderBatch does and hand every picture's decoded
buffer to exactly one hevce_session_download_decoded, after a hevce_session_deblock of its chunk.  No kernel, CUDA
runtime or GPU is involved."""
import ctypes
import os
import subprocess

import pytest

import test_host_api as HA

STUB_DECODED = os.path.join(HA.ROOT, "tests", "sim", "hevce_apistub_decoded.c")
ERR_ARG, ERR_CUDA, ERR_STATE = -1, -2, -3
DEC_BASE, DEC_STEP = 1 << 20, 16   # fake decoded-buffer addresses: picture i gets DEC_BASE + DEC_STEP * i


@pytest.fixture(scope="module")
def api(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("apistub_dec") / "libhevce_apistub.so")
    subprocess.run(["gcc", "-O2", "-Wall", "-fPIC", "-shared", "-pthread", "-I", HA.CSRC, "-o", so,
                    os.path.join(HA.CSRC, "hevce_api.c"), HA.STUB, STUB_DECODED], check=True)
    return ctypes.CDLL(so, mode=os.RTLD_NOW)


def run(L, sizes, ndev=1, decoded=True, decs="all", fail_deblock=0, fail_download_decoded=0, fail_configure=0, fail_code=0):
    """One batch call over `ndev` stub devices.  Returns the return code, the sorted configure calls, the sorted
    (device, picture, decoded buffer) log of hevce_session_download_decoded, the number of hevce_session_deblock calls
    and the sizes written back."""
    n = len(sizes)
    L.apistub_reset(ndev, fail_configure, 0, fail_code)
    L.apistub_decoded_reset(fail_deblock, fail_download_decoded, fail_code)
    assert L.hevce_set_devices(ndev, (ctypes.c_int * ndev)(*range(ndev))) == 0
    L.hevce_set_max_dim(8192)
    ys = (ctypes.c_int * n)(*[h for h, _ in sizes])
    xs = (ctypes.c_int * n)(*[w for _, w in sizes])
    qs = (ctypes.c_int * n)(*[2] * n)
    lens = (ctypes.c_int * n)(*[-1] * n)
    dummy = (ctypes.c_void_p * n)(*[1] * n)   # never dereferenced by the stub
    L.apistub_set_base(ys)
    L.apistub_decoded_set_base(ys)
    L.hevce_internal_set_device(HA.CALLER_DEVICE)
    if not decoded:
        rc = L.HEVCImageEncoderBatch(n, dummy, dummy, dummy, ys, xs, qs, lens)
    else:
        ptrs = [DEC_BASE + DEC_STEP * i for i in range(n)]
        if decs == "null_entry":
            ptrs[n // 2] = None
        arr = None if decs == "null" else (ctypes.c_void_p * n)(*ptrs)
        rc = L.HEVCImageEncoderBatchDecoded(n, dummy, dummy, dummy, arr, ys, xs, qs, lens)
    assert L.hevce_internal_get_device() == HA.CALLER_DEVICE
    rows = (ctypes.c_longlong * (6 * 4096))()
    m = L.apistub_calls(rows, 4096)
    calls = sorted(tuple(rows[6 * i:6 * i + 6]) for i in range(m))
    drows = (ctypes.c_longlong * (3 * 65536))()
    k = L.apistub_decoded_log(drows, 65536)
    assert k <= 65536
    dlog = sorted(tuple(drows[3 * i:3 * i + 3]) for i in range(k))
    return rc, calls, dlog, L.apistub_deblocks(), list(zip(ys, xs))


CASES = ["56_same", "1036_same", "85_ragged", "2072_same_2dev", "10_ragged_3dev"]


@pytest.mark.parametrize("case", CASES)
def test_same_split_and_one_download_per_picture(api, case):
    sizes, ndev, _, want = HA.CASES[case]
    rc0, calls0, dlog0, ndeb0, sizes0 = run(api, sizes, ndev, decoded=False)
    rc, calls, dlog, ndeb, sizes_out = run(api, sizes, ndev)
    assert rc0 == rc == 0
    assert calls0 == calls == want                   # the split of the batch did not move
    assert dlog0 == [] and ndeb0 == 0                # HEVCImageEncoderBatch never asks for decoded pictures
    assert sizes_out == sizes0
    assert ndeb == len(calls)                        # one deblock per chunk
    assert [p for _, p, _ in dlog] == list(range(len(sizes)))            # every picture once
    assert all(ptr == DEC_BASE + DEC_STEP * p for _, p, ptr in dlog)      # with its own buffer
    for dev, first, count, *_ in calls:              # on the device of the chunk that holds it
        assert all(d == dev for d, p, _ in dlog[first:first + count])


@pytest.mark.parametrize("ndev,where,code", [(1, "deblock", ERR_CUDA), (1, "download_decoded", ERR_STATE),
                                             (2, "deblock", ERR_STATE), (2, "download_decoded", ERR_CUDA)])
def test_injected_failure(api, ndev, where, code):
    """A failed deblock or decoded download fails the call with its code and leaves the caller's sizes as they were."""
    sizes = [HA.P] * 2072
    rc, calls, _, _, sizes_out = run(api, sizes, ndev, **{f"fail_{where}": 2, "fail_code": code})
    assert rc == code
    assert sizes_out == sizes
    assert 2 <= len(calls) <= 8


@pytest.mark.parametrize("decs", ["null", "null_entry"])
def test_null_decoded_buffers(api, decs):
    sizes = [HA.P] * 60
    rc, calls, dlog, ndeb, sizes_out = run(api, sizes, 1, decs=decs)
    assert rc == ERR_ARG
    assert calls == [] and dlog == [] and ndeb == 0
    assert sizes_out == sizes


def test_empty_batch(api):
    assert api.HEVCImageEncoderBatchDecoded(0, None, None, None, None, None, None, None, None) == 0
    assert api.HEVCImageEncoderBatchDecoded(-1, None, None, None, None, None, None, None, None) == ERR_ARG


def test_linked_without_the_decoded_calls(tmp_path):
    """hevce_api.c still links and loads with a CUDA layer that lacks the two decoded-picture calls (the chunk-planner
    test links it so); HEVCImageEncoderBatchDecoded then fails instead of calling through a null reference."""
    so = str(tmp_path / "libhevce_apistub_plain.so")
    subprocess.run(["gcc", "-O2", "-Wall", "-fPIC", "-shared", "-pthread", "-I", HA.CSRC, "-o", so,
                    os.path.join(HA.CSRC, "hevce_api.c"), HA.STUB], check=True)
    L = ctypes.CDLL(so, mode=os.RTLD_NOW)
    L.apistub_reset(1, 0, 0, 0)
    n = 3
    ys, xs, qs = (ctypes.c_int * n)(32, 32, 32), (ctypes.c_int * n)(32, 32, 32), (ctypes.c_int * n)(2, 2, 2)
    dummy = (ctypes.c_void_p * n)(1, 1, 1)
    assert L.HEVCImageEncoderBatchDecoded(n, dummy, dummy, dummy, dummy, ys, xs, qs, None) == ERR_STATE
    assert L.HEVCImageEncoderBatch(n, dummy, dummy, dummy, ys, xs, qs, None) == 0
