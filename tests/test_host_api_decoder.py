"""HEVCImageDecoderBatch on the CPU: csrc/hevce_api.c, unmodified, linked with the stand-in for the CUDA layer
(tests/sim/hevce_apistub.c) and a stand-in for the decoder calls (tests/sim/hevce_apistub_decoder.c).  Checks how a batch
of streams is split into shards and chunks, the per-picture status, failures, argument checks and a build without the
decoder.  No kernel, CUDA runtime or GPU is involved."""
import ctypes
import os
import subprocess

import pytest

import test_host_api as HA

STUB_DECODER = os.path.join(HA.ROOT, "tests", "sim", "hevce_apistub_decoder.c")
ERR_ARG, ERR_CUDA, ERR_STATE = -1, -2, -3


@pytest.fixture(scope="module")
def api(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("apistub_decoder") / "libhevce_apistub.so")
    subprocess.run(["gcc", "-O2", "-Wall", "-fPIC", "-shared", "-pthread", "-I", HA.CSRC, "-o", so,
                    os.path.join(HA.CSRC, "hevce_api.c"), HA.STUB, STUB_DECODER], check=True)
    return ctypes.CDLL(so, mode=os.RTLD_NOW)


def stub_stream(h, w, q=2, bad=0):
    return b"HVC6" + bytes([h // 32, w // 32, q, bad])


def run(L, sizes, ndev=1, bad=(), fail=(0, 0, 0, 0), code=0, with_status=True, corrupt=None):
    """One call over `ndev` stub devices.  Returns the return code, the sorted (device, first, count) uploads, the status
    array and the first byte of every output picture."""
    n = len(sizes)
    L.hevce_release()                                  # no decoder cached by an earlier call
    L.apistub_reset(ndev, 0, 0, 0)
    L.apistub_decoder_reset(*fail, code)
    assert L.hevce_set_devices(ndev, (ctypes.c_int * ndev)(*range(ndev))) == 0
    raw = [stub_stream(h, w, bad=int(i in bad)) for i, (h, w) in enumerate(sizes)]
    if corrupt is not None:
        raw[corrupt] = b"HVC7" + raw[corrupt][4:]
    bufs = [ctypes.create_string_buffer(s, len(s)) for s in raw]
    streams = (ctypes.c_void_p * n)(*[ctypes.addressof(b) for b in bufs])
    lens = (ctypes.c_int * n)(*[len(s) for s in raw])
    outs = [ctypes.create_string_buffer(1) for _ in range(n)]
    decs = (ctypes.c_void_p * n)(*[ctypes.addressof(o) for o in outs])
    st = (ctypes.c_int * n)(*[7] * n)
    L.apistub_decoder_set_base(streams)
    L.hevce_internal_set_device(HA.CALLER_DEVICE)
    rc = L.HEVCImageDecoderBatch(n, streams, lens, decs, st if with_status else None)
    assert L.hevce_internal_get_device() == HA.CALLER_DEVICE
    rows = (ctypes.c_longlong * (3 * 4096))()
    m = L.apistub_decoder_log(rows, 4096)
    ups = sorted(tuple(rows[3 * i:3 * i + 3]) for i in range(m))
    return rc, ups, list(st), [o.raw[0] for o in outs]


P, K4 = (512, 768), (2176, 3840)   # the bench picture; a 3840x2160 picture after padding
CASES = {   # sizes, devices -> (device, first, count) of every upload
    "1036_same": ([P] * 1036, 1, [(0, 0, 1036)]),
    "2500_same": ([P] * 2500, 1, [(0, 0, 2048), (0, 2048, 452)]),   # CHUNK_PIXELS = 2048 pictures of 768x512
    "100_4k": ([K4] * 100, 1, [(0, 0, 96), (0, 96, 4)]),
    "ragged": ([P, K4, (32, 32), (64, 96), K4, P], 1, [(0, 0, 6)]),
    "2072_2dev": ([P] * 2072, 2, [(0, 0, 1036), (1, 1036, 1036)]),
    "10_ragged_3dev": ([P, K4, (32, 32), K4, P, P, (64, 96), K4, P, (32, 32)], 3, [(0, 0, 3), (1, 3, 3), (2, 6, 4)]),
    "2_on_3dev": ([P, P], 3, [(0, 0, 1), (1, 1, 1)]),
}


@pytest.mark.parametrize("case", list(CASES))
def test_shards_and_chunks(api, case):
    sizes, ndev, want = CASES[case]
    rc, ups, st, first = run(api, sizes, ndev)
    assert rc == 0
    assert ups == want
    assert st == [0] * len(sizes)
    assert first == [(i + 1) & 0xff for i in range(len(sizes))]   # every picture written once, by its own chunk


def test_shards_follow_the_encoder(api):
    """The cut is the encoder's: the padded sizes of a ragged encoder batch split the same way over the devices."""
    sizes, ndev, _, enc = HA.CASES["10_ragged_3dev"]
    padded = [((h + 31) // 32 * 32, (w + 31) // 32 * 32) for h, w in sizes]
    _, ups, _, _ = run(api, padded, ndev)
    shards = {}
    for d, f, c, *_ in enc:
        lo, hi = shards.get(d, (f, f + c))
        shards[d] = (min(lo, f), max(hi, f + c))
    assert sorted((d, lo, hi - lo) for d, (lo, hi) in shards.items()) == ups


def test_status_write_back(api):
    sizes = [P] * 2500
    rc, ups, st, first = run(api, sizes, 1, bad=(5, 2100))
    assert rc == ERR_STATE
    assert len(ups) == 2                               # the chunk after a failed picture still runs
    assert [i for i, s in enumerate(st) if s] == [5, 2100] and st[5] == ERR_STATE
    rc, _, _, _ = run(api, sizes, 1, bad=(5,), with_status=False)
    assert rc == ERR_STATE


@pytest.mark.parametrize("which,code", [(0, ERR_CUDA), (1, ERR_CUDA), (2, ERR_STATE), (3, ERR_CUDA)])
def test_injected_failure(api, which, code):
    fail = [0, 0, 0, 0]
    fail[which] = 1
    rc, ups, _, _ = run(api, [P] * 2500, 1, fail=tuple(fail), code=code)
    assert rc == (ERR_CUDA if which == 0 else code)
    assert len(ups) <= 1                               # a failure stops the shard


def test_rejected_header_before_any_decoder_call(api):
    rc, ups, st, first = run(api, [P] * 10, 1, corrupt=4)
    assert rc == ERR_ARG
    assert ups == [] and all(api.apistub_decoder_calls(k) == 0 for k in range(4))
    assert st == [7] * 10 and first == [0] * 10


def test_null_arguments(api):
    api.apistub_reset(1, 0, 0, 0)
    api.apistub_decoder_reset(0, 0, 0, 0, 0)
    one = (ctypes.c_void_p * 1)(1)
    ln = (ctypes.c_int * 1)(8)
    assert api.HEVCImageDecoderBatch(0, None, None, None, None) == 0
    assert api.HEVCImageDecoderBatch(-1, None, None, None, None) == ERR_ARG
    assert api.HEVCImageDecoderBatch(1, None, ln, one, None) == ERR_ARG
    assert api.HEVCImageDecoderBatch(1, one, None, one, None) == ERR_ARG
    assert api.HEVCImageDecoderBatch(1, one, ln, None, None) == ERR_ARG
    s = ctypes.create_string_buffer(stub_stream(64, 64), 8)
    assert api.HEVCImageDecoderBatch(1, (ctypes.c_void_p * 1)(ctypes.addressof(s)), ln, (ctypes.c_void_p * 1)(None), None) == ERR_ARG
    assert all(api.apistub_decoder_calls(k) == 0 for k in range(4))


def test_one_cached_decoder_per_device(api):
    run(api, [P] * 2072, 2)
    assert api.apistub_decoders_live() == 2           # kept after the call, one per device
    api.hevce_release()
    assert api.apistub_decoders_live() == 0


def test_linked_without_the_decoder(tmp_path):
    so = str(tmp_path / "libhevce_apistub_plain.so")
    subprocess.run(["gcc", "-O2", "-Wall", "-fPIC", "-shared", "-pthread", "-I", HA.CSRC, "-o", so,
                    os.path.join(HA.CSRC, "hevce_api.c"), HA.STUB], check=True)
    L = ctypes.CDLL(so, mode=os.RTLD_NOW)
    L.apistub_reset(1, 0, 0, 0)
    one = (ctypes.c_void_p * 1)(1)
    assert L.HEVCImageDecoderBatch(1, one, (ctypes.c_int * 1)(8), one, None) == ERR_STATE
    L.hevce_release()
