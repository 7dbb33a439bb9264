"""The decoder (csrc/hevce_decode.h, run by hevce_parse_kernel / hevce_recon_kernel, then hevce_deblock_kernel) on the
CPU: tests/sim/hevce_simdecode.cpp runs the kernels' own functions over whole pictures in their phase order.  Streams of
the reference (the small goldens) and of the simulator must decode to their reconstructions before deblocking, to the
filter model and to libavcodec after it; rejected headers and corrupt slice data must end in a status, never a fault."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import deblock_model as D
import decode_util as U
import golden_util as G
import simutil as S

_u8p = ctypes.POINTER(ctypes.c_ubyte)
SRC = os.path.join(S.SIM_DIR, "hevce_simdecode.cpp")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("simdecode") / "libhevce_simdecode.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-w", *S.variant_flags("g7"), "-I", S.CSRC, "-o", so, SRC], check=True)
    return ctypes.CDLL(so)


def info(L, stream):
    s = np.frombuffer(bytes(stream), np.uint8).copy()
    h, w, q = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    n = L.hevce_simdecode_info(s.ctypes.data_as(_u8p), len(s), ctypes.byref(h), ctypes.byref(w), ctypes.byref(q))
    return None if n < 0 else (h.value, w.value, q.value)


def decode(L, streams, order=0):
    """[(status, rcon, dec, cu_size, mode, kind)] of the streams, decoded in one harness call."""
    arrs = [np.frombuffer(bytes(s), np.uint8).copy() for s in streams]
    n = len(arrs)
    shapes = [info(L, a)[:2] for a in arrs]
    rcons = [np.full(s, 0xEE, np.uint8) for s in shapes]
    decs = [np.full(s, 0xEE, np.uint8) for s in shapes]
    cus = [np.zeros((h // 4, w // 4), np.uint8) for h, w in shapes]
    modes = [np.zeros((h // 4, w // 4), np.uint8) for h, w in shapes]
    kinds = [np.zeros((h // 8, w // 8), np.uint8) for h, w in shapes]
    st = (ctypes.c_int * n)()
    arr = lambda xs: (_u8p * n)(*[x.ctypes.data_as(_u8p) for x in xs])
    rc = L.hevce_simdecode(n, arr(arrs), (ctypes.c_int * n)(*[a.size for a in arrs]), arr(rcons), arr(decs), arr(cus), arr(modes), arr(kinds),
                           st, int(order))
    assert rc == 0
    return [(st[i], rcons[i], decs[i], cus[i], modes[i], kinds[i]) for i in range(n)]


@pytest.mark.parametrize("order", [0, 1])
def test_reference_goldens(harness, order):
    """All 85 small goldens (reference-written): the picture before deblocking is the reference's reconstruction, the
    decoded picture is the filter model's output and libavcodec's luma, and the header gives the padded shape and q."""
    npz, meta = G.small_cases()
    names = sorted(meta)
    streams = [npz[f"{n}/q{q}/stream"].tobytes() for n in names for q in range(5)]
    out = decode(harness, streams, order)
    k = 0
    for name in names:
        for q in range(5):
            rcon = npz[f"{name}/q{q}/rcon"]
            st, r, d, cu, _, kind = out[k]
            assert info(harness, streams[k]) == (rcon.shape[0], rcon.shape[1], q)
            assert st == 0, (name, q)
            assert np.array_equal(r, rcon), (name, q)
            assert np.array_equal(d, D.deblock(rcon, cu, kind, q)), (name, q)
            luma = U.decode_luma(streams[k], rcon.shape) if order == 0 else None
            if luma is not None:
                assert np.array_equal(d, luma), (name, q)
            k += 1


def random_picture(rng, h, w, kind):
    if kind == "noise":
        return rng.integers(0, 256, (h, w)).astype(np.uint8)
    if kind == "flat":
        return np.full((h, w), int(rng.integers(0, 256)), np.uint8)
    if kind == "checker":
        c = int(rng.integers(2, 9))
        yy, xx = np.mgrid[0:h, 0:w]
        return np.where(((yy // c) + (xx // c)) % 2 == 0, 30, 220).astype(np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    base = 120 + 60 * np.sin(xx / (5 + 10 * rng.random()) + rng.random() * 6) + 40 * np.cos(yy / (4 + 8 * rng.random()))
    return np.clip(base + rng.integers(-3, 4, (h, w)), 0, 255).astype(np.uint8)


CASES = [(kind, h, w) for kind in ("smooth", "noise", "flat", "checker") for h, w in ((45, 70), (160, 224), (32, 32), (100, 33))]


@pytest.mark.parametrize("q", [0, 1, 2, 3, 4])
def test_simulator_streams(harness, q):
    """Random pictures encoded by the simulator: reconstruction, partition and (where libavcodec decodes) the decoded
    picture are the encoder's."""
    rng = np.random.default_rng(600 + q)
    for kind, h, w in CASES:
        img = random_picture(rng, h, w, kind)
        s, rcon, err = S.sim_encode(img, q)
        assert err == 0
        cu0, mode0, kind0 = S.sim_last_partition(rcon.shape)
        st, r, d, cu, mode, kd = decode(harness, [s], order=q % 2)[0]
        assert st == 0, (kind, h, w)
        assert np.array_equal(r, rcon), (kind, h, w)
        assert np.array_equal(cu, cu0) and np.array_equal(mode, mode0) and np.array_equal(kd, kind0), (kind, h, w)
        assert np.array_equal(d, D.deblock(rcon, cu0, kind0, q)), (kind, h, w)
        luma = U.decode_luma(s, rcon.shape)
        if luma is not None:
            assert np.array_equal(d, luma), (kind, h, w)


def test_rejected_headers(harness):
    npz, _ = G.small_cases()
    s = npz["k01_64x128/q2/stream"].tobytes()
    assert info(harness, s) == (64, 128, 2)
    hdr = 27 + 22 + 8 + 11 + 8
    for pos in (5, 30, 52, 60, 70, hdr - 1):           # VPS, SPS, SPS size field, PPS, slice header
        b = bytearray(s)
        b[pos] ^= 0x10
        assert info(harness, bytes(b)) is None, pos
    for cut in (0, 10, 49, 60, hdr - 1):
        assert info(harness, s[:cut]) is None, cut
    assert info(harness, b"\x00" * 100) is None


def test_size_limit(harness):
    """The header check takes sizes up to 16384 and not beyond (streams from the simulator at the raised limit)."""
    img = np.full((40, 16400), 90, np.uint8)
    s, rcon, err = S.sim_encode(img, 2, max_dim=16384)
    assert err == 0 and rcon.shape == (64, 16384)
    assert info(harness, s) == (64, 16384, 2)
    n = 27 + 22                # pic_width_in_luma_samples: ue(v) at bit 4 after the VPS and the fixed SPS bytes
    bits = "".join(f"{x:08b}" for x in s[n:n + 8])
    assert bits[4:4 + 29] == f"{16385:029b}"          # ue(v) of 16384: 14 zeros, then 16385 in 15 bits
    wider = bits[:4] + f"{16417:029b}" + bits[4 + 29:]   # 16416 = 16384 + 32, the same length of code
    b = s[:n] + int(wider, 2).to_bytes(8, "big") + s[n + 8:]
    assert info(harness, b) is None


@pytest.fixture(scope="module")
def asan_prog(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("simdecode_asan") / "hevce_simdecode")
    try:
        subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-w", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                        "-DHEVCE_SIMDECODE_MAIN", *S.variant_flags("g7"), "-I", S.CSRC, "-o", exe, SRC], check=True)
    except subprocess.CalledProcessError:
        pytest.skip("no sanitizer runtime for this compiler")
    return exe


@pytest.mark.parametrize("case", [("k01_64x128", 2), ("noise_64", 0), ("checker1_64", 4)])
def test_corrupt_slice_data(asan_prog, tmp_path, case):
    """Every truncation and 1500 single-bit flips of the slice data: status 0 or failure, no sanitizer report."""
    npz, _ = G.small_cases()
    name, q = case
    p = tmp_path / "s.h265"
    p.write_bytes(npz[f"{name}/q{q}/stream"].tobytes())
    r = subprocess.run([asan_prog, str(p), "1500", str(q)], capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "ERROR" not in r.stderr and "runtime error" not in r.stderr, r.stderr
    f = dict(zip(r.stdout.split()[::2], map(int, r.stdout.split()[1::2])))
    assert f["bad"] == 0 and f["failed"] > 0
