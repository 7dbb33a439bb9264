"""GPU tests of the decoder (DESIGN.md section 1, row f6): hevce_parse_kernel, hevce_recon_kernel and hevce_deblock_kernel
through HEVCImageDecoderBatch and the Decoder object.  Every stream the encoder writes must decode to the encoder's own
decoded picture (and to its reconstruction at qpd6 0-1, where the filter changes nothing), the reference's goldens to the
filter model's output, and libavcodec must agree where OpenCV can decode HEVC."""
import os

import numpy as np
import pytest

import decode_util as U
import golden_util as G
import test_decode as TD
import workloads as WL

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def H():
    import hevce_b200
    hevce_b200.set_devices([0])
    return hevce_b200


@pytest.fixture(scope="module")
def kodak_encoded(H):
    K = WL.kodak_landscape()
    imgs = [k for k in K for _ in range(5)]
    qs = [q for _ in K for q in range(5)]
    streams, rcons, decs = H.HEVCImageEncoderBatchDecoded(imgs, qs)
    return streams, rcons, decs, qs


def test_kodak(H, kodak_encoded):
    """All 120 Kodak encodes decode, in a fresh decoder after release(), to the encoder's decoded pictures."""
    streams, rcons, decs, qs = kodak_encoded
    H.release()                                      # nothing of the encode is reused
    got = H.HEVCImageDecoderBatch(streams)
    for i, (g, d, r, q) in enumerate(zip(got, decs, rcons, qs)):
        assert g.shape == d.shape and np.array_equal(g, d), i
        if q <= 1:
            assert np.array_equal(g, r), i
    for i in range(0, 120, 7):                       # libavcodec on a spread of the batch
        luma = U.decode_luma(streams[i], decs[i].shape)
        if luma is None:
            break
        assert np.array_equal(got[i], luma), i


def test_decoder_object(H):
    """The 85 small goldens through a Decoder: the same pictures as HEVCImageDecoderBatch, three kernel times."""
    npz, meta = G.small_cases()
    streams = [npz[f"{n}/q{q}/stream"].tobytes() for n in sorted(meta) for q in range(5)]
    dec = H.Decoder(0)
    dec.upload(streams)
    assert dec.run() > 0
    got = dec.download()
    assert dec.parse_ms > 0 and dec.recon_ms > 0 and dec.deblock_ms > 0
    ref = H.HEVCImageDecoderBatch(streams)
    k = 0
    for n in sorted(meta):
        for q in range(5):
            assert np.array_equal(got[k], ref[k]), (n, q)
            if q <= 1:
                assert np.array_equal(got[k], npz[f"{n}/q{q}/rcon"]), (n, q)
            k += 1
    dec.close()


def test_goldens_against_model(H):
    """The decoded goldens equal deblock_model.deblock of the golden reconstruction with the partition the CPU harness
    parses from the same stream."""
    import ctypes
    import subprocess
    import tempfile
    import deblock_model as D
    import simutil as S
    so = os.path.join(tempfile.mkdtemp(), "libhevce_simdecode.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-w", *S.variant_flags("g7"), "-I", S.CSRC, "-o", so, TD.SRC], check=True)
    L = ctypes.CDLL(so)
    npz, meta = G.small_cases()
    streams = [npz[f"{n}/q{q}/stream"].tobytes() for n in sorted(meta) for q in range(5)]
    cpu = TD.decode(L, streams)
    got = H.HEVCImageDecoderBatch(streams)
    k = 0
    for n in sorted(meta):
        for q in range(5):
            rcon = npz[f"{n}/q{q}/rcon"]
            _, _, _, cu, _, kind = cpu[k]
            assert np.array_equal(got[k], D.deblock(rcon, cu, kind, q)), (n, q)
            k += 1


def test_mixed_batch_and_single(H):
    rng = np.random.default_rng(66)
    shapes = [(45, 70), (512, 768), (100, 33), (256, 256), (64, 1000), (333, 222), (32, 32)]
    imgs = [TD.random_picture(rng, h, w, ("smooth", "noise", "checker", "flat")[i % 4]) for i, (h, w) in enumerate(shapes)]
    qs = [i % 5 for i in range(len(imgs))]
    streams, rcons, decs = H.HEVCImageEncoderBatchDecoded(imgs, qs)
    got = H.HEVCImageDecoderBatch(streams)
    for i in range(len(imgs)):
        assert np.array_equal(got[i], decs[i]), i
    (one,) = H.HEVCImageDecoderBatch([streams[1]])
    assert np.array_equal(one, decs[1])
    assert [H.stream_info(s) for s in streams] == [(d.shape[0], d.shape[1], q) for d, q in zip(decs, qs)]


def test_bench_workload(H):
    """The benchmark's 1036 pictures of 768x512 at qpd6 2, decoded in one call."""
    imgs = WL.config3_batch(0, 1036)
    streams, _, decs = H.HEVCImageEncoderBatchDecoded(imgs, 2)
    got = H.HEVCImageDecoderBatch(streams)
    bad = [i for i in range(len(imgs)) if not np.array_equal(got[i], decs[i])]
    assert bad == []


def test_large_pictures(H):
    img = WL.config4_image(0)
    streams, _, decs = H.HEVCImageEncoderBatchDecoded([img], 2)
    (got,) = H.HEVCImageDecoderBatch(streams)
    assert np.array_equal(got, decs[0])


@pytest.mark.skipif(os.environ.get("HEVCE_SLOW") != "1", reason="HEVCE_SLOW=1: the 16000x12000 picture")
def test_raised_limit_picture(H):
    old = H.set_max_dim(16384)
    try:
        img = WL.config5_image()
        streams, _, decs = H.HEVCImageEncoderBatchDecoded([img], 2)
        (got,) = H.HEVCImageDecoderBatch(streams)
        assert np.array_equal(got, decs[0])
    finally:
        H.set_max_dim(old)


def test_errors(H, kodak_encoded):
    streams, _, decs, _ = kodak_encoded
    bad = bytearray(streams[2])
    bad[30] ^= 0x04
    with pytest.raises(H.HevceError) as e:
        H.HEVCImageDecoderBatch([streams[0], bytes(bad)])
    assert e.value.code == H.ERR_ARG
    batch = [streams[0], streams[7][: len(streams[7]) // 2], streams[13]]
    got, st = H.HEVCImageDecoderBatch(batch, return_status=True)
    assert st == [0, H.ERR_STATE, 0]
    assert np.array_equal(got[0], decs[0]) and np.array_equal(got[2], decs[13])
    assert not got[1].any()
    with pytest.raises(H.HevceError) as e:
        H.HEVCImageDecoderBatch(batch)
    assert e.value.code == H.ERR_STATE


def test_two_devices(H, kodak_encoded):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    streams, _, decs, _ = kodak_encoded
    H.set_devices([0, 1])
    try:
        got = H.HEVCImageDecoderBatch(streams)
    finally:
        H.set_devices([0])
    assert all(np.array_equal(g, d) for g, d in zip(got, decs))
