"""GPU tests of SSIM on the device and the quality-target entry point (DESIGN.md section 1, row f7): hevce_ssim_kernel
through Session.ssim must equal the host SSIM of tools/hevc_eval.py and be bit-identical however a picture is batched;
HEVCImageEncoderBatchTarget must choose, per picture, what the search rule picks from an oracle that encodes every qpd6,
and return that encode's stream, reconstruction, decoded picture and quality."""
import os
import sys

import numpy as np
import pytest

import test_decode as TD
import test_ssim as TS
import workloads as WL

sys.path.insert(0, os.path.join(TS.S.ROOT, "tools"))
import hevc_eval  # noqa: E402

pytestmark = pytest.mark.gpu

SSIM_TARGETS = [0.85, 0.93, 0.98, 1.01]
PSNR_TARGETS = [30.0, 38.0, 45.0]


@pytest.fixture(scope="module")
def H():
    import hevce_b200
    hevce_b200.set_devices([0])
    return hevce_b200


def mixed_batch():
    """The mixed-size batch of test_gpu_decode.py."""
    rng = np.random.default_rng(66)
    shapes = [(45, 70), (512, 768), (100, 33), (256, 256), (64, 1000), (333, 222), (32, 32)]
    return [TD.random_picture(rng, h, w, ("smooth", "noise", "checker", "flat")[i % 4]) for i, (h, w) in enumerate(shapes)]


@pytest.fixture(scope="module")
def pictures():
    return WL.kodak_landscape() + mixed_batch()


def measure(H, imgs, qs):
    """Session run: (recons, decoded, ssim of recons, ssim of decoded, decoded PSNR)."""
    ses = H.Session(0, [i.shape for i in imgs], qs)
    ses.upload(imgs)
    ses.encode()
    _, rcons = ses.download()
    s_rcon = ses.ssim()
    assert ses.ssim_ms > 0
    ses.deblock()
    decs = ses.download_decoded()
    s_dec = ses.ssim(decoded=True)
    _, psnr = ses.decoded_quality()
    ses.close()
    return rcons, decs, s_rcon, s_dec, psnr


def test_ssim_matches_host(H, pictures):
    """24 Kodak pictures at qpd6 0-4 and the mixed batch: reconstructions and decoded pictures within 1e-10 of the host."""
    imgs = [p for p in pictures[:24] for _ in range(5)] + pictures[24:]
    qs = [q for _ in range(24) for q in range(5)] + [i % 5 for i in range(len(pictures) - 24)]
    rcons, decs, s_rcon, s_dec, _ = measure(H, imgs, qs)
    for i, img in enumerate(imgs):
        c = TS.coded(img)
        assert abs(s_rcon[i] - hevc_eval.ssim(c, rcons[i])) <= 1e-10, (i, qs[i])
        assert abs(s_dec[i] - hevc_eval.ssim(c, decs[i])) <= 1e-10, (i, qs[i])
        if qs[i] <= 1:
            assert s_dec[i] == s_rcon[i]                      # the filter changes nothing at qpd6 0-1


def test_ssim_of_clamped_picture(H):
    rng = np.random.default_rng(9)
    img = TD.random_picture(rng, 300, 170, "smooth")
    old = H.set_max_dim(200)
    try:
        rcons, decs, s_rcon, s_dec, _ = measure(H, [img], 3)
    finally:
        H.set_max_dim(old)
    c = TS.coded(img, 200)
    assert rcons[0].shape == c.shape == (224, 192)
    assert abs(s_rcon[0] - hevc_eval.ssim(c, rcons[0])) <= 1e-10
    assert abs(s_dec[0] - hevc_eval.ssim(c, decs[0])) <= 1e-10


def test_ssim_is_deterministic(H, pictures):
    """Bit-identical across two runs and between a one-picture session and the whole batch."""
    qs = [i % 5 for i in range(len(pictures))]
    ses = H.Session(0, [i.shape for i in pictures], qs)
    ses.upload(pictures)
    ses.encode()
    a = ses.ssim()
    ses.deblock()
    d = ses.ssim(decoded=True)
    assert ses.ssim().tobytes() == a.tobytes() and ses.ssim(decoded=True).tobytes() == d.tobytes()
    ses.close()
    for i in (0, 13, 23, 24, 25, len(pictures) - 1):
        _, _, s_rcon, s_dec, _ = measure(H, [pictures[i]], qs[i])
        assert s_rcon[0].tobytes() == a[i].tobytes() and s_dec[0].tobytes() == d[i].tobytes(), i


def test_state_errors(H):
    img = np.full((64, 64), 9, np.uint8)
    img[:, 32:] = 30
    ses = H.Session(0, [img.shape], 4)
    ses.upload([img])
    for decoded in (False, True):
        with pytest.raises(H.HevceError) as e:
            ses.ssim(decoded)
        assert e.value.code == H.ERR_STATE
    ses.encode()
    assert 0.0 < ses.ssim()[0] <= 1.0
    with pytest.raises(H.HevceError) as e:
        ses.ssim(decoded=True)
    assert e.value.code == H.ERR_STATE
    ses.close()


@pytest.fixture(scope="module")
def oracle(H, pictures):
    """Every picture encoded at all five qpd6 by HEVCImageEncoderBatchDecoded, measured by the session."""
    out = []
    for q in range(5):
        streams, rcons, decs = H.HEVCImageEncoderBatchDecoded(pictures, q)
        _, sdecs, _, s_dec, psnr = measure(H, pictures, q)
        assert all(np.array_equal(a, b) for a, b in zip(decs, sdecs))
        out.append({"streams": streams, "rcons": rcons, "decs": decs, "ssim": s_dec, "psnr": psnr})
    return out


def rule(row, target):
    lo, hi = -1, 5
    while hi - lo > 1:
        q = (lo + hi) // 2
        if row[q] >= target:
            lo = q
        else:
            hi = q
    return lo if lo >= 0 else 0


@pytest.mark.parametrize("metric,target", [("ssim", t) for t in SSIM_TARGETS] + [("psnr", t) for t in PSNR_TARGETS])
def test_target_matches_oracle(H, pictures, oracle, metric, target):
    streams, rcons, decs, qpd6, quality = H.HEVCImageEncoderBatchTarget(pictures, target, metric, decoded=True)
    for i in range(len(pictures)):
        row = [oracle[q][metric][i] for q in range(5)]
        c = rule(row, target)
        assert qpd6[i] == c, (i, row)
        assert quality[i].tobytes() == row[c].tobytes(), i
        o = oracle[c]
        assert streams[i] == o["streams"][i], i
        assert np.array_equal(rcons[i], o["rcons"][i]) and np.array_equal(decs[i], o["decs"][i]), i
    if metric == "ssim" and target > 1.0:
        assert list(qpd6) == [0] * len(pictures)              # no setting reaches SSIM 1.01: qpd6 0, and it shows
        assert all(quality < target)
    got = H.HEVCImageDecoderBatch(streams)
    assert all(np.array_equal(g, d) for g, d in zip(got, decs))


def test_target_per_picture_and_without_decoded(H, pictures, oracle):
    targets = [(0.80, 0.90, 0.95, 0.99)[i % 4] for i in range(len(pictures))]
    streams, rcons, qpd6, quality = H.HEVCImageEncoderBatchTarget(pictures, targets, "ssim")
    for i, t in enumerate(targets):
        c = rule([oracle[q]["ssim"][i] for q in range(5)], t)
        assert qpd6[i] == c and streams[i] == oracle[c]["streams"][i] and np.array_equal(rcons[i], oracle[c]["rcons"][i]), i
    with pytest.raises(H.HevceError) as e:
        H.HEVCImageEncoderBatchTarget(pictures[:2], float("nan"))
    assert e.value.code == H.ERR_ARG


def test_bench_batch(H):
    """The benchmark's 1036 pictures of 768x512 at SSIM 0.95; the choice of a sample checked against all five qpd6."""
    imgs = WL.config3_batch(0, 1036)
    streams, rcons, qpd6, quality = H.HEVCImageEncoderBatchTarget(imgs, 0.95, "ssim")
    assert all(0 <= q <= 4 for q in qpd6)
    assert all((s >= 0.95) or q == 0 for s, q in zip(quality, qpd6))
    sample = sorted(np.random.default_rng(3).choice(len(imgs), 5, replace=False).tolist())
    sub = [imgs[i] for i in sample]
    rows = [measure(H, sub, q)[3] for q in range(5)]
    for k, i in enumerate(sample):
        row = [rows[q][k] for q in range(5)]
        c = rule(row, 0.95)
        assert qpd6[i] == c and quality[i] == row[c], i
        ses_streams, _ = H.HEVCImageEncoderBatch([imgs[i]], c)
        assert ses_streams[0] == streams[i], i


def test_two_devices(H, pictures, oracle):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    H.set_devices([0, 1])
    try:
        streams, _, decs, qpd6, quality = H.HEVCImageEncoderBatchTarget(pictures, 0.93, "ssim", decoded=True)
    finally:
        H.set_devices([0])
    for i in range(len(pictures)):
        c = rule([oracle[q]["ssim"][i] for q in range(5)], 0.93)
        assert qpd6[i] == c and quality[i] == oracle[c]["ssim"][i] and streams[i] == oracle[c]["streams"][i], i
