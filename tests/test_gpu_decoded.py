"""GPU tests of the decoded picture (DESIGN.md section 1, row f5): hevce_deblock_kernel runs the in-loop deblocking filter
over the reconstructions, and what comes back through the session, the batch API and the Python binding must be what
libavcodec decodes from the streams and what the numpy model of the filter (tests/deblock_model.py) computes."""
import numpy as np
import pytest

import deblock_model as D
import decode_util as U
import golden_util as G
import simutil as S
import workloads as WL

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def H():
    import hevce_b200
    return hevce_b200


@pytest.fixture(scope="module")
def K():
    return WL.kodak_landscape()


def ref_quality(img, plane):
    """calcImagePSNR (HEVCeMain.c:116-133) in numpy."""
    hm, wm = min(img.shape[0], plane.shape[0]), min(img.shape[1], plane.shape[1])
    d = img[:hm, :wm].astype(np.int64) - plane[:hm, :wm].astype(np.int64)
    mse = max(float((d * d).sum()) / hm / wm, 1e-9)
    return mse, 10.0 * np.log10(255 * 255 / mse)


def session_run(H, imgs, q, partitions=True):
    ses = H.Session(0, [i.shape for i in imgs], q)
    ses.upload(imgs)
    ses.encode()
    streams, rcons = ses.download()
    ms = ses.deblock()
    decs = ses.download_decoded()
    mse, psnr = ses.decoded_quality()
    parts = [ses.partition(i) for i in range(len(imgs))] if partitions else None
    ses.close()
    return streams, rcons, decs, parts, (mse, psnr), ms


def pictures(K):
    data, _ = G.small_cases()
    imgs = [K[0], K[7][:480, :700], K[13][100:301, 50:505], K[20][:77, :333]]       # a ragged Kodak batch
    imgs += [WL.config3_image(4001, K), WL.config3_image(7777, K)[:301, :455]]      # far beyond the oracle runs
    imgs += [data[f"{n}/in"] for n in G.small_case_names()]
    return imgs


@pytest.mark.parametrize("q", [0, 1, 2, 3, 4])
def test_decoded_equals_decoder_and_model(H, K, q):
    imgs = pictures(K)
    streams, rcons, decs, parts, (mse, psnr), ms = session_run(H, imgs, q)
    assert ms > 0
    decoder = True
    for i, (img, s, r, d) in enumerate(zip(imgs, streams, rcons, decs)):
        assert d.shape == r.shape
        cu, _, kind = parts[i]
        assert np.array_equal(d, D.deblock(r, cu, kind, q)), (i, q)
        if q <= 1:
            assert np.array_equal(d, r), (i, q)
        m, p = ref_quality(img, d)
        assert mse[i] == pytest.approx(m, rel=1e-12, abs=0) and psnr[i] == pytest.approx(p, rel=1e-12), (i, q)
        if decoder:
            luma = U.decode_luma(s, r.shape)
            if luma is None:
                decoder = False
                continue
            assert np.array_equal(d, luma), (i, q)
    if not decoder:
        pytest.skip("no HEVC decoder in this OpenCV build (model comparison passed)")


def test_variants_give_identical_decoded_pictures(H, K):
    imgs = [WL.config3_image(i, K)[:160, :224] for i in range(9)]
    got = {}
    try:
        for tag in S.variants():
            H.set_variant(tag)
            _, rcons, decs, _, _, _ = session_run(H, imgs, 3, partitions=False)
            got[tag] = decs
    finally:
        H.set_variant(None)
    first = next(iter(got.values()))
    for tag, decs in got.items():
        assert all(np.array_equal(a, b) for a, b in zip(decs, first)), tag


def test_decoded_quality_of_clamped_picture(H):
    """A picture taller than the 8192 clamp: quality is taken over the rows both buffers have."""
    rng = np.random.default_rng(3)
    img = np.clip(np.cumsum(rng.integers(-2, 3, (8200, 33)), axis=0) + 120, 0, 255).astype(np.uint8)
    _, rcons, decs, _, (mse, psnr), _ = session_run(H, [img], 3, partitions=False)
    assert decs[0].shape == (8192, 64)
    m, p = ref_quality(img, decs[0])
    assert mse[0] == pytest.approx(m, rel=1e-12) and psnr[0] == pytest.approx(p, rel=1e-12)


def test_state_errors(H):
    img = np.full((64, 64), 9, np.uint8)
    img[:, 32:] = 30
    ses = H.Session(0, [img.shape], 4)
    ses.upload([img])

    def code(f):
        with pytest.raises(H.HevceError) as e:
            f()
        return e.value.code

    assert code(ses.deblock) == H.ERR_STATE                 # before an encode
    ses.encode()
    assert code(ses.download_decoded) == H.ERR_STATE        # before a deblock
    assert code(ses.decoded_quality) == H.ERR_STATE
    ses.deblock()
    assert ses.deblock_ms > 0
    d = ses.download_decoded()[0]
    ses.decoded_quality()
    ses.upload([img])                                       # a re-upload clears both
    assert code(ses.deblock) == H.ERR_STATE
    assert code(ses.download_decoded) == H.ERR_STATE
    ses.encode()
    assert code(ses.download_decoded) == H.ERR_STATE        # a new encode needs a new deblock
    ses.deblock()
    assert np.array_equal(ses.download_decoded()[0], d)
    ses.close()


def check_batch(H, imgs, qs, sample):
    streams0, rcons0 = H.HEVCImageEncoderBatch(imgs, qs)
    streams, rcons, decs = H.HEVCImageEncoderBatchDecoded(imgs, qs)
    assert streams == streams0
    assert all(np.array_equal(a, b) for a, b in zip(rcons, rcons0))
    sub = [imgs[i] for i in sample]
    ses = H.Session(0, [i.shape for i in sub], [qs[i] for i in sample])
    ses.upload(sub)
    ses.encode()
    parts = [ses.partition(k) for k in range(len(sub))]
    ses.close()
    for k, i in enumerate(sample):
        cu, _, kind = parts[k]
        assert np.array_equal(decs[i], D.deblock(rcons[i], cu, kind, qs[i])), i
        luma = U.decode_luma(streams[i], rcons[i].shape)
        if luma is not None:
            assert np.array_equal(decs[i], luma), i


def test_batch_decoded_same_size(H, K):
    """1,036 pictures of 768x512: the same-size path with four chunks per device."""
    imgs = [WL.config3_image(i, K) for i in range(1036)]
    qs = [2] * len(imgs)
    sample = sorted(np.random.default_rng(11).choice(len(imgs), 6, replace=False).tolist())
    check_batch(H, imgs, qs, sample)


def test_batch_decoded_ragged(H, K):
    rng = np.random.default_rng(12)
    imgs = []
    for i in range(40):
        h, w = int(rng.integers(8, 400)), int(rng.integers(8, 500))
        y, x = int(rng.integers(0, 512 - h)), int(rng.integers(0, 768 - w))
        imgs.append(K[i % 24][y:y + h, x:x + w])
    qs = [i % 5 for i in range(len(imgs))]
    check_batch(H, imgs, qs, [0, 7, 13, 22, 39])


def test_batch_decoded_over_every_device(H, K):
    import torch
    nd = torch.cuda.device_count()
    if nd < 2:
        pytest.skip("needs two or more devices")
    imgs = [WL.config3_image(i, K)[: 96 + 32 * (i % 5), :] for i in range(60)]
    qs = [i % 5 for i in range(len(imgs))]
    try:
        H.set_devices(list(range(nd)))
        check_batch(H, imgs, qs, [0, 29, 59])
    finally:
        H.set_devices([0])


def test_batch_decoded_rejects_small_buffers(H):
    img = np.zeros((40, 40), np.uint8)
    outs, rcons = H.alloc_outputs([img.shape])
    with pytest.raises(H.HevceError):
        H.HEVCImageEncoderBatchDecoded([img], 2, outputs=(outs, rcons, [np.zeros((32, 32), np.uint8)]))
