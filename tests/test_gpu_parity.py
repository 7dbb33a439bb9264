"""GPU parity tests: the sm_100a path, called through the C ABI (libhevce_b200.so), against
  * the committed goldens made by the unmodified reference (small cases: full bytes; Kodak: SHA-256 manifest whose
    qpd6=4 column equals the reference's shipped testimage_out/*.h265),
  * the CPU oracle run live on seeded inputs (oracle/_ref when present, else the restatement),
  * size-independent properties at the benchmark's full size (determinism, batch == single entry, decodability).
Bar: bit-exact bitstream and reconstruction.  Nothing here reads /root/reference.
"""
import os

import numpy as np
import pytest

import golden_util as G
import refutil as R
import workloads as WL

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def H():
    import hevce_b200
    assert os.path.exists(hevce_b200.LIB_PATH), "libhevce_b200.so missing: the CUDA extension must be built in-tree"
    return hevce_b200


def checker():
    """The strongest CPU checker available on this box."""
    return R.ref() if os.path.exists(R.REF_SO) else R.oracle()


def test_small_cases_batch_ragged(H):
    """17 inputs x qpd6 0..4 = 85 pictures of different sizes and QPs in ONE batch call (incl. 1x1, padding,
    flat, noise, checkerboards)."""
    data, _ = G.small_cases()
    names = G.small_case_names()
    imgs, qs, keys = [], [], []
    for n in names:
        for q in range(5):
            imgs.append(data[f"{n}/in"]); qs.append(q); keys.append((n, q))
    streams, rcons = H.HEVCImageEncoderBatch(imgs, qs)
    for (n, q), s, r in zip(keys, streams, rcons):
        assert s == data[f"{n}/q{q}/stream"].tobytes(), (n, q)
        assert np.array_equal(r, data[f"{n}/q{q}/rcon"]), (n, q)


def test_single_entry_point_is_drop_in(H):
    data, _ = G.small_cases()
    for n, q in (("k01_45x70", 2), ("k01_1x1", 0), ("noise_64", 4), ("k01_33x97", 1)):
        s, r = H.HEVCImageEncoder(data[f"{n}/in"], q)
        assert s == data[f"{n}/q{q}/stream"].tobytes()
        assert np.array_equal(r, data[f"{n}/q{q}/rcon"])
        assert r.shape == tuple((d + 31) // 32 * 32 for d in data[f"{n}/in"].shape)   # size write-back, HEVCe.c:1643


def test_kodak_24x5_manifest(H):
    """BASELINE.json configs[1]: all 24 Kodak PGMs x qpd6 0..4 (120 encodes) batched on one GPU."""
    imgs, man = G.kodak()
    keys = [(k, q) for q in range(5) for k in sorted(man)]
    streams, rcons = H.HEVCImageEncoderBatch([imgs["k" + k] for k, _ in keys], [q for _, q in keys])
    bad = []
    for (k, q), s, r in zip(keys, streams, rcons):
        m = man[k]["q"][str(q)]
        if len(s) != m["len"] or R.sha(s) != m["stream_sha256"] or R.sha(r.tobytes()) != m["rcon_sha256"]:
            bad.append((k, q, len(s), m["len"]))
        if q == 4:
            assert R.sha(s) == man[k]["shipped_q4_sha256"]      # the reference's own golden vectors
    assert not bad, bad


def test_random_inputs_vs_live_oracle(H):
    rng = np.random.default_rng(2024)
    imgs, qs = [], []
    for i in range(24):
        h, w = int(rng.integers(1, 100)), int(rng.integers(1, 100))
        kind = i % 4
        if kind == 0:
            a = rng.integers(0, 256, (h, w))
        elif kind == 1:
            yy, xx = np.mgrid[0:h, 0:w]
            a = 128 + 60 * np.sin(xx / (2 + i)) * np.cos(yy / (3 + i)) + rng.integers(-4, 5, (h, w))
        elif kind == 2:
            a = np.kron(rng.integers(0, 256, ((h + 7) // 8, (w + 7) // 8)), np.ones((8, 8)))[:h, :w] + rng.integers(-2, 3, (h, w))
        else:
            a = np.cumsum(rng.integers(-3, 4, (h, w)), axis=1) + 128
        imgs.append(np.clip(a, 0, 255).astype(np.uint8)); qs.append(int(rng.integers(0, 5)))
    streams, rcons = H.HEVCImageEncoderBatch(imgs, qs)
    lib = checker()
    for im, q, s, r in zip(imgs, qs, streams, rcons):
        ws, wr = R.encode_with(lib, im, q)
        assert s == ws, (im.shape, q)
        assert np.array_equal(r, wr), (im.shape, q)


def test_clamp_to_8192_matches_crop(H):
    """A picture wider than 8192 encodes exactly like its 8192-wide crop (HEVCe.c:1581-1582)."""
    rng = np.random.default_rng(5)
    strip = np.clip(np.cumsum(rng.integers(-2, 3, (32, 8240)), axis=1) + 120, 0, 255).astype(np.uint8)
    s1, r1 = H.HEVCImageEncoder(strip, 3)
    s2, r2 = H.HEVCImageEncoder(np.ascontiguousarray(strip[:, :8192]), 3)
    assert r1.shape == (32, 8192) and s1 == s2 and np.array_equal(r1, r2)


def test_padding_equals_edge_replication(H):
    data, _ = G.small_cases()
    img = data["k01_45x70/in"]
    padded = np.pad(img, ((0, 64 - 45), (0, 96 - 70)), mode="edge")
    for q in (0, 3):
        a, ra = H.HEVCImageEncoder(img, q)
        b, rb = H.HEVCImageEncoder(padded, q)
        assert a == b and np.array_equal(ra, rb)


def test_config3_properties_full_size(H):
    """Config-3-shaped synthetic pictures (768x512, qpd6=2): determinism, session == batch == single entry, one
    picture against the live oracle, and FFmpeg decodability where OpenCV offers it."""
    n = 16
    imgs = WL.config3_batch(0, n)
    s1, r1 = H.HEVCImageEncoderBatch(imgs, 2)
    s2, r2 = H.HEVCImageEncoderBatch(imgs, 2)
    assert s1 == s2 and all(np.array_equal(a, b) for a, b in zip(r1, r2))
    ses = H.Session(0, [i.shape for i in imgs], 2)
    ses.upload(imgs)
    ms = ses.encode()
    s3, r3 = ses.download()
    ses.close()
    assert ms > 0 and s3 == s1 and all(np.array_equal(a, b) for a, b in zip(r1, r3))
    ss, rs = H.HEVCImageEncoder(imgs[5], 2)
    assert ss == s1[5] and np.array_equal(rs, r1[5])
    ws, wr = R.encode_with(checker(), imgs[0], 2)       # ~15 s of CPU
    assert ws == s1[0] and np.array_equal(wr, r1[0])
    checksum = R.sha(b"".join(R.sha(s).encode() for s in s1))
    assert len(checksum) == 64


def test_decoder_agrees_at_low_qp(H, tmp_path):
    """Independent check: libavcodec (via OpenCV) decodes our stream to exactly img_rcon at qpd6 0-1, where the
    in-loop deblocking filter the stream leaves enabled is a no-op (SURVEY.md section 4-5)."""
    cv2 = pytest.importorskip("cv2")
    img = WL.config3_image(3)[:256, :384]
    for q in (0, 1):
        s, r = H.HEVCImageEncoder(img, q)
        p = str(tmp_path / f"t{q}.h265")
        open(p, "wb").write(s)
        cap = cv2.VideoCapture(p, cv2.CAP_FFMPEG)
        cap.set(cv2.CAP_PROP_CONVERT_RGB, 0)
        ok, frame = cap.read()
        if not ok:
            pytest.skip("OpenCV build cannot decode HEVC here")
        luma = np.asarray(frame).reshape(-1)[: r.size].reshape(r.shape)
        assert np.array_equal(luma, r)


def test_raised_limit_extension(H):
    """hevce_set_max_dim(16384) behaves like a reference build with MAX_YSZ/MAX_XSZ raised (config 5b path)."""
    xl = os.path.join(R.ORACLE_DIR, "libhevc_oracle_xl.so")
    if not os.path.exists(xl):
        pytest.skip("XL oracle not built")
    rng = np.random.default_rng(11)
    strip = np.clip(np.cumsum(rng.integers(-2, 3, (33, 8243)), axis=1) + 100, 0, 255).astype(np.uint8)
    old = H.set_max_dim(16384)
    try:
        s, r = H.HEVCImageEncoder(strip, 2)
    finally:
        H.set_max_dim(old)
    lib = R._load(xl)
    import ctypes
    rc = np.zeros((64, 8256), np.uint8)
    buf = np.zeros(256 + 2 * rc.size, np.uint8)
    ys, xs = ctypes.c_int(33), ctypes.c_int(8243)
    u8p = ctypes.POINTER(ctypes.c_ubyte)
    n = lib.HEVCImageEncoder(buf.ctypes.data_as(u8p), strip.ctypes.data_as(u8p), rc.ctypes.data_as(u8p), ctypes.byref(ys), ctypes.byref(xs), 2)
    assert (ys.value, xs.value) == (64, 8256) == r.shape
    assert s == buf[:n].tobytes() and np.array_equal(r, rc)


def test_wide_and_tall_pictures(H):
    """Long CTU rows / columns (map line buffer, above-right availability at the right edge, ragged last CTU)."""
    wide = WL.config4_image(0)[:70, :2150]
    tall = np.ascontiguousarray(WL.config4_image(1)[:2100, :50])
    streams, rcons = H.HEVCImageEncoderBatch([wide, tall], [3, 1])
    lib = checker()
    for im, q, s, r in zip((wide, tall), (3, 1), streams, rcons):
        ws, wr = R.encode_with(lib, im, q)
        assert s == ws and np.array_equal(r, wr), im.shape


@pytest.mark.slow
def test_config4_one_4k_picture(H):
    """BASELINE.json configs[3]: one synthetic 3840x2160 picture (padded to 3840x2176, 8,160 CTUs) at qpd6=4 against the
    live CPU checker (~5 CPU-minutes; opt-in with HEVCE_SLOW=1).  Large single pictures are latency-bound by design."""
    import time
    img = WL.config4_image(0)
    t0 = time.time()
    s, r = H.HEVCImageEncoder(img, 4)
    t1 = time.time()
    ws, wr = R.encode_with(checker(), img, 4)
    t2 = time.time()
    print(f"config4: GPU {t1 - t0:.1f} s, CPU checker {t2 - t1:.1f} s, {len(s)} bytes")
    assert r.shape == (2176, 3840) and s == ws and np.array_equal(r, wr)
