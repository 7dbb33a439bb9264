"""The drop-in boundary under the conditions a host application creates (SURVEY.md section 8b): the reference's own,
unmodified CLI main linked against libhevce_b200.so; concurrent callers; several devices behind one call; the raised
size limit; releasing the cached sessions."""
import ctypes
import os
import subprocess
import threading

import numpy as np
import pytest

import golden_util as G
import refutil as R
import workloads as WL

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "HEVCe")
REF_MAIN_ON_US = os.path.join(ROOT, "oracle", "_ref", "HEVCeMain_on_b200")
DROPIN_CLI = os.path.join(ROOT, "hevc-image-encoder-lite_b200", "HEVCe")


@pytest.fixture(scope="module")
def H():
    import hevce_b200
    assert os.path.exists(hevce_b200.LIB_PATH)
    hevce_b200.set_variant(None)
    return hevce_b200


def write_pgm(path, img):
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n255\n" % (img.shape[1], img.shape[0]))
        f.write(np.ascontiguousarray(img, np.uint8).tobytes())


@pytest.mark.parametrize("pic,q", [("k05", "2"), ("k19", "4")])
def test_reference_main_runs_on_this_library(tmp_path, pic, q):
    """HEVCeMain.c:197 calls HEVCImageEncoder; HEVCeMain_on_b200 is that file, unmodified, linked against
    libhevce_b200.so (oracle/Makefile), and hevc-image-encoder-lite_b200/HEVCe is the drop-in CLI.  On two full Kodak
    pictures (one landscape, one portrait) each .h265 and reconstruction PGM must be the reference's (length and SHA-256
    in the Kodak manifest) and each report must give the figures of that stream and reconstruction.  Where oracle/_ref
    holds the reference CLI built from the reference's own sources, both must also equal its output byte for byte,
    report included."""
    imgs, man = G.kodak()
    want = man[pic[1:]]["q"][q]
    src = tmp_path / "in.pgm"
    write_pgm(src, imgs[pic])
    outs = {}
    for tag, exe in (("ref", REF_CLI), ("ours", REF_MAIN_ON_US), ("dropin", DROPIN_CLI)):
        if tag != "dropin" and not os.path.exists(exe):
            continue
        h265, rec = tmp_path / f"{tag}.h265", tmp_path / f"{tag}.pgm"
        r = subprocess.run([exe, str(src), str(h265), q, str(rec)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        outs[tag] = (h265.read_bytes(), rec.read_bytes(), r.stdout.replace(str(h265), "<s>").replace(str(rec), "<r>"))
        assert len(outs[tag][0]) == want["len"] and R.sha(outs[tag][0]) == want["stream_sha256"], tag
        assert R.sha(outs[tag][1]) == want["rcon_pgm_sha256"], tag
        report = outs[tag][2].splitlines()
        for line in R.report_figures(imgs[pic], R.read_pgm(str(rec)), want["len"]):
            assert line in report, (tag, line)
    if "ref" in outs:
        for tag in set(outs) - {"ref"}:
            assert outs[tag] == outs["ref"], tag


def test_concurrent_callers(H):
    """HEVCImageEncoder from four host threads at once (the reference is re-entrant, README.md:25-28) equals the serial
    results; a batch call runs beside them."""
    data, _ = G.small_cases()
    cases = [("k01_45x70", 2), ("noise_64", 0), ("k01_64x128", 4), ("k01_33x97", 1), ("checker2_64", 3), ("k01_96x64", 2)]
    want = {c: (data[f"{c[0]}/q{c[1]}/stream"].tobytes(), np.array(data[f"{c[0]}/q{c[1]}/rcon"])) for c in cases}
    inputs = {c: np.array(data[f"{c[0]}/in"]) for c in cases}     # materialised: the npz reader is not thread-safe
    errors = []

    def worker(k):
        try:
            for rep in range(3):
                for c in cases[k % 2::2] if k < 4 else cases:
                    s, r = H.HEVCImageEncoder(inputs[c], c[1])
                    if s != want[c][0] or not np.array_equal(r, want[c][1]):
                        errors.append((k, c))
        except Exception as e:   # noqa: BLE001
            errors.append((k, repr(e)))

    def batch_worker():
        try:
            s, r = H.HEVCImageEncoderBatch([inputs[c] for c in cases], [c[1] for c in cases])
            for c, a, b in zip(cases, s, r):
                if a != want[c][0] or not np.array_equal(b, want[c][1]):
                    errors.append(("batch", c))
        except Exception as e:   # noqa: BLE001
            errors.append(("batch", repr(e)))

    th = [threading.Thread(target=worker, args=(k,)) for k in range(4)] + [threading.Thread(target=batch_worker)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors


def test_one_call_over_several_devices(H):
    """The library's own multi-device split (hevce_api.c): one HEVCImageEncoderBatch call, all visible devices, a
    ragged batch against the goldens and same-size pictures against a single-device run."""
    import torch
    nd = torch.cuda.device_count()
    if nd < 2:
        pytest.skip("needs at least 2 GPUs")
    data, _ = G.small_cases()
    imgs, qs, keys = [], [], []
    for n in G.small_case_names():
        for q in range(5):
            imgs.append(data[f"{n}/in"]); qs.append(q); keys.append((n, q))
    same = [WL.config3_image(i)[:128, :160].copy() for i in range(6 * nd + 1)]
    try:
        H.set_devices([0])
        s0, r0 = H.HEVCImageEncoderBatch(same, 2)
        H.set_devices(list(range(nd)))
        streams, rcons = H.HEVCImageEncoderBatch(imgs, qs)
        s1, r1 = H.HEVCImageEncoderBatch(same, 2)
    finally:
        H.set_devices([0])
    for (n, q), s, r in zip(keys, streams, rcons):
        assert s == data[f"{n}/q{q}/stream"].tobytes() and np.array_equal(r, data[f"{n}/q{q}/rcon"]), (n, q)
    assert s0 == s1 and all(np.array_equal(a, b) for a, b in zip(r0, r1))


def test_raised_limit_sizes_buffers_from_the_library(H):
    """With the limit raised, the default-argument calls must size their outputs from the library's limit (a picture
    wider than 8192 then needs more than an 8192-wide reconstruction)."""
    rng = np.random.default_rng(3)
    strip = np.clip(np.cumsum(rng.integers(-2, 3, (32, 8250)), axis=1) + 90, 0, 255).astype(np.uint8)
    old = H.set_max_dim(16384)
    try:
        assert H.get_max_dim() == 16384
        s, r = H.HEVCImageEncoder(strip, 3)
        (s2,), (r2,) = H.HEVCImageEncoderBatch([strip], 3)
    finally:
        H.set_max_dim(old)
    assert r.shape == (32, 8256) and s == s2 and np.array_equal(r, r2)
    s3, r3 = H.HEVCImageEncoder(strip, 3)                      # back at 8192: the crop
    assert r3.shape == (32, 8192) and s3 != s


def test_release_and_reuse(H):
    data, _ = G.small_cases()
    img, want = data["k01_64x64/in"], data["k01_64x64/q2/stream"].tobytes()
    assert H.HEVCImageEncoder(img, 2)[0] == want
    H.release()
    H.release()
    assert H.HEVCImageEncoder(img, 2)[0] == want


def test_caller_device_is_left_alone(H):
    """The call must not change the calling thread's current CUDA device."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    data, _ = G.small_cases()
    torch.cuda.set_device(1)
    torch.zeros(1, device="cuda")
    try:
        H.set_devices([0])
        H.HEVCImageEncoder(data["k01_32x32/in"], 2)
        try:
            rt = ctypes.CDLL("libcudart.so.12")
        except OSError:
            pytest.skip("no shared CUDA runtime to ask")
        d = ctypes.c_int(-1)
        assert rt.cudaGetDevice(ctypes.byref(d)) == 0 and d.value == 1
    finally:
        torch.cuda.set_device(0)
