"""HEVCImageEncoderBatchTarget on the CPU: csrc/hevce_api.c, unmodified, linked with a stand-in for the whole CUDA layer
(tests/sim/hevce_apistub_target.c) that writes (picture, qpd6) markers into every output buffer and returns each
(picture, qpd6)'s quality from a table the test sets.  The chosen qpd6, quality, buffers and rounds must be those of the
search rule in include/hevce.h, restated below.  No kernel, CUDA runtime or GPU is involved."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hevc-image-encoder-lite_b200", "csrc")
STUB = os.path.join(ROOT, "tests", "sim", "hevce_apistub_target.c")
ERR_ARG, ERR_CUDA, ERR_STATE = -1, -2, -3
PSNR, SSIM = 0, 1
MAX_ID = 4096


def build(path, *defs):
    subprocess.run(["gcc", "-O2", "-Wall", "-fPIC", "-shared", "-pthread", *defs, "-I", CSRC, "-o", path,
                    os.path.join(CSRC, "hevce_api.c"), STUB], check=True)
    return ctypes.CDLL(path, mode=os.RTLD_NOW)


@pytest.fixture(scope="module")
def api(tmp_path_factory):
    return build(str(tmp_path_factory.mktemp("apistub_target") / "libhevce_apistub_target.so"))


def search(row, target):
    """The search rule of include/hevce.h: (chosen qpd6, probes in order)."""
    lo, hi, probes = -1, 5, []
    while hi - lo > 1:
        q = (lo + hi) // 2
        probes.append(q)
        if row[q] >= target:
            lo = q
        else:
            hi = q
    return (lo if lo >= 0 else 0), probes


def padded(v):
    return (min(v, 8192) + 31) // 32 * 32


class Call:
    """One HEVCImageEncoderBatchTarget call over stub devices with caller-owned buffers for every picture."""

    def __init__(self, L, sizes, table, targets, metric=SSIM, ndev=1, decoded=True, fail_configure=0, fail_code=0,
                 with_quality=True, with_lens=True):
        n = len(sizes)
        self.sizes, self.table, self.targets = sizes, table, targets
        L.apistub_target_reset(ndev, fail_configure, fail_code)
        assert L.hevce_set_devices(ndev, (ctypes.c_int * ndev)(*range(ndev))) == 0
        L.hevce_set_max_dim(8192)
        tab = (ctypes.c_double * (MAX_ID * 5)).in_dll(L, "apistub_target_table")
        for i in range(n):
            for q in range(5):
                tab[5 * i + q] = table[i][q]
        self.imgs = [np.array([i], np.int32).view(np.uint8) for i in range(n)]
        px = [padded(h) * padded(w) for h, w in sizes]
        self.pbs = [np.zeros(256 + 2 * p, np.uint8) for p in px]
        self.rcons = [np.zeros(p, np.uint8) for p in px]
        self.decs = [np.zeros(p, np.uint8) for p in px] if decoded else None
        arr = lambda xs: (ctypes.c_void_p * n)(*[x.ctypes.data for x in xs])
        self.ys = (ctypes.c_int * n)(*[h for h, _ in sizes])
        self.xs = (ctypes.c_int * n)(*[w for _, w in sizes])
        tg = (ctypes.c_double * n)(*targets)
        self.qpd6 = (ctypes.c_int * n)(*[-7] * n)
        self.quality = (ctypes.c_double * n)(*[-7.0] * n) if with_quality else None
        self.lens = (ctypes.c_int * n)(*[-7] * n) if with_lens else None
        L.HEVCImageEncoderBatchTarget.argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 4 + [ctypes.c_void_p] * 2 + \
            [ctypes.c_int] + [ctypes.c_void_p] * 4
        L.hevce_internal_set_device(5)
        self.rc = L.HEVCImageEncoderBatchTarget(n, arr(self.pbs), arr(self.imgs), arr(self.rcons), arr(self.decs) if decoded else None,
                                                self.ys, self.xs, metric, tg, self.qpd6, self.quality, self.lens)
        assert L.hevce_internal_get_device() == 5                    # the caller's device is restored
        rows = (ctypes.c_longlong * (6 * 65536))()
        m = L.apistub_target_log(rows, 65536)
        self.log = [tuple(rows[6 * i:6 * i + 6]) for i in range(m)]   # (configure no., device, id, qpd6, ysz, xsz)
        self.quality_calls = (L.apistub_target_quality_calls(PSNR), L.apistub_target_quality_calls(SSIM))

    def check(self):
        n = len(self.sizes)
        assert self.rc == 0
        want = [search(self.table[i], self.targets[i]) for i in range(n)]
        assert list(self.qpd6) == [c for c, _ in want]
        if self.quality is not None:
            assert list(self.quality) == [self.table[i][c] for i, (c, _) in enumerate(want)]
        for i, (c, _) in enumerate(want):                           # the chosen probe's outputs
            assert tuple(self.pbs[i][:8].view(np.int32)) == (i, c) and self.pbs[i][8] == ord("S"), i
            assert tuple(self.rcons[i][:8].view(np.int32)) == (i, c) and self.rcons[i][8] == ord("R"), i
            if self.decs is not None:
                assert tuple(self.decs[i][:8].view(np.int32)) == (i, c) and self.decs[i][8] == ord("D"), i
            if self.lens is not None:
                assert self.lens[i] == 16 + (5 * i + c) % 200, i
        assert list(zip(self.ys, self.xs)) == [(padded(h), padded(w)) for h, w in self.sizes]   # written back once
        # every picture was configured with its own size at exactly the probes of the rule, in order ...
        by_pic = {}
        for cfg, _, i, q, h, w in sorted(self.log):
            assert (h, w) == self.sizes[i]
            by_pic.setdefault(i, []).append((cfg, q))
        assert sorted(by_pic) == list(range(n))
        assert all([q for _, q in by_pic[i]] == want[i][1] for i in range(n))
        # ... in at most three rounds: all k-th probes are configured after every (k-1)-th probe, before any (k+1)-th
        rounds = max(len(p) for _, p in want)
        assert rounds <= 3
        for k in range(1, rounds):
            assert max(v[k - 1][0] for v in by_pic.values() if len(v) > k - 1) < min(v[k][0] for v in by_pic.values() if len(v) > k)
        return want


RAGGED = [(32, 32), (45, 70), (64, 64), (100, 33), (8, 8), (96, 64)]


def random_table(rng, n, metric):
    """Per picture: a monotone, a non-monotone, a never-met or an always-met row, and a target."""
    lo, hi = (0.5, 1.0) if metric == SSIM else (20.0, 50.0)
    rows, targets = [], []
    for i in range(n):
        row = rng.uniform(lo, hi, 5)
        kind = i % 4
        if kind == 0:
            row = np.sort(row)[::-1]
        t = float(rng.uniform(lo, hi))
        if kind == 2:
            t = hi + 1.0
        elif kind == 3:
            t = lo - 1.0
        if rng.random() < 0.1:
            t = float(row[int(rng.integers(0, 5))])                  # equal to a probe's quality: that probe passes
        rows.append([float(v) for v in row])
        targets.append(t)
    return rows, targets


@pytest.mark.parametrize("metric", [SSIM, PSNR])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_search_rule_ragged(api, metric, seed):
    rng = np.random.default_rng(seed)
    sizes = [RAGGED[i % len(RAGGED)] for i in range(40)]
    table, targets = random_table(rng, len(sizes), metric)
    call = Call(api, sizes, table, targets, metric)
    want = call.check()
    assert {len(p) for _, p in want} >= {2, 3}
    assert call.quality_calls[metric] > 0 and call.quality_calls[1 - metric] == 0


@pytest.mark.parametrize("decoded", [True, False])
def test_search_rule_same_size(api, decoded):
    """Same-size pictures: every round takes the four-worker path of the chunk planner."""
    rng = np.random.default_rng(10)
    sizes = [(64, 96)] * 120
    table, targets = random_table(rng, len(sizes), SSIM)
    Call(api, sizes, table, targets, SSIM, decoded=decoded).check()


def test_every_probe_path(api):
    """The six probe sequences: 2-3-4 (pass, pass / fail), 2-3 fail, 2-0-1 (pass / fail), 2-0 fail."""
    rows = [[0, 0, 1, 1, 1], [0, 0, 1, 1, 0], [0, 0, 1, 0, 1], [1, 1, 0, 1, 1], [1, 0, 0, 1, 1], [0, 1, 0, 1, 1]]
    call = Call(api, [(32, 32)] * 6, rows, [0.5] * 6)
    want = call.check()
    assert [p for _, p in want] == [[2, 3, 4], [2, 3, 4], [2, 3], [2, 0, 1], [2, 0, 1], [2, 0]]
    assert [c for c, _ in want] == [4, 3, 2, 1, 0, 0]


def test_optional_outputs(api):
    rng = np.random.default_rng(4)
    sizes = [RAGGED[i % len(RAGGED)] for i in range(12)]
    table, targets = random_table(rng, len(sizes), PSNR)
    Call(api, sizes, table, targets, PSNR, decoded=False, with_quality=False, with_lens=False).check()


@pytest.mark.parametrize("ndev", [2, 3])
def test_multiple_devices(api, ndev):
    rng = np.random.default_rng(20 + ndev)
    sizes = [RAGGED[i % len(RAGGED)] for i in range(30)] + [(64, 96)] * 64
    table, targets = random_table(rng, len(sizes), SSIM)
    call = Call(api, sizes, table, targets, SSIM, ndev=ndev)
    call.check()
    assert {dev for _, dev, *_ in call.log} == set(range(ndev))


@pytest.mark.parametrize("bad", ["nan", "metric"])
def test_bad_arguments_before_any_device_work(api, bad):
    sizes = [(32, 32)] * 5
    table = [[0.9] * 5] * 5
    targets = [0.8, 0.8, math.nan if bad == "nan" else 0.8, 0.8, 0.8]
    call = Call(api, sizes, table, targets, 7 if bad == "metric" else SSIM)
    assert call.rc == ERR_ARG
    assert call.log == []
    assert list(zip(call.ys, call.xs)) == sizes
    assert list(call.qpd6) == [-7] * 5


def test_failure_in_round_two(api):
    """A configure that fails in the second round fails the call with its code and leaves the sizes as they were."""
    sizes = [RAGGED[i % len(RAGGED)] for i in range(20)]
    table = [[0.9, 0.9, 0.9, 0.9, 0.9]] * 20
    dry = Call(api, sizes, table, [0.8] * 20)
    dry.check()
    first_round = max(cfg for cfg, _, _, q, _, _ in dry.log if q == 2)
    call = Call(api, sizes, table, [0.8] * 20, fail_configure=first_round + 1, fail_code=ERR_CUDA)
    assert call.rc == ERR_CUDA
    assert list(zip(call.ys, call.xs)) == sizes
    assert list(call.qpd6) == [-7] * 20


def test_empty_and_null(api):
    f = api.HEVCImageEncoderBatchTarget
    assert f(0, None, None, None, None, None, None, SSIM, None, None, None, None) == 0
    assert f(-1, None, None, None, None, None, None, SSIM, None, None, None, None) == ERR_ARG
    assert f(1, None, None, None, None, None, None, SSIM, None, None, None, None) == ERR_ARG


def test_existing_entry_points_make_no_quality_call(api):
    n = 60
    api.apistub_target_reset(1, 0, 0)
    imgs = [np.array([i], np.int32).view(np.uint8) for i in range(n)]
    bufs = [np.zeros(256 + 2 * 64 * 64, np.uint8) for _ in range(n)]
    arr = lambda xs: (ctypes.c_void_p * n)(*[x.ctypes.data for x in xs])
    ys, xs, qs = (ctypes.c_int * n)(*[64] * n), (ctypes.c_int * n)(*[64] * n), (ctypes.c_int * n)(*[3] * n)
    assert api.HEVCImageEncoderBatch(n, arr(bufs), arr(imgs), arr(bufs), ys, xs, qs, None) == 0
    assert api.HEVCImageEncoderBatchDecoded(n, arr(bufs), arr(imgs), arr(bufs), arr(bufs), ys, xs, qs, None) == 0
    assert (api.apistub_target_quality_calls(PSNR), api.apistub_target_quality_calls(SSIM)) == (0, 0)


def test_linked_without_the_quality_calls(tmp_path):
    """hevce_api.c links and loads with a CUDA layer that lacks hevce_session_ssim and hevce_session_decoded_quality;
    the target call then fails with HEVCE_ERR_STATE before any device work, and the other entry points still run."""
    L = build(str(tmp_path / "libhevce_apistub_noq.so"), "-DAPISTUB_NO_QUALITY")
    for metric in (SSIM, PSNR):
        call = Call(L, [(32, 32)] * 3, [[0.9] * 5] * 3, [0.5] * 3, metric)
        assert call.rc == ERR_STATE and call.log == []
    n = 3
    imgs = [np.array([i], np.int32).view(np.uint8) for i in range(n)]
    bufs = [np.zeros(256 + 2 * 32 * 32, np.uint8) for _ in range(n)]
    arr = (ctypes.c_void_p * n)(*[x.ctypes.data for x in bufs])
    ys, xs, qs = (ctypes.c_int * n)(32, 32, 32), (ctypes.c_int * n)(32, 32, 32), (ctypes.c_int * n)(2, 2, 2)
    assert L.HEVCImageEncoderBatch(n, arr, (ctypes.c_void_p * n)(*[x.ctypes.data for x in imgs]), arr, ys, xs, qs, None) == 0
