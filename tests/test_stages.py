"""Stage-level known answers (SURVEY.md section 4 item 2, section 8c): single stages of the kernel source, run on the
host (tests/sim/hevce_simstage.cpp), against the functions of the UNMODIFIED reference they replace, called through
ctypes in oracle/_ref/libhevce_ref.so -- getBorder (HEVCe.c:196), predict (:262), transform (:497), quantize (:540),
deQuantize (:600), putCoef (:1173) + CABAClen (:835) -- on random and adversarial inputs.  End-to-end bytes already
agree; these tests localise a first mismatch when the kernel is restructured."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import refutil as R
import simutil as S

STAGE_SO = os.path.join(S.SIM_DIR, "libhevce_simstage.so")
_u8p = ctypes.POINTER(ctypes.c_ubyte)
_ip = ctypes.POINTER(ctypes.c_int)


class Ctx(ctypes.Structure):
    _fields_ = [("b", ctypes.c_ubyte * 142)]


class Cab(ctypes.Structure):
    _fields_ = [("tmpbuf", ctypes.c_ubyte * 3200), ("tmpcnt", ctypes.c_int), ("count00", ctypes.c_int), ("range", ctypes.c_int),
                ("low", ctypes.c_int), ("nbits", ctypes.c_int), ("nbytes", ctypes.c_int), ("bufbyte", ctypes.c_int)]


@pytest.fixture(scope="module")
def ours():
    srcs = [os.path.join(S.SIM_DIR, "hevce_simstage.cpp"), os.path.join(S.CSRC, "hevce_core.h")]
    if not os.path.exists(STAGE_SO) or any(os.path.getmtime(STAGE_SO) < os.path.getmtime(s) for s in srcs):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", S.CSRC, "-o", STAGE_SO, srcs[0]], check=True)
    ours = ctypes.CDLL(STAGE_SO)
    # the same source with every bypass string coded call for call as the reference does (HEVCE_OPT_BYPMERGE=0): its
    # coder state must equal the reference's field by field; the product configuration (merged calls) keeps the bytes and
    # the rate but may hold a carry in `low` where the reference already added it to the pending byte
    plain_so = STAGE_SO.replace(".so", "_plain.so")
    if not os.path.exists(plain_so) or any(os.path.getmtime(plain_so) < os.path.getmtime(x) for x in srcs):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-DHEVCE_OPT_BYPMERGE=0", "-I", S.CSRC, "-o", plain_so, srcs[0]], check=True)
    ours.plain = ctypes.CDLL(plain_so)
    return ours


@pytest.fixture(scope="module")
def libs(ours):
    if not os.path.exists(R.REF_SO):
        pytest.skip("oracle/_ref not built (needs the reference tree)")
    ref = ctypes.CDLL(R.REF_SO, mode=ctypes.RTLD_LOCAL)
    ref.newContextSet.restype = Ctx
    ref.newContextSet.argtypes = [ctypes.c_int]
    ref.newCABACcoder.restype = Cab
    ref.CABAClen.restype = ctypes.c_int
    return ours, ref


def ref_pixel(ref, T, mode, q, win, orig, ty, tx, av):
    """The reference's own stage functions chained as processCURecurs chains them (HEVCe.c:1426-1432)."""
    p8 = lambda a: a.ctypes.data_as(_u8p)
    pi = lambda a: a.ctypes.data_as(_ip)
    ub = [np.zeros(1, np.uint8), np.zeros(64, np.uint8), np.zeros(64, np.uint8), np.zeros(1, np.uint8), np.zeros(64, np.uint8), np.zeros(64, np.uint8)]
    view = ctypes.cast(ctypes.addressof(win.ctypes.data_as(_u8p).contents) + (1 + ty) * 65 + 1 + tx, _u8p)
    ref.getBorder(T, ctypes.c_ubyte(av[0]), ctypes.c_ubyte(av[1]), ctypes.c_ubyte(av[2]), ctypes.c_ubyte(av[3]), view, *[p8(a) for a in ub])
    pred = np.zeros((32, 32), np.uint8)
    ref.predict(T, 0, mode, ctypes.c_ubyte(int(ub[0][0])), p8(ub[1]), p8(ub[2]), ctypes.c_ubyte(int(ub[3][0])), p8(ub[4]), p8(ub[5]), p8(pred))
    o = orig[ty:ty + T, tx:tx + T].astype(np.int32)
    res = np.zeros((32, 32), np.int32)
    res[:T, :T] = o - pred[:T, :T]
    coef, lev, deq, rres = (np.zeros((32, 32), np.int32) for _ in range(4))
    ref.transform(T, ctypes.c_ubyte(0), pi(res), pi(coef))
    ref.quantize(q, T, mode, pi(coef), pi(lev))
    ref.deQuantize(q, T, pi(lev), pi(deq))
    ref.transform(T, ctypes.c_ubyte(1), pi(deq), pi(rres))
    rec = np.clip(pred[:T, :T].astype(np.int32) + rres[:T, :T], 0, 255).astype(np.uint8)
    sse = int(((o - rec.astype(np.int32)) ** 2).sum())
    return pred[:T, :T].copy(), lev[:T, :T].copy(), rec, sse


def our_pixel(ours, T, mode, q, win, orig, ty, tx, av):
    pred, rec, lev, sse = np.zeros((T, T), np.uint8), np.zeros((T, T), np.uint8), np.zeros((T, T), np.int32), ctypes.c_int(0)
    ours.hevce_stage_pixel(T, mode, q, win.ctypes.data_as(_u8p), orig.ctypes.data_as(_u8p), ty, tx, *av,
                           pred.ctypes.data_as(_u8p), lev.ctypes.data_as(_ip), rec.ctypes.data_as(_u8p), ctypes.byref(sse))
    return pred, lev, rec, sse.value


def windows(rng):
    """Reconstruction windows / originals: natural-ish, noise, extremes."""
    yy, xx = np.mgrid[0:33, 0:65]
    yield np.clip(120 + 50 * np.sin(xx / 6.0) + 40 * np.cos(yy / 4.0) + rng.integers(-5, 6, (33, 65)), 0, 255).astype(np.uint8)
    yield rng.integers(0, 256, (33, 65)).astype(np.uint8)
    yield (rng.integers(0, 2, (33, 65)) * 255).astype(np.uint8)
    yield np.full((33, 65), 255, np.uint8)
    yield np.clip(np.cumsum(rng.integers(-3, 4, (33, 65)), axis=1) + 128, 0, 255).astype(np.uint8)


@pytest.mark.parametrize("T", [4, 8, 16, 32])
def test_pixel_stages_match_reference_functions(libs, T):
    """All 35 modes x availability patterns x qpd6: prediction (incl. reference-sample substitution and smoothing), final
    levels (transform + RDOQ + group zero-out), reconstruction (dequantisation + inverse transform) and SSE."""
    ours, ref = libs
    rng = np.random.default_rng(100 + T)
    avails = [(1, 1, 1, 1), (0, 0, 0, 0), (1, 0, 1, 0), (0, 0, 1, 1), (1, 1, 0, 0), (1, 0, 1, 1)]
    n = 0
    for wi, win in enumerate(windows(rng)):
        win = np.ascontiguousarray(win)
        orig = np.ascontiguousarray(np.clip(win[1:, 1:33].astype(np.int32) + rng.integers(-25, 26, (32, 32)), 0, 255).astype(np.uint8))
        if wi == 2:
            orig = (rng.integers(0, 2, (32, 32)) * 255).astype(np.uint8)
        for mode in range(35):
            av = avails[(mode + wi) % len(avails)]
            q = (mode + wi) % 5
            ty = 0 if T == 32 else int(rng.integers(0, (32 - T) // 4 + 1)) * 4
            tx = 0 if T == 32 else int(rng.integers(0, (32 - T) // 4 + 1)) * 4
            if tx + 2 * T > 64:                      # the window holds 64 columns right of column -1 and 32 rows below row -1
                av = (av[0], av[1], av[2], 0)
            if ty + 2 * T > 32:
                av = (av[0], 0, av[2], av[3])
            a, b = our_pixel(ours, T, mode, q, win, orig, ty, tx, av), ref_pixel(ref, T, mode, q, win, orig, ty, tx, av)
            assert np.array_equal(a[0], b[0]), ("prediction", T, mode, av, wi)
            assert np.array_equal(a[1], b[1]), ("levels", T, mode, q, wi)
            assert np.array_equal(a[2], b[2]), ("reconstruction", T, mode, q, wi)
            assert a[3] == b[3], ("sse", T, mode, q, wi)
            n += 1
    assert n == 175


@pytest.mark.parametrize("T", [4, 8, 16, 32])
def test_rdoq_every_coefficient_value(libs, T):
    """The per-coefficient RDOQ decision for EVERY coefficient value -32767..32767, every TU size and qpd6, against the
    reference's quantize() (HEVCe.c:540).  The kernel evaluates two candidate levels through a rate-step table where the
    reference scans three with calcRDcost; this is the exhaustive check of that shortcut.  Every coefficient group of the
    reference's input carries one large guard value so that the group zero-out (HEVCe.c:589) never clears the group."""
    ours, ref = libs
    vals = np.concatenate([np.arange(0, 32768), -np.arange(1, 32768)]).astype(np.int32)
    ncg = (T // 4) ** 2
    per_block = 15 * ncg
    pad = (-len(vals)) % per_block
    vals = np.concatenate([vals, np.zeros(pad, np.int32)])
    slots = [(4 * gy + r, 4 * gx + c) for gy in range(T // 4) for gx in range(T // 4) for r in range(4) for c in range(4) if (r, c) != (0, 0)]
    ys, xs = np.array([s[0] for s in slots]), np.array([s[1] for s in slots])
    for q in range(5):
        got = np.zeros(len(vals), np.int32)
        ours.hevce_stage_rdoq(T, q, len(vals), vals.ctypes.data_as(_ip), got.ctypes.data_as(_ip))
        want = np.zeros(len(vals), np.int32)
        for b in range(len(vals) // per_block):
            coef, lev = np.zeros((32, 32), np.int32), np.zeros((32, 32), np.int32)
            coef[0:T:4, 0:T:4] = 32767                                            # the guards
            coef[ys, xs] = vals[b * per_block:(b + 1) * per_block]
            ref.quantize(q, T, 0, coef.ctypes.data_as(_ip), lev.ctypes.data_as(_ip))
            want[b * per_block:(b + 1) * per_block] = lev[ys, xs]
        bad = np.nonzero(got != want)[0]
        assert len(bad) == 0, (T, q, int(vals[bad[0]]), int(got[bad[0]]), int(want[bad[0]]))


def test_probability_state_63_is_unreachable(ours):
    """Probability state 63 (context bytes 126, 127) is closed off in the kernel's tables: no transition from a lower
    state and no initial value of any context reaches it, so the renormalisation shift computed from the LPS range
    never meets the one state where it differs from the reference's table."""
    st, dr, cx = (ctypes.c_int * (128 * 6))(), (ctypes.c_int * 8)(), (ctypes.c_int * (5 * 92))()
    assert ours.hevce_stage_tables(st, dr, cx) == 92
    assert all(st[v * 6 + 4] < 126 and st[v * 6 + 5] < 126 for v in range(126))
    assert all(cx[i] < 126 for i in range(5 * 92))


def test_coder_tables_match_the_reference_tables(libs):
    """The kernel's packed tables against the arrays and functions the reference exports: the 64-bit word per context
    state (LPS ranges, both next states: CABAC_LPS_TABLE, CONTEXT_NEXT_STATE_LPS / _MPS, HEVCe.c:701-713), the
    renormalisation shift the kernel derives from the LPS range (CABAC_RENORM_TABLE, :715), the RDOQ rate steps
    (estimateCoeffRate, :522) and the initial value of every context of the compact layout (newContextSet, :763)."""
    ours, ref = libs
    st, dr, cx = (ctypes.c_int * (128 * 6))(), (ctypes.c_int * 8)(), (ctypes.c_int * (5 * 92))()
    n = ours.hevce_stage_tables(st, dr, cx)
    assert n == 92
    lps = (ctypes.c_ubyte * 256).in_dll(ref, "CABAC_LPS_TABLE")
    renorm = (ctypes.c_ubyte * 32).in_dll(ref, "CABAC_RENORM_TABLE")
    nlps = (ctypes.c_ubyte * 128).in_dll(ref, "CONTEXT_NEXT_STATE_LPS")
    nmps = (ctypes.c_ubyte * 128).in_dll(ref, "CONTEXT_NEXT_STATE_MPS")
    for v in range(128):
        for q in range(4):
            r = st[v * 6 + q]
            assert r == lps[(v >> 1) * 4 + q], (v, q)
            if v < 126:   # probability state 63 is reserved for the terminate bin (no context ever holds it)
                assert 9 - r.bit_length() == renorm[r >> 3], (v, q, r)
        assert (st[v * 6 + 4], st[v * 6 + 5]) == (nlps[v], nmps[v]), v
    ref.estimateCoeffRate.restype = ctypes.c_int
    rate = [ref.estimateCoeffRate(l) for l in range(0, 9000)]
    for l in range(1, 9000):      # levels reach 8192 (|coefficient| <= 32767 at qpd6 = 0, 32x32)
        step = dr[min(l, 7)] + (65536 if l >= 7 and ((l - 5) & (l - 6)) == 0 else 0)
        assert step == rate[l] - rate[l - 1], l
    # compact context index -> byte offset in the reference's ContextSet (HEVCe.c:745-759)
    m = {}
    for i in range(3):
        m[0 + i], m[3 + i] = 16 + i, 41 + i                       # last_x / last_y of 4x4 TUs
    for i in range(16):
        m[6 + i] = 112 + i                                        # greater1
    for i in range(4):
        m[22 + i] = 136 + i                                       # greater2
    for i in range(27):
        m[26 + i] = 68 + i                                        # sig_coeff (luma)
    for i in range(12):
        m[53 + i] = i                                             # split_cu .. cbf_chroma[0]
    m[65], m[66] = 66, 67                                         # coded_sub_block
    for row, (off, cnt) in enumerate([(0, 3), (3, 4), (7, 5)], start=1):
        for i in range(cnt):
            m[67 + off + i], m[79 + off + i] = 16 + 5 * row + i, 41 + 5 * row + i
    assert sorted(m) == list(range(91))
    for q in range(5):
        want = ref.newContextSet(q)
        for i, o in m.items():
            assert cx[q * 92 + i] == want.b[o], (q, i, o)


def ref_residual(ref, T, mode, q, lev):
    cab, ctx = ref.newCABACcoder(), ref.newContextSet(q)
    blk = np.zeros((32, 32), np.int32)
    blk[:T, :T] = lev
    l0 = ref.CABAClen(ctypes.byref(cab))
    ref.putCoef(ctypes.byref(cab), ctypes.byref(ctx), T, 0, mode, blk.ctypes.data_as(_ip))
    return ref.CABAClen(ctypes.byref(cab)) - l0, (cab.range, cab.low, cab.nbits, cab.nbytes, cab.bufbyte, cab.count00, cab.tmpcnt)


def our_residual(ours, T, mode, q, lev):
    st = (ctypes.c_int * 7)()
    bits = ours.hevce_stage_residual(T, mode, q, np.ascontiguousarray(lev, np.int32).ctypes.data_as(_ip), st)
    return bits, tuple(st)


def spot_blocks():
    z = np.zeros((4, 4), np.int32)
    a = z.copy(); a[0, 0] = 5; a[1, 2] = -1
    b = np.zeros((8, 8), np.int32); b[0, 0] = -12; b[3, 3] = 2; b[7, 7] = 1
    c = np.zeros((32, 32), np.int32); c[0, 0] = 300; c[31, 31] = -1
    return ((4, 0, 2, z), (4, 26, 2, a), (8, 10, 0, b), (32, 1, 4, c))


def test_residual_coding_spot_values(ours):
    """The known answers of SURVEY.md section 8c (fresh coder, fresh contexts), measured on the reference."""
    z, a, b, c = spot_blocks()
    assert our_residual(ours, *z)[0] == 4                              # putCoef on an all-zero block codes last=(0,0)
    bits, st = our_residual(ours, *a)
    assert bits == 25 and st[:5] == (464, 126432, 14, 1, 191) and st[6] == 1
    assert our_residual(ours, *b)[0] == 52
    assert our_residual(ours, *c)[0] == 61


def test_residual_coding_spot_values_match_putcoef(libs):
    """The same blocks, every field of the call-for-call build's coder state against the reference's putCoef."""
    ours, ref = libs
    for T, m, q, blk in spot_blocks():
        assert our_residual(ours.plain, T, m, q, blk) == ref_residual(ref, T, m, q, blk)


@pytest.mark.parametrize("T", [4, 8, 16, 32])
def test_residual_coding_matches_putcoef(libs, T):
    """Random sparse / dense / large-magnitude level blocks, every scan type: bits AND the full coder end state
    {range, low, nbits, nbytes, held byte, zero run, bytes} equal the reference's putCoef + CABAClen."""
    ours, ref = libs
    rng = np.random.default_rng(7 + T)
    for trial in range(60):
        mode = int(rng.integers(0, 35))
        q = int(rng.integers(0, 5))
        kind = trial % 6
        lev = np.zeros((T, T), np.int32)
        if kind == 0:
            k = int(rng.integers(1, 4))
            lev[rng.integers(0, T, k), rng.integers(0, T, k)] = rng.integers(-3, 4, k)
        elif kind == 1:
            lev = (rng.integers(-2, 3, (T, T)) * (rng.random((T, T)) < 0.3)).astype(np.int32)
        elif kind == 2:
            lev = rng.integers(-40, 41, (T, T)).astype(np.int32)
        elif kind == 3:
            lev[:4, :4] = rng.integers(-2000, 2001, (4, 4))
            lev[T - 1, T - 1] = 1
        elif kind == 4:
            lev = (rng.integers(-1, 2, (T, T)) * (rng.random((T, T)) < 0.05)).astype(np.int32)
        else:
            lev = np.where(rng.random((T, T)) < 0.5, 32767, -32768).astype(np.int32) * (rng.random((T, T)) < 0.2)
        want = ref_residual(ref, T, mode, q, lev)
        assert our_residual(ours.plain, T, mode, q, lev) == want, (T, mode, q, kind, trial)      # call for call: every field
        bits, st = our_residual(ours, T, mode, q, lev)                                           # merged bypass calls:
        assert bits == want[0] and (st[0], st[2]) == (want[1][0], want[1][2]), (T, mode, q, kind, trial)   # rate, range, bit position
        assert st[3] + st[6] == want[1][3] + want[1][6], (T, mode, q, kind, trial)               # bytes produced (pending + written)


def test_bypass_grouping_does_not_change_the_bytes(ours):
    """The kernel codes the bypass strings of one syntax element with one call where the reference issues several (one
    per bit for the last-position suffixes, prefix and suffix of an escape level separately).  Bypass coding is linear
    and bytes leave the coder's window at the same bit positions whatever the grouping: 300 random sequences of context
    bins and bypass strings (incl. zero runs that trigger emulation prevention) give identical byte streams."""
    n = ctypes.c_int(0)
    total = 0
    for seed in range(300):
        assert ours.hevce_stage_bypass_grouping(12345 + 7919 * seed, 400 + seed, ctypes.byref(n)) == 0, seed
        total += n.value
    assert total > 300 * 400
