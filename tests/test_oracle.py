"""Pin the CPU oracle (oracle/hevc_oracle.c, our restatement) before anything trusts it.

Golden sources: (1) tests/golden/small_cases.npz -- full streams + reconstructions produced by the UNMODIFIED
reference (oracle/_ref, built from /root/reference/src/HEVCe.c) for 17 inputs x qpd6 0..4; (2) the SHA-256
manifest of all 24 Kodak images x qpd6 0..4, whose qpd6=4 column is also checked against the reference's own
shipped goldens testimage_out/NN.h265 when the manifest is generated (tools/make_golden.py).
"""
import ctypes
import json
import os

import numpy as np
import pytest

import golden_util as G
import refutil as R


@pytest.mark.parametrize("name", G.small_case_names())
def test_oracle_matches_reference_small(name):
    data, meta = G.small_cases()
    img = data[f"{name}/in"]
    for q in range(5):
        s, r = R.oracle_encode(img, q)
        assert s == data[f"{name}/q{q}/stream"].tobytes(), (name, q)
        assert np.array_equal(r, data[f"{name}/q{q}/rcon"]), (name, q)
        assert R.sha(s) == meta[name]["q"][str(q)]["stream_sha256"]


def test_known_small_hashes_from_baseline_md():
    # BASELINE.md section 6 (measured in the survey): 01[0:45,0:70] at qpd6=2 -> 1531 bytes, sha 51a9bf7497b1
    data, _ = G.small_cases()
    s, r = R.oracle_encode(data["k01_45x70/in"], 2)
    assert len(s) == 1531 and R.sha(s)[:12] == "51a9bf7497b1" and R.sha(r.tobytes())[:12] == "ed24f08e9181"
    assert r.shape == (64, 96)


def test_oracle_kodak_01_q4_matches_shipped_golden():
    """One full Kodak image (7 s): oracle restatement == reference's shipped testimage_out/01.h265 (qpd6=4)."""
    imgs, man = G.kodak()
    s, r = R.oracle_encode(imgs["k01"], 4)
    assert len(s) == man["01"]["shipped_q4_len"] == 72067
    assert R.sha(s) == man["01"]["shipped_q4_sha256"] == man["01"]["q"]["4"]["stream_sha256"]
    assert R.sha(r.tobytes()) == man["01"]["q"]["4"]["rcon_sha256"]


@pytest.mark.slow
@pytest.mark.parametrize("q", range(5))
def test_oracle_kodak_all(q):
    imgs, man = G.kodak()
    for k in sorted(man):
        s, r = R.oracle_encode(imgs["k" + k], q)
        assert R.sha(s) == man[k]["q"][str(q)]["stream_sha256"], (k, q)
        assert R.sha(r.tobytes()) == man[k]["q"][str(q)]["rcon_sha256"], (k, q)


def test_generated_tables_match_reference_exports():
    """DCT/DST matrices, CABAC state tables, context init and scan orders are generated from the HEVC definitions
    in the oracle; compare with the symbols the reference library exports.  Where oracle/_ref is absent, the context
    sets are compared with the SHA-256 prefixes recorded from the reference (tests/golden/reference_tables.json); the
    matrices, state tables and scan orders are then pinned only through the end-to-end goldens."""
    orc = R.oracle()
    if not os.path.exists(R.REF_SO):
        want = json.load(open(os.path.join(G.GOLD, "reference_tables.json")))["context_set_sha256_12"]
        for q in range(5):
            mine = (ctypes.c_ubyte * 142)()
            orc.oracle_ctx_init(mine, q)
            assert R.sha(bytes(mine))[:12] == want[q], q
        return
    ref = R.ref()
    for t, (sym, n) in enumerate([("DST4_MAT", 4), ("DCT8_MAT", 8), ("DCT16_MAT", 16), ("DCT32_MAT", 32)]):
        m = np.ctypeslib.as_array((ctypes.c_int * (n * 32)).in_dll(ref, sym)).reshape(n, 32)[:, :n]
        mine = np.array([[orc.oracle_tm(t, k, i) for i in range(n)] for k in range(n)])
        assert np.array_equal(m, mine), sym
    mps = np.ctypeslib.as_array((ctypes.c_ubyte * 128).in_dll(ref, "CONTEXT_NEXT_STATE_MPS"))
    lps = np.ctypeslib.as_array((ctypes.c_ubyte * 128).in_dll(ref, "CONTEXT_NEXT_STATE_LPS"))
    assert [orc.oracle_next_state(0, c) for c in range(128)] == list(mps)
    assert [orc.oracle_next_state(1, c) for c in range(128)] == list(lps)

    class Ctx(ctypes.Structure):
        _fields_ = [("b", ctypes.c_ubyte * 142)]
    ref.newContextSet.restype = Ctx
    for q in range(5):
        mine = (ctypes.c_ubyte * 142)()
        orc.oracle_ctx_init(mine, q)
        assert bytes(ref.newContextSet(q).b) == bytes(mine)
    # scan orders
    ref.getScanOrder.restype = ctypes.c_int
    for sz, l2 in ((4, 0), (8, 1), (16, 2), (32, 3)):
        for pm, typ in ((0, 0), (26, 1), (10, 2)):
            p = ctypes.POINTER(ctypes.c_ubyte * 2)()
            got = ref.getScanOrder(sz, pm, ctypes.byref(p))
            want_type = typ if sz <= 8 else 0
            assert got == want_type
            for i in range(sz * sz):
                v = orc.oracle_scan(want_type, l2, i)
                assert (p[i][0], p[i][1]) == (v >> 5, v & 31), (sz, pm, i)


def test_header_bytes_match_reference():
    """The oracle's header bytes against the reference's putHeaderToBuffer; where oracle/_ref is absent, against the
    first bytes of every stream the reference wrote for the small goldens (five padded sizes x qpd6 0..4)."""
    orc = R.oracle()
    if not os.path.exists(R.REF_SO):
        data, _ = G.small_cases()
        for name in G.small_case_names():
            for q in range(5):
                b = (ctypes.c_ubyte * 256)()
                nb = orc.oracle_header(b, q, *data[f"{name}/q{q}/rcon"].shape)
                assert bytes(b[:nb]) == data[f"{name}/q{q}/stream"].tobytes()[:nb], (name, q)
        return
    ref = R.ref()
    for q in range(5):
        for (h, w) in ((32, 32), (512, 768), (768, 512), (2176, 3840), (8192, 8192), (64, 96)):
            a = (ctypes.c_ubyte * 256)()
            b = (ctypes.c_ubyte * 256)()
            pa = ctypes.cast(a, ctypes.POINTER(ctypes.c_ubyte))
            ppa = ctypes.pointer(pa)
            ref.putHeaderToBuffer(ppa, q, h, w)
            na = ctypes.addressof(pa.contents) - ctypes.addressof(a)
            nb = orc.oracle_header(b, q, h, w)
            assert na == nb and bytes(a[:na]) == bytes(b[:nb])
