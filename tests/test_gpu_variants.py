"""Every kernel variant of the library (hevce_variants.h: gangs of 7 / 4 / 2 pictures per CTA, the wide one-picture
variant and the parent || child one-picture variant) must produce the reference's bytes: the same committed goldens and live CPU checks, once per forced variant,
through the C ABI.  Short gangs (fewer same-size pictures than a CTA holds) leave slots empty instead of repeating work;
the automatic choice is checked for the batch shapes BASELINE.json names."""
import os

import numpy as np
import pytest

import golden_util as G
import refutil as R
import simutil as S
import workloads as WL

pytestmark = pytest.mark.gpu
VARIANTS = tuple(S.variants())


@pytest.fixture(scope="module")
def H():
    import hevce_b200
    assert os.path.exists(hevce_b200.LIB_PATH), "libhevce_b200.so missing: the CUDA extension must be built in-tree"
    yield hevce_b200
    hevce_b200.set_variant(None)


def checker():
    return R.ref() if os.path.exists(R.REF_SO) else R.oracle()


@pytest.mark.parametrize("variant", VARIANTS)
def test_variant_ragged_goldens(H, variant):
    """85 pictures of 17 different sizes x 5 qpd6 in one call: every gang is short (5 same-size pictures)."""
    H.set_variant(variant)
    data, _ = G.small_cases()
    imgs, qs, keys = [], [], []
    for n in G.small_case_names():
        for q in range(5):
            imgs.append(data[f"{n}/in"]); qs.append(q); keys.append((n, q))
    streams, rcons = H.HEVCImageEncoderBatch(imgs, qs)
    for (n, q), s, r in zip(keys, streams, rcons):
        assert s == data[f"{n}/q{q}/stream"].tobytes(), (variant, n, q)
        assert np.array_equal(r, data[f"{n}/q{q}/rcon"]), (variant, n, q)


@pytest.mark.parametrize("variant", VARIANTS)
def test_variant_full_and_short_gangs_vs_live_checker(H, variant):
    """23 same-size pictures (full gangs plus a short one for every gang size) with mixed qpd6 against the CPU checker."""
    H.set_variant(variant)
    K = WL.kodak_landscape()
    imgs = [WL.config3_image(40 + i, K)[11 * i:11 * i + 64, 17 * i:17 * i + 96].copy() for i in range(23)]
    qs = [(3 * i + 1) % 5 for i in range(23)]
    ses = H.Session(0, [i.shape for i in imgs], qs)
    assert ses.variant == variant
    ses.upload(imgs)
    ses.encode()
    streams, rcons = ses.download()
    ses.close()
    lib = checker()
    for i, (im, q, s, r) in enumerate(zip(imgs, qs, streams, rcons)):
        ws, wr = R.encode_with(lib, im, q)
        assert s == ws and np.array_equal(r, wr), (variant, i, q)


def test_variants_agree_on_kodak_size(H):
    """One Kodak-size picture (384 CTUs, all node sizes and CU kinds occur) per variant: identical streams, and equal
    to the reference manifest."""
    imgs, man = G.kodak()
    want = man["23"]["q"]["4"]
    for v in VARIANTS:
        H.set_variant(v)
        s, r = H.HEVCImageEncoder(imgs["k23"], 4)
        assert len(s) == want["len"] and R.sha(s) == want["stream_sha256"] and R.sha(r.tobytes()) == want["rcon_sha256"], v
        assert R.sha(s) == man["23"]["shipped_q4_sha256"]


def test_automatic_choice(H):
    H.set_variant(None)
    shape = [(64, 64)]
    for n, want in ((1, ("w1", "t1", "c2")), (100, ("w1", "t1", "c2")), (148 * 7, ("g7",)), (148 * 7 * 3, ("g7",))):
        ses = H.Session(0, shape * n, 2)
        got = ses.variant
        ses.close()
        assert got in want, (n, got)      # few pictures: one picture per CTA; whole waves of 7: the 7-picture gangs
    for n in (148 * 2, 148 * 4):          # between the extremes any variant is legal; the estimate must fill the GPU
        ses = H.Session(0, shape * n, 2)
        assert ses.grid == 148, (n, ses.variant, ses.grid)
        ses.close()
    with pytest.raises(H.HevceError):
        H.set_variant("g9")
