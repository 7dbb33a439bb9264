"""The C-ABI shared library loads without a GPU and exports exactly what include/hevce.h declares."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = os.path.join(ROOT, "include", "hevce.h")


def _ensure_built():
    import hevce_b200
    if not os.path.exists(hevce_b200.LIB_PATH):
        subprocess.run(["make", "-C", os.path.join(ROOT, "hevc-image-encoder-lite_b200", "csrc")], check=True)
    return hevce_b200


def _declared():
    src = open(HDR).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = "\n".join(l for l in src.splitlines() if not l.lstrip().startswith("#"))
    return sorted(set(re.findall(r"HEVCE_API[^;(]*?\b(\w+)\s*\(", src)))


def test_header_symbols_exported():
    H = _ensure_built()
    lib = H.lib()
    names = _declared()
    assert "HEVCImageEncoder" in names and "HEVCImageEncoderBatch" in names and len(names) >= 16
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(H.EXPORTS) == names


def test_only_declared_symbols_are_exported():
    H = _ensure_built()
    out = subprocess.run(["nm", "-D", "--defined-only", H.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = sorted(l.split()[-1] for l in out.splitlines() if l.strip() and l.split()[-2] in "TDBR")
    assert exported == _declared(), exported   # the reference exports predict/transform/...; we must not collide


def test_argument_validation_needs_no_gpu():
    H = _ensure_built()
    lib = H.lib()
    u8p = ctypes.POINTER(ctypes.c_ubyte)
    img = np.zeros((32, 32), np.uint8)
    out = np.zeros(4096, np.uint8)
    ys, xs = ctypes.c_int(32), ctypes.c_int(32)
    p = lambda a: a.ctypes.data_as(u8p)
    assert lib.HEVCImageEncoder(p(out), p(img), p(img.copy()), ctypes.byref(ys), ctypes.byref(xs), 5) == H.ERR_ARG
    assert lib.HEVCImageEncoder(p(out), p(img), p(img.copy()), ctypes.byref(ys), ctypes.byref(xs), -1) == H.ERR_ARG
    assert lib.HEVCImageEncoder(None, p(img), p(img.copy()), ctypes.byref(ys), ctypes.byref(xs), 2) == H.ERR_ARG
    ys0 = ctypes.c_int(0)
    assert lib.HEVCImageEncoder(p(out), p(img), p(img.copy()), ctypes.byref(ys0), ctypes.byref(xs), 2) == H.ERR_ARG
    assert lib.HEVCImageEncoderBatch(0, None, None, None, None, None, None, None) == 0
    assert lib.HEVCImageEncoderBatch(-1, None, None, None, None, None, None, None) == H.ERR_ARG
    assert (ys.value, xs.value) == (32, 32)


def test_set_variant_accepts_every_makefile_variant():
    """hevce_set_variant knows every kernel variant csrc/Makefile builds (HEVCE_VARIANT_LIST is in step with it) and
    rejects any other tag.  No GPU needed: the variant table is filled by host-side functions only."""
    import simutil as S
    H = _ensure_built()
    try:
        for tag in S.variants():
            H.set_variant(tag)
        with pytest.raises(H.HevceError):
            H.set_variant("g9")
    finally:
        H.set_variant(None)


def test_no_cpu_fallback():
    """Without a CUDA device the product must fail loudly, never fall back to a CPU path."""
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("GPU present")
    except ImportError:
        pass
    H = _ensure_built()
    with pytest.raises(H.HevceError) as e:
        H.HEVCImageEncoder(np.zeros((32, 32), np.uint8), 2)
    assert e.value.code == H.ERR_CUDA


def test_product_does_not_reference_oracle():
    pkg = os.path.join(ROOT, "hevc-image-encoder-lite_b200")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".c", ".cu", ".h", ".py", ".cuh", "Makefile")):
                txt = open(os.path.join(d, f), errors="ignore").read()
                assert "oracle" not in txt.lower() or f == "hevce_core.h" and "the oracle inside the build container" in txt, os.path.join(d, f)
