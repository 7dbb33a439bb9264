"""ctypes wrapper for the host-compiled kernel simulator (tests/sim, TEST INFRASTRUCTURE ONLY)."""
import ctypes
import os
import re
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIM_DIR = os.path.join(ROOT, "tests", "sim")
SIM_SO = os.path.join(SIM_DIR, "libhevce_sim.so")
CSRC = os.path.join(ROOT, "hevc-image-encoder-lite_b200", "csrc")
_u8p = ctypes.POINTER(ctypes.c_ubyte)


def variants():
    """The kernel variants linked into the library, {tag: compile flags}, from csrc/Makefile's VARIANTS and VDEF_<tag>
    lines (the only place they are written)."""
    mk = open(os.path.join(CSRC, "Makefile")).read()
    line = lambda name: re.search(rf"^{name} := (.*)$", mk, re.M).group(1).split()
    return {tag: line(f"VDEF_{tag}") for tag in line("VARIANTS")}


def variant_flags(variant):
    return variants()[variant]


def variant_gang(variant):
    """(pictures per CTA, CTAs per picture) of a variant."""
    opt = dict(f.removeprefix("-DHEVCE_OPT_").split("=") for f in variant_flags(variant))
    return int(opt["GANG"]), int(opt.get("CLUSTER", 0)) or 1


def _build(src, so, variant, extra=()):
    srcs = [os.path.join(SIM_DIR, src), os.path.join(CSRC, "hevce_core.h"), os.path.join(CSRC, "hevce_xform_gen.h")]
    if os.path.exists(so) and all(os.path.getmtime(so) >= os.path.getmtime(s) for s in srcs):
        return
    xflags = os.environ.get("HEVCE_SIM_XFLAGS", "").split()   # development: extra -DHEVCE_OPT_... switches for an A/B candidate
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", *extra, *variant_flags(variant), *xflags, "-I", CSRC, "-o", so, srcs[0]], check=True)


def build_sim(force=False, variant="g7"):
    so = SIM_SO if variant == "g7" else SIM_SO.replace(".so", f"_{variant}.so")
    if force and os.path.exists(so):
        os.remove(so)
    _build("hevce_sim.cpp", so, variant)
    return so


_libs = {}


def sim(variant="g7"):
    if variant not in _libs:
        L = ctypes.CDLL(build_sim(variant=variant))
        L.hevce_sim_encode.restype = ctypes.c_int
        _libs[variant] = L
    return _libs[variant]


def sim_encode(img, q, order=0, max_dim=8192, variant="g7"):
    img = np.ascontiguousarray(img, dtype=np.uint8)
    h, w = img.shape
    hp, wp = (min(h, max_dim) + 31) // 32 * 32, (min(w, max_dim) + 31) // 32 * 32
    rcon = np.zeros((hp, wp), np.uint8)
    cap = 256 + 2 * hp * wp
    out = np.zeros(cap, np.uint8)
    ys, xs, err = ctypes.c_int(h), ctypes.c_int(w), ctypes.c_int(0)
    n = sim(variant).hevce_sim_encode(out.ctypes.data_as(_u8p), cap, img.ctypes.data_as(_u8p), rcon.ctypes.data_as(_u8p),
                               ctypes.byref(ys), ctypes.byref(xs), int(q), int(order), int(max_dim), ctypes.byref(err))
    assert (ys.value, xs.value) == (hp, wp)
    return out[:n].tobytes(), rcon, err.value


def sim_last_partition(shape, variant="g7"):
    """(cu_size, mode, kind) maps of the last sim_encode call; shape = padded picture shape."""
    hp, wp = shape
    cu, mode, kind = np.zeros((hp // 4, wp // 4), np.uint8), np.zeros((hp // 4, wp // 4), np.uint8), np.zeros((hp // 8, wp // 8), np.uint8)
    sim(variant).hevce_sim_last_partition(cu.ctypes.data_as(_u8p), mode.ctypes.data_as(_u8p), kind.ctypes.data_as(_u8p))
    return cu, mode, kind


# ---- gang simulator: one host thread per picture of a gang (tests/sim/hevce_simgang.cpp)
SIMGANG_SO = os.path.join(SIM_DIR, "libhevce_simgang.so")
_glibs = {}


def build_simgang(force=False, variant="g7"):
    so = SIMGANG_SO if variant == "g7" else SIMGANG_SO.replace(".so", f"_{variant}.so")
    if force and os.path.exists(so):
        os.remove(so)
    _build("hevce_simgang.cpp", so, variant, extra=("-pthread",))
    return so


def simgang(variant="g7"):
    if variant not in _glibs:
        L = ctypes.CDLL(build_simgang(variant=variant))
        L.hevce_simgang_encode.restype = ctypes.c_int
        L.hevce_simgang_size.restype = ctypes.c_int
        _glibs[variant] = L
    return _glibs[variant]


def simgang_encode(imgs, qs, order=0, variant="g7"):
    """Encode up to GANG pictures of identical size as one gang. Returns [(stream, rcon, err), ...]."""
    imgs = [np.ascontiguousarray(i, dtype=np.uint8) for i in imgs]
    n = len(imgs)
    h, w = imgs[0].shape
    assert all(i.shape == (h, w) for i in imgs)
    hp, wp = (h + 31) // 32 * 32, (w + 31) // 32 * 32
    cap = 256 + 2 * hp * wp
    outs = [np.zeros(cap, np.uint8) for _ in range(n)]
    rcons = [np.zeros((hp, wp), np.uint8) for _ in range(n)]
    arr = lambda xs: (_u8p * n)(*[x.ctypes.data_as(_u8p) for x in xs])
    qa = (ctypes.c_int * n)(*[int(q) for q in qs])
    lens, errs = (ctypes.c_int * n)(), (ctypes.c_int * n)()
    rc = simgang(variant).hevce_simgang_encode(n, arr(outs), cap, arr(imgs), arr(rcons), h, w, qa, int(order), lens, errs)
    assert rc == 0
    return [(outs[i][: lens[i]].tobytes(), rcons[i], errs[i]) for i in range(n)]


# ---- track simulator: one host thread per track of a parent || child variant (tests/sim/hevce_simtrack.cpp)
_tlibs = {}


def build_simtrack(variant="t1"):
    so = os.path.join(SIM_DIR, f"libhevce_simtrack_{variant}.so")
    _build("hevce_simtrack.cpp", so, variant, extra=("-pthread",))
    return so


def simtrack_encode(img, q, order=0, variant="t1"):
    if variant not in _tlibs:
        L = ctypes.CDLL(build_simtrack(variant))
        L.hevce_simtrack_encode.restype = ctypes.c_int
        _tlibs[variant] = L
    img = np.ascontiguousarray(img, dtype=np.uint8)
    h, w = img.shape
    hp, wp = (h + 31) // 32 * 32, (w + 31) // 32 * 32
    rcon = np.zeros((hp, wp), np.uint8)
    cap = 256 + 2 * hp * wp
    out = np.zeros(cap, np.uint8)
    ys, xs, err = ctypes.c_int(h), ctypes.c_int(w), ctypes.c_int(0)
    n = _tlibs[variant].hevce_simtrack_encode(out.ctypes.data_as(_u8p), cap, img.ctypes.data_as(_u8p), rcon.ctypes.data_as(_u8p),
                                             ctypes.byref(ys), ctypes.byref(xs), int(q), int(order), ctypes.byref(err))
    return out[:n].tobytes(), rcon, err.value
