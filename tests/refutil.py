"""ctypes access to the two CPU checkers (TEST INFRASTRUCTURE ONLY).

* ``ref()``    -> oracle/_ref/libhevce_ref.so : the UNMODIFIED reference, compiled by ``make -C oracle``
                  straight from /root/reference/src/HEVCe.c (never copied into this repo).
* ``oracle()`` -> oracle/libhevc_oracle.so    : our own plain-C restatement (oracle/hevc_oracle.c).

Both export ``HEVCImageEncoder`` with the reference prototype (HEVCe.h:5-12).  Nothing in the product
package imports this module.
"""
import ctypes
import hashlib
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libhevce_ref.so")
ORACLE_SO = os.path.join(ORACLE_DIR, "libhevc_oracle.so")

_u8p = ctypes.POINTER(ctypes.c_ubyte)
_ip = ctypes.POINTER(ctypes.c_int)


def build_oracles():
    subprocess.run(["make", "-C", ORACLE_DIR], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)


def _load(path):
    if not os.path.exists(path):
        build_oracles()
    lib = ctypes.CDLL(path, mode=ctypes.RTLD_LOCAL)
    lib.HEVCImageEncoder.restype = ctypes.c_int
    lib.HEVCImageEncoder.argtypes = [_u8p, _u8p, _u8p, _ip, _ip, ctypes.c_int]
    return lib


_cache = {}


def ref():
    if "ref" not in _cache:
        _cache["ref"] = _load(REF_SO)
    return _cache["ref"]


def oracle():
    if "oracle" not in _cache:
        _cache["oracle"] = _load(ORACLE_SO)
    return _cache["oracle"]


def padded(n, limit=8192):
    return (min(n, limit) + 31) // 32 * 32


def encode_with(lib, img, qpd6):
    """Run ``HEVCImageEncoder`` of ``lib`` on a 2-D uint8 array. Returns (stream bytes, recon array)."""
    img = np.ascontiguousarray(img, dtype=np.uint8)
    h, w = img.shape
    hp, wp = padded(h), padded(w)
    rcon = np.zeros((hp, wp), dtype=np.uint8)
    cap = 256 + hp * wp * 2 + (hp // 32) * (wp // 32) * 64
    buf = np.zeros(cap, dtype=np.uint8)
    ys, xs = ctypes.c_int(h), ctypes.c_int(w)
    n = lib.HEVCImageEncoder(buf.ctypes.data_as(_u8p), img.ctypes.data_as(_u8p), rcon.ctypes.data_as(_u8p),
                             ctypes.byref(ys), ctypes.byref(xs), int(qpd6))
    assert (ys.value, xs.value) == (hp, wp), (ys.value, xs.value, hp, wp)
    return buf[:n].tobytes(), rcon


def ref_encode(img, qpd6):
    return encode_with(ref(), img, qpd6)


def oracle_encode(img, qpd6):
    return encode_with(oracle(), img, qpd6)


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def report_figures(img, rcon, n):
    """The result lines the reference CLI prints (HEVCeMain.c) for input `img`, reconstruction `rcon` and an n-byte
    stream: sizes, ratio, bits per pixel, MSE over the overlap of the two sizes (floored at 1e-9) and PSNR."""
    hp, wp = rcon.shape
    hm, wm = min(img.shape[0], hp), min(img.shape[1], wp)
    mse = max(float(((img[:hm, :wm].astype(np.int64) - rcon[:hm, :wm]) ** 2).sum()) / hm / wm, 1e-9)
    return [f"  padded image size               = {wp} x {hp}",
            f"  original   length               = {wp * hp} Bytes",
            f"  compressed length               = {n} Bytes",
            f"  compression ratio               = {wp * hp / n:.5f}",
            f"  bits per pixel                  = {8.0 * n / (wp * hp):.5f}",
            f"  mean square error (MSE)         = {mse:.7f}",
            f"  peak signal/noise ratio (PSNR)  = {10.0 * np.log10(255 * 255 / mse):.4f} dB"]


def read_pgm(path):
    with open(path, "rb") as f:
        data = f.read()
    # P5\n<w> <h>\n255\n
    parts = data.split(b"\n", 3)
    assert parts[0] == b"P5"
    w, h = map(int, parts[1].split())
    assert parts[2] == b"255"
    return np.frombuffer(parts[3][: w * h], dtype=np.uint8).reshape(h, w).copy()
