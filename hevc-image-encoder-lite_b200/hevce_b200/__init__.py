"""hevce_b200 -- Python host-side binding of libhevce_b200.so (ctypes over the C ABI in include/hevce.h).

Mirrors the reference's one-function interface (HEVCe.h:5-12): ``HEVCImageEncoder(img, qpd6)`` returns the byte
stream and the padded reconstruction exactly as the C entry point fills ``pbuffer`` / ``img_rcon``, and
``HEVCImageEncoderBatch`` does the same for a list of pictures.  All work happens in the sm_100a kernels of the
shared library; there is no Python or CPU implementation behind these calls -- importing works without a GPU (so
the symbol table can be checked), calling raises ``HevceError`` when no CUDA device is usable.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "libhevce_b200.so")

ERR_ARG, ERR_CUDA, ERR_STATE = -1, -2, -3

_u8p = ctypes.POINTER(ctypes.c_ubyte)
_ip = ctypes.POINTER(ctypes.c_int)

EXPORTS = [
    "HEVCImageEncoder", "HEVCImageEncoderBatch", "hevce_set_devices", "hevce_set_max_dim", "hevce_version",
    "hevce_measure_int_peak", "hevce_session_create", "hevce_session_upload", "hevce_session_encode",
    "hevce_session_download", "hevce_session_kernel_ms", "hevce_session_commit_ms", "hevce_session_launches", "hevce_session_grid",
    "hevce_session_h2d_bytes", "hevce_session_d2h_bytes", "hevce_session_destroy",
    "hevce_session_quality", "hevce_session_quality_ms", "hevce_session_partition",
    "hevce_set_variant", "hevce_session_variant", "hevce_get_max_dim", "hevce_release",
]


class HevceError(RuntimeError):
    def __init__(self, code, what):
        names = {ERR_ARG: "invalid argument", ERR_CUDA: "CUDA device/runtime unavailable", ERR_STATE: "internal consistency check failed"}
        super().__init__(f"{what}: {names.get(code, 'error')} ({code})")
        self.code = code


_lib = None


def lib():
    """Load libhevce_b200.so (built in-tree by `make -C hevc-image-encoder-lite_b200/csrc`). No fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HevceError(ERR_CUDA, f"{LIB_PATH} is missing (run __graft_entry__.build())")
        L = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_LOCAL)
        L.HEVCImageEncoder.restype = ctypes.c_int
        L.HEVCImageEncoder.argtypes = [_u8p, _u8p, _u8p, _ip, _ip, ctypes.c_int]
        L.HEVCImageEncoderBatch.restype = ctypes.c_int
        L.HEVCImageEncoderBatch.argtypes = [ctypes.c_int, ctypes.POINTER(_u8p), ctypes.POINTER(_u8p), ctypes.POINTER(_u8p), _ip, _ip, _ip, _ip]
        L.hevce_set_devices.restype = ctypes.c_int
        L.hevce_set_devices.argtypes = [ctypes.c_int, _ip]
        L.hevce_set_max_dim.restype = ctypes.c_int
        L.hevce_set_max_dim.argtypes = [ctypes.c_int]
        L.hevce_get_max_dim.restype = ctypes.c_int
        L.hevce_get_max_dim.argtypes = []
        L.hevce_release.restype = None
        L.hevce_release.argtypes = []
        L.hevce_version.restype = ctypes.c_char_p
        L.hevce_set_variant.restype = ctypes.c_int
        L.hevce_set_variant.argtypes = [ctypes.c_char_p]
        L.hevce_session_variant.restype = ctypes.c_char_p
        L.hevce_session_variant.argtypes = [ctypes.c_void_p]
        L.hevce_measure_int_peak.restype = ctypes.c_double
        L.hevce_measure_int_peak.argtypes = [ctypes.c_int]
        L.hevce_session_create.restype = ctypes.c_void_p
        L.hevce_session_create.argtypes = [ctypes.c_int, ctypes.c_int, _ip, _ip, _ip]
        for f in ("hevce_session_upload",):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [ctypes.c_void_p, ctypes.POINTER(_u8p)]
        L.hevce_session_encode.restype = ctypes.c_int
        L.hevce_session_encode.argtypes = [ctypes.c_void_p]
        L.hevce_session_download.restype = ctypes.c_int
        L.hevce_session_download.argtypes = [ctypes.c_void_p, ctypes.POINTER(_u8p), ctypes.POINTER(_u8p), _ip]
        L.hevce_session_quality.restype = ctypes.c_int
        L.hevce_session_quality.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
        L.hevce_session_partition.restype = ctypes.c_int
        L.hevce_session_partition.argtypes = [ctypes.c_void_p, ctypes.c_int, _u8p, _u8p, _u8p]
        for f in ("hevce_session_kernel_ms", "hevce_session_commit_ms", "hevce_session_quality_ms"):
            getattr(L, f).restype = ctypes.c_float
            getattr(L, f).argtypes = [ctypes.c_void_p]
        for f in ("hevce_session_launches", "hevce_session_grid"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [ctypes.c_void_p]
        for f in ("hevce_session_h2d_bytes", "hevce_session_d2h_bytes"):
            getattr(L, f).restype = ctypes.c_longlong
            getattr(L, f).argtypes = [ctypes.c_void_p]
        L.hevce_session_destroy.restype = None
        L.hevce_session_destroy.argtypes = [ctypes.c_void_p]
        _lib = L
    return _lib


def padded(n, limit=None):
    """Size after the clamp to the library's limit (default 8192, hevce_set_max_dim) and padding to a multiple of 32."""
    return (min(int(n), limit or get_max_dim()) + 31) // 32 * 32


def _ptr_array(arrs):
    return (_u8p * len(arrs))(*[a.ctypes.data_as(_u8p) for a in arrs])


def _out_buffers(shapes, limit):
    rcons = [np.zeros((padded(h, limit), padded(w, limit)), np.uint8) for h, w in shapes]
    outs = [np.zeros(256 + 2 * r.size, np.uint8) for r in rcons]
    return outs, rcons


def HEVCImageEncoder(img, qpd6, max_dim=None):
    """One picture through the drop-in C entry point. Returns (stream bytes, reconstruction HxW uint8).
    Output buffers are sized from the library's own size limit (hevce_get_max_dim), not from an argument."""
    max_dim = get_max_dim()
    img = np.ascontiguousarray(img, dtype=np.uint8)
    if img.ndim != 2:
        raise HevceError(ERR_ARG, "HEVCImageEncoder needs a 2-D uint8 array")
    (out,), (rcon,) = _out_buffers([img.shape], max_dim)
    ys, xs = ctypes.c_int(img.shape[0]), ctypes.c_int(img.shape[1])
    n = lib().HEVCImageEncoder(out.ctypes.data_as(_u8p), img.ctypes.data_as(_u8p), rcon.ctypes.data_as(_u8p),
                               ctypes.byref(ys), ctypes.byref(xs), int(qpd6))
    if n < 0:
        raise HevceError(n, "HEVCImageEncoder")
    assert (ys.value, xs.value) == rcon.shape
    return out[:n].tobytes(), rcon


def alloc_outputs(shapes, max_dim=None):
    """Caller-owned output buffers (stream, reconstruction) for pictures of the given shapes; reusable across calls,
    exactly like the pbuffer / img_rcon arrays a C caller keeps."""
    return _out_buffers(shapes, get_max_dim())


def HEVCImageEncoderBatch(imgs, qpd6, max_dim=None, outputs=None, copy_streams=True):
    """n pictures in one call (sharded over the selected GPUs). qpd6: int or sequence. Returns (streams, recons).
    outputs: buffers from alloc_outputs() to reuse; copy_streams=False returns views into them instead of bytes."""
    imgs = [np.ascontiguousarray(i, dtype=np.uint8) for i in imgs]
    n = len(imgs)
    qs = [int(qpd6)] * n if np.isscalar(qpd6) else [int(q) for q in qpd6]
    limit = get_max_dim()
    outs, rcons = outputs if outputs is not None else _out_buffers([i.shape for i in imgs], limit)
    for i, o, r in zip(imgs, outs, rcons):      # the library clamps with ITS limit: never hand it a smaller buffer
        need = padded(i.shape[0], limit) * padded(i.shape[1], limit)
        if r.size < need or o.size < 256 + 2 * need:
            raise HevceError(ERR_ARG, "HEVCImageEncoderBatch: output buffers smaller than the library's size limit requires")
    ys = (ctypes.c_int * n)(*[i.shape[0] for i in imgs])
    xs = (ctypes.c_int * n)(*[i.shape[1] for i in imgs])
    qa = (ctypes.c_int * n)(*qs)
    lens = (ctypes.c_int * n)()
    rc = lib().HEVCImageEncoderBatch(n, _ptr_array(outs), _ptr_array(imgs), _ptr_array(rcons), ys, xs, qa, lens)
    if rc < 0:
        raise HevceError(rc, "HEVCImageEncoderBatch")
    if not copy_streams:
        return [outs[i][: lens[i]] for i in range(n)], rcons
    return [outs[i][: lens[i]].tobytes() for i in range(n)], rcons


def set_devices(ordinals):
    arr = (ctypes.c_int * len(ordinals))(*ordinals)
    rc = lib().hevce_set_devices(len(ordinals), arr)
    if rc < 0:
        raise HevceError(rc, "hevce_set_devices")


def set_variant(name=None):
    """Kernel variant for the following batches: "g7", "g4", "g2", "w1", "t1", "c2", or None / "auto" to choose per batch."""
    rc = lib().hevce_set_variant(name.encode() if name else None)
    if rc < 0:
        raise HevceError(rc, "hevce_set_variant")


def set_max_dim(v):
    return lib().hevce_set_max_dim(int(v))


def get_max_dim():
    return lib().hevce_get_max_dim()


def release():
    """Free the library's cached sessions (HBM buffers and pinned staging of earlier calls)."""
    lib().hevce_release()


def measure_int_peak(device=0):
    v = lib().hevce_measure_int_peak(int(device))
    if v < 0:
        raise HevceError(int(v), "hevce_measure_int_peak")
    return v


class Session:
    """Device-resident batch on one GPU: upload once, encode (timed with CUDA events), download."""

    def __init__(self, device, shapes, qpd6, max_dim=None):
        n = len(shapes)
        self.n, self.shapes, self.max_dim = n, list(shapes), get_max_dim()
        qs = [int(qpd6)] * n if np.isscalar(qpd6) else [int(q) for q in qpd6]
        ys = (ctypes.c_int * n)(*[s[0] for s in shapes])
        xs = (ctypes.c_int * n)(*[s[1] for s in shapes])
        qa = (ctypes.c_int * n)(*qs)
        self._h = lib().hevce_session_create(int(device), n, ys, xs, qa)
        if not self._h:
            raise HevceError(ERR_CUDA, "hevce_session_create")

    def upload(self, imgs):
        imgs = [np.ascontiguousarray(i, dtype=np.uint8) for i in imgs]
        assert [i.shape for i in imgs] == [tuple(s) for s in self.shapes]
        rc = lib().hevce_session_upload(self._h, _ptr_array(imgs))
        if rc < 0:
            raise HevceError(rc, "hevce_session_upload")

    def encode(self):
        rc = lib().hevce_session_encode(self._h)
        if rc < 0:
            raise HevceError(rc, "hevce_session_encode")
        return lib().hevce_session_kernel_ms(self._h)

    @property
    def commit_ms(self):
        return lib().hevce_session_commit_ms(self._h)

    def download(self):
        outs, rcons = _out_buffers(self.shapes, self.max_dim)
        lens = (ctypes.c_int * self.n)()
        rc = lib().hevce_session_download(self._h, _ptr_array(outs), _ptr_array(rcons), lens)
        if rc < 0:
            raise HevceError(rc, "hevce_session_download")
        return [outs[i][: lens[i]].tobytes() for i in range(self.n)], rcons

    def quality(self):
        """(mse, psnr) of every picture of the last encode, reduced on the device (calcImagePSNR, HEVCeMain.c:116-133)."""
        mse, psnr = np.zeros(self.n, np.float64), np.zeros(self.n, np.float64)
        dp = ctypes.POINTER(ctypes.c_double)
        rc = lib().hevce_session_quality(self._h, mse.ctypes.data_as(dp), psnr.ctypes.data_as(dp))
        if rc < 0:
            raise HevceError(rc, "hevce_session_quality")
        return mse, psnr

    @property
    def quality_ms(self):
        return lib().hevce_session_quality_ms(self._h)

    def partition(self, i):
        """Decisions of picture i: (cu_size, mode) per 4x4 unit and kind per 8x8 unit (0 one TU, 1 four TUs, 2 NxN)."""
        h, w = padded(self.shapes[i][0], self.max_dim), padded(self.shapes[i][1], self.max_dim)
        cu, mode, kind = np.zeros((h // 4, w // 4), np.uint8), np.zeros((h // 4, w // 4), np.uint8), np.zeros((h // 8, w // 8), np.uint8)
        rc = lib().hevce_session_partition(self._h, int(i), cu.ctypes.data_as(_u8p), mode.ctypes.data_as(_u8p), kind.ctypes.data_as(_u8p))
        if rc < 0:
            raise HevceError(rc, "hevce_session_partition")
        return cu, mode, kind

    @property
    def launches(self):
        return lib().hevce_session_launches(self._h)

    @property
    def grid(self):
        return lib().hevce_session_grid(self._h)

    @property
    def variant(self):
        return lib().hevce_session_variant(self._h).decode()

    @property
    def h2d_bytes(self):
        return lib().hevce_session_h2d_bytes(self._h)

    @property
    def d2h_bytes(self):
        return lib().hevce_session_d2h_bytes(self._h)

    def close(self):
        if self._h:
            lib().hevce_session_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
