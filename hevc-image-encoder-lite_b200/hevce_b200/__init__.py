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
METRIC_PSNR, METRIC_SSIM = 0, 1

_u8p = ctypes.POINTER(ctypes.c_ubyte)
_ip = ctypes.POINTER(ctypes.c_int)

EXPORTS = [
    "HEVCImageEncoder", "HEVCImageEncoderBatch", "hevce_set_devices", "hevce_set_max_dim", "hevce_version",
    "hevce_measure_int_peak", "hevce_session_create", "hevce_session_upload", "hevce_session_encode",
    "hevce_session_download", "hevce_session_kernel_ms", "hevce_session_commit_ms", "hevce_session_launches", "hevce_session_grid",
    "hevce_session_h2d_bytes", "hevce_session_d2h_bytes", "hevce_session_destroy",
    "hevce_session_quality", "hevce_session_quality_ms", "hevce_session_partition",
    "hevce_set_variant", "hevce_session_variant", "hevce_get_max_dim", "hevce_release",
    "HEVCImageEncoderBatchDecoded", "hevce_session_deblock", "hevce_session_deblock_ms", "hevce_session_download_decoded",
    "hevce_session_decoded_quality",
    "hevce_stream_info", "HEVCImageDecoderBatch", "hevce_decoder_create", "hevce_decoder_upload", "hevce_decoder_run",
    "hevce_decoder_download", "hevce_decoder_parse_ms", "hevce_decoder_recon_ms", "hevce_decoder_deblock_ms", "hevce_decoder_destroy",
    "hevce_session_ssim", "hevce_session_ssim_ms", "HEVCImageEncoderBatchTarget",
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
        L.HEVCImageEncoderBatchDecoded.restype = ctypes.c_int
        L.HEVCImageEncoderBatchDecoded.argtypes = [ctypes.c_int] + [ctypes.POINTER(_u8p)] * 4 + [_ip, _ip, _ip, _ip]
        _dp = ctypes.POINTER(ctypes.c_double)
        L.HEVCImageEncoderBatchTarget.restype = ctypes.c_int
        L.HEVCImageEncoderBatchTarget.argtypes = [ctypes.c_int] + [ctypes.POINTER(_u8p)] * 4 + [_ip, _ip, ctypes.c_int, _dp, _ip, _dp, _ip]
        L.hevce_session_ssim.restype = ctypes.c_int
        L.hevce_session_ssim.argtypes = [ctypes.c_void_p, ctypes.c_int, _dp]
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
        for f in ("hevce_session_quality", "hevce_session_decoded_quality"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
        L.hevce_session_deblock.restype = ctypes.c_int
        L.hevce_session_deblock.argtypes = [ctypes.c_void_p]
        L.hevce_session_download_decoded.restype = ctypes.c_int
        L.hevce_session_download_decoded.argtypes = [ctypes.c_void_p, ctypes.POINTER(_u8p)]
        L.hevce_session_partition.restype = ctypes.c_int
        L.hevce_session_partition.argtypes = [ctypes.c_void_p, ctypes.c_int, _u8p, _u8p, _u8p]
        for f in ("hevce_session_kernel_ms", "hevce_session_commit_ms", "hevce_session_quality_ms", "hevce_session_deblock_ms",
                  "hevce_session_ssim_ms"):
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
        L.hevce_stream_info.restype = ctypes.c_int
        L.hevce_stream_info.argtypes = [_u8p, ctypes.c_int, _ip, _ip, _ip]
        L.HEVCImageDecoderBatch.restype = ctypes.c_int
        L.HEVCImageDecoderBatch.argtypes = [ctypes.c_int, ctypes.POINTER(_u8p), _ip, ctypes.POINTER(_u8p), _ip]
        L.hevce_decoder_create.restype = ctypes.c_void_p
        L.hevce_decoder_create.argtypes = [ctypes.c_int]
        L.hevce_decoder_upload.restype = ctypes.c_int
        L.hevce_decoder_upload.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(_u8p), _ip]
        L.hevce_decoder_run.restype = ctypes.c_int
        L.hevce_decoder_run.argtypes = [ctypes.c_void_p]
        L.hevce_decoder_download.restype = ctypes.c_int
        L.hevce_decoder_download.argtypes = [ctypes.c_void_p, ctypes.POINTER(_u8p), _ip]
        for f in ("hevce_decoder_parse_ms", "hevce_decoder_recon_ms", "hevce_decoder_deblock_ms"):
            getattr(L, f).restype = ctypes.c_float
            getattr(L, f).argtypes = [ctypes.c_void_p]
        L.hevce_decoder_destroy.restype = None
        L.hevce_decoder_destroy.argtypes = [ctypes.c_void_p]
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


def HEVCImageEncoder(img, qpd6):
    """One picture through the drop-in C entry point. Returns (stream bytes, reconstruction HxW uint8).
    Output buffers are sized from the library's own size limit (hevce_get_max_dim)."""
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


def alloc_outputs(shapes):
    """Caller-owned output buffers (stream, reconstruction) for pictures of the given shapes; reusable across calls,
    exactly like the pbuffer / img_rcon arrays a C caller keeps."""
    return _out_buffers(shapes, get_max_dim())


def HEVCImageEncoderBatch(imgs, qpd6, outputs=None, copy_streams=True):
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


def HEVCImageEncoderBatchDecoded(imgs, qpd6, outputs=None):
    """HEVCImageEncoderBatch that also returns the decoded pictures: the reconstructions after the in-loop deblocking
    filter, which is what a conforming decoder shows for the streams.  Returns (streams, recons, decoded).
    outputs: (streams, recons, decoded) buffers to reuse, e.g. alloc_outputs() plus one more list like recons."""
    imgs = [np.ascontiguousarray(i, dtype=np.uint8) for i in imgs]
    n = len(imgs)
    qs = [int(qpd6)] * n if np.isscalar(qpd6) else [int(q) for q in qpd6]
    limit = get_max_dim()
    if outputs is not None:
        outs, rcons, decs = outputs
    else:
        outs, rcons = _out_buffers([i.shape for i in imgs], limit)
        decs = [np.zeros_like(r) for r in rcons]
    for i, o, r, d in zip(imgs, outs, rcons, decs):   # the library clamps with ITS limit: never hand it a smaller buffer
        need = padded(i.shape[0], limit) * padded(i.shape[1], limit)
        if r.size < need or d.size < need or o.size < 256 + 2 * need:
            raise HevceError(ERR_ARG, "HEVCImageEncoderBatchDecoded: output buffers smaller than the library's size limit requires")
    ys = (ctypes.c_int * n)(*[i.shape[0] for i in imgs])
    xs = (ctypes.c_int * n)(*[i.shape[1] for i in imgs])
    qa = (ctypes.c_int * n)(*qs)
    lens = (ctypes.c_int * n)()
    rc = lib().HEVCImageEncoderBatchDecoded(n, _ptr_array(outs), _ptr_array(imgs), _ptr_array(rcons), _ptr_array(decs), ys, xs, qa, lens)
    if rc < 0:
        raise HevceError(rc, "HEVCImageEncoderBatchDecoded")
    return [outs[i][: lens[i]].tobytes() for i in range(n)], rcons, decs


def HEVCImageEncoderBatchTarget(imgs, target, metric="ssim", decoded=False):
    """Each picture at the coarsest qpd6 whose decoded picture meets `target` (scalar or one per picture): SSIM
    (metric="ssim", hevce_session_ssim of the decoded picture) or PSNR in dB (metric="psnr").  The search rule is that of
    include/hevce.h; a picture no qpd6 satisfies gets qpd6 0, and its quality shows it missed the target.
    Returns (streams, recons, qpd6, quality), with the decoded pictures after recons when decoded=True."""
    metrics = {"psnr": METRIC_PSNR, "ssim": METRIC_SSIM}
    if metric not in metrics:
        raise HevceError(ERR_ARG, f"HEVCImageEncoderBatchTarget: metric must be one of {sorted(metrics)}")
    imgs = [np.ascontiguousarray(i, dtype=np.uint8) for i in imgs]
    n = len(imgs)
    tg = np.full(n, float(target)) if np.isscalar(target) else np.ascontiguousarray(target, dtype=np.float64)
    if tg.shape != (n,):
        raise HevceError(ERR_ARG, "HEVCImageEncoderBatchTarget: one target per picture")
    outs, rcons = _out_buffers([i.shape for i in imgs], get_max_dim())
    decs = [np.zeros_like(r) for r in rcons] if decoded else None
    ys = (ctypes.c_int * n)(*[i.shape[0] for i in imgs])
    xs = (ctypes.c_int * n)(*[i.shape[1] for i in imgs])
    qs = np.zeros(n, np.int32)
    qual = np.zeros(n, np.float64)
    lens = (ctypes.c_int * n)()
    dp = ctypes.POINTER(ctypes.c_double)
    rc = lib().HEVCImageEncoderBatchTarget(n, _ptr_array(outs), _ptr_array(imgs), _ptr_array(rcons), _ptr_array(decs) if decoded else None,
                                           ys, xs, metrics[metric], tg.ctypes.data_as(dp), qs.ctypes.data_as(_ip), qual.ctypes.data_as(dp), lens)
    if rc < 0:
        raise HevceError(rc, "HEVCImageEncoderBatchTarget")
    streams = [outs[i][: lens[i]].tobytes() for i in range(n)]
    return (streams, rcons, decs, qs, qual) if decoded else (streams, rcons, qs, qual)


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

    def __init__(self, device, shapes, qpd6):
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

    def deblock(self):
        """Run the in-loop deblocking filter over the last encode's reconstructions on the device; returns its kernel ms."""
        rc = lib().hevce_session_deblock(self._h)
        if rc < 0:
            raise HevceError(rc, "hevce_session_deblock")
        return lib().hevce_session_deblock_ms(self._h)

    @property
    def deblock_ms(self):
        return lib().hevce_session_deblock_ms(self._h)

    def download_decoded(self):
        """The decoded pictures (padded, like the reconstructions) after deblock()."""
        decs = [np.zeros((padded(h, self.max_dim), padded(w, self.max_dim)), np.uint8) for h, w in self.shapes]
        rc = lib().hevce_session_download_decoded(self._h, _ptr_array(decs))
        if rc < 0:
            raise HevceError(rc, "hevce_session_download_decoded")
        return decs

    def decoded_quality(self):
        """(mse, psnr) of every decoded picture against its source, as quality() does for the reconstructions."""
        mse, psnr = np.zeros(self.n, np.float64), np.zeros(self.n, np.float64)
        dp = ctypes.POINTER(ctypes.c_double)
        rc = lib().hevce_session_decoded_quality(self._h, mse.ctypes.data_as(dp), psnr.ctypes.data_as(dp))
        if rc < 0:
            raise HevceError(rc, "hevce_session_decoded_quality")
        return mse, psnr

    def ssim(self, decoded=False):
        """Mean SSIM of every picture, reduced on the device: the coded picture (the source padded by edge replication)
        against the reconstruction of the last encode, or with decoded=True against the decoded picture after deblock()."""
        out = np.zeros(self.n, np.float64)
        rc = lib().hevce_session_ssim(self._h, 1 if decoded else 0, out.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
        if rc < 0:
            raise HevceError(rc, "hevce_session_ssim")
        return out

    @property
    def ssim_ms(self):
        return lib().hevce_session_ssim_ms(self._h)

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


# ---- f6: decoding the streams this library writes --------------------------------------------------------------
def _streams(streams):
    arrs = [np.frombuffer(bytes(s), np.uint8).copy() for s in streams]
    return arrs, (ctypes.c_int * len(arrs))(*[a.size for a in arrs])


def stream_info(stream):
    """(ysz, xsz, qpd6) of a stream this library wrote: its padded size and qpd6.  A header check on the host, no device.
    Raises HevceError(ERR_ARG) for a stream whose parameter sets are not the ones this library writes."""
    a = np.frombuffer(bytes(stream), np.uint8).copy()
    y, x, q = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    rc = lib().hevce_stream_info(a.ctypes.data_as(_u8p), int(a.size), ctypes.byref(y), ctypes.byref(x), ctypes.byref(q))
    if rc < 0:
        raise HevceError(rc, "hevce_stream_info")
    return y.value, x.value, q.value


def HEVCImageDecoderBatch(streams, return_status=False):
    """Decode streams of this library on the device: the decoded pictures at their padded size (what
    HEVCImageEncoderBatchDecoded returns as decoded).  A stream whose slice data does not parse raises HevceError(ERR_STATE),
    unless return_status: then (pictures, status) is returned, status[i] 0 or ERR_STATE (that picture is all zeros)."""
    arrs, lens = _streams(streams)
    n = len(arrs)
    decs = []
    for a in arrs:
        y, x, _ = stream_info(a)
        decs.append(np.zeros((y, x), np.uint8))
    st = (ctypes.c_int * n)()
    rc = lib().HEVCImageDecoderBatch(n, _ptr_array(arrs), lens, _ptr_array(decs), st)
    if rc < 0 and not (return_status and rc == ERR_STATE):
        raise HevceError(rc, "HEVCImageDecoderBatch")
    return (decs, list(st)) if return_status else decs


class Decoder:
    """Device-resident decoder on one GPU: upload streams, run the parse / reconstruction / deblocking kernels (timed with
    CUDA events), download the decoded pictures."""

    def __init__(self, device=0):
        self._h = lib().hevce_decoder_create(int(device))
        if not self._h:
            raise HevceError(ERR_CUDA, "hevce_decoder_create")
        self.shapes = []

    def upload(self, streams):
        arrs, lens = _streams(streams)
        shapes = [stream_info(a)[:2] for a in arrs]
        rc = lib().hevce_decoder_upload(self._h, len(arrs), _ptr_array(arrs), lens)
        if rc < 0:
            raise HevceError(rc, "hevce_decoder_upload")
        self.shapes = shapes

    def run(self):
        """Decode the uploaded streams (synchronous); returns the three kernels' total ms."""
        rc = lib().hevce_decoder_run(self._h)
        if rc < 0:
            raise HevceError(rc, "hevce_decoder_run")
        return self.parse_ms + self.recon_ms + self.deblock_ms

    def download(self, return_status=False):
        decs = [np.zeros(s, np.uint8) for s in self.shapes]
        st = (ctypes.c_int * max(1, len(decs)))()
        rc = lib().hevce_decoder_download(self._h, _ptr_array(decs), st)
        if rc < 0 and not (return_status and rc == ERR_STATE):
            raise HevceError(rc, "hevce_decoder_download")
        return (decs, list(st)[:len(decs)]) if return_status else decs

    @property
    def parse_ms(self):
        return lib().hevce_decoder_parse_ms(self._h)

    @property
    def recon_ms(self):
        return lib().hevce_decoder_recon_ms(self._h)

    @property
    def deblock_ms(self):
        return lib().hevce_decoder_deblock_ms(self._h)

    def close(self):
        if self._h:
            lib().hevce_decoder_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
