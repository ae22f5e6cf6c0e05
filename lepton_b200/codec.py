"""ctypes binding of include/lepton_b200.h -- the host-side mirror of the reference's plug-in boundary.

Reference interface mirrored (file:line in /root/reference):
  * ``BaseEncoder::encode_chunk(const UncompressedComponents*, FileWriter*, const ThreadHandoff*, unsigned)``
    (src/lepton/base_coders.hh:59-62)  ->  :meth:`LeptonB200Codec.encode_images`
  * ``BaseDecoder::decode_chunk(UncompressedComponents*)`` (src/lepton/base_coders.hh:31)
    ->  :meth:`LeptonB200Codec.decode_images`
A :class:`CoefImage` carries what ``UncompressedComponents`` + the selected ``ThreadHandoff`` splits carry:
component geometry, quantisation tables (zig-zag order), coefficient planes in AlignedBlock order, segment starts.
Per-segment results use the reference's ExitCode values (src/vp8/util/memory.hh:13-39).
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
MAX_SEGMENTS = 16


class LeptonB200Error(RuntimeError):
    pass


def library_path() -> str:
    """The C-ABI library.  LEPB200_LIBRARY selects another build of the same sources (tuning variants built with
    `python -m lepton_b200.build --variant NAME` land in lepton_b200/variants/)."""
    return os.environ.get("LEPB200_LIBRARY") or os.path.join(HERE, "liblepton_b200.so")


class _Image(ctypes.Structure):
    _fields_ = [
        ("ncmp", ctypes.c_int32), ("mcuv", ctypes.c_int32),
        ("bch", ctypes.c_int32 * 3), ("bcv", ctypes.c_int32 * 3),
        ("trunc_bcv", ctypes.c_int32 * 3), ("trunc_bc", ctypes.c_int32 * 3),
        ("qtable_zigzag", (ctypes.c_uint16 * 64) * 3),
        ("planes", ctypes.c_void_p * 3),
        ("nseg", ctypes.c_int32),
        ("luma_y_start", ctypes.c_int32 * MAX_SEGMENTS),
        ("seg_token_bound", ctypes.c_uint32 * MAX_SEGMENTS),
    ]


class _Stream(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("len", ctypes.c_uint64), ("status", ctypes.c_int32),
                ("reserved", ctypes.c_uint32), ("ndecisions", ctypes.c_uint64)]


_LIB = None

_EXPORTS = [
    "lepb200_create", "lepb200_destroy", "lepb200_last_error", "lepb200_pinned_alloc", "lepb200_pinned_free",
    "lepb200_encode_images", "lepb200_decode_images", "lepb200_encode_upload", "lepb200_encode_launch",
    "lepb200_encode_fetch", "lepb200_decode_upload", "lepb200_decode_launch", "lepb200_decode_fetch",
    "lepb200_last_kernel_ms", "lepb200_kernel_launches", "lepb200_last_algorithmic_bytes", "lepb200_model_bytes",
    "lepb200_device_available", "lepb200_sync", "lepb200_last_symbolise_ms", "lepb200_codec_create", "lepb200_codec_destroy", "lepb200_codec_last_error",
    "lepb200_codec_ctx", "lepb200_codec_last_timing", "lepb200_codec_kernel_launches", "lepb200_codec_set_chunk_images",
    "lepb200_codec_set_gpu_huffman", "lepb200_codec_set_allow_progressive", "lepb200_codec_set_encode_threads", "lepb200_host_jpeg_open_threads", "lepb200_host_jpeg_open_split", "lepb200_codec_set_even_split", "lepb200_codec_set_verify", "lepb200_shard_by_size", "lepb200_compress_jpegs_multi", "lepb200_decompress_leps_multi", "lepb200_huffman_decode_to_device", "lepb200_encode_upload_resident", "lepb200_compress_jpegs", "lepb200_host_jpeg_open",
    "lepb200_host_jpeg_error", "lepb200_host_jpeg_image", "lepb200_host_jpeg_scan", "lepb200_last_huffman_iterations", "lepb200_huffman_encode_resident_parts", "lepb200_huffman_encode_parts", "lepb200_huffman_encode_wait_part", "lepb200_decode_fetch_status", "lepb200_decode_upload_gather", "lepb200_encode_fetch_files", "lepb200_host_jpeg_write_lep", "lepb200_host_jpeg_header", "lepb200_host_mux_plan", "lepb200_host_lep_henc_image", "lepb200_host_brotli_available", "lepb200_host_lep_lazy_equal", "lepb200_host_jpeg_close",
    "lepb200_decompress_leps", "lepb200_host_lep_open", "lepb200_host_lep_error", "lepb200_host_lep_image",
    "lepb200_host_lep_stream", "lepb200_host_lep_recode", "lepb200_host_lep_close", "lepb200_host_frontend_seconds",
]


def lib():
    """Load the C-ABI library; raises (never falls back) if it has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise LeptonB200Error("%s not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)" % path)
    L = ctypes.CDLL(path)
    for name in _EXPORTS:
        if not hasattr(L, name):
            raise LeptonB200Error("liblepton_b200.so does not export %s" % name)
    vp, ip = ctypes.c_void_p, ctypes.POINTER(_Image)
    sp = ctypes.POINTER(_Stream)
    L.lepb200_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int]
    L.lepb200_create.restype = ctypes.c_int
    L.lepb200_destroy.argtypes = [vp]
    L.lepb200_destroy.restype = None
    L.lepb200_last_error.argtypes = [vp]
    L.lepb200_last_error.restype = ctypes.c_char_p
    L.lepb200_pinned_alloc.argtypes = [ctypes.c_size_t]
    L.lepb200_pinned_alloc.restype = vp
    L.lepb200_pinned_free.argtypes = [vp]
    L.lepb200_pinned_free.restype = None
    L.lepb200_encode_images.argtypes = [vp, ip, ctypes.c_int, sp]
    L.lepb200_encode_upload.argtypes = [vp, ip, ctypes.c_int]
    L.lepb200_encode_launch.argtypes = [vp]
    L.lepb200_encode_fetch.argtypes = [vp, sp]
    L.lepb200_decode_images.argtypes = [vp, ip, ctypes.c_int, sp, ctypes.POINTER(ctypes.c_int32)]
    L.lepb200_decode_upload.argtypes = [vp, ip, ctypes.c_int, sp]
    L.lepb200_decode_launch.argtypes = [vp]
    L.lepb200_decode_fetch.argtypes = [vp, ip, ctypes.c_int, ctypes.POINTER(ctypes.c_int32)]
    for f in ("lepb200_encode_images", "lepb200_encode_upload", "lepb200_encode_launch", "lepb200_encode_fetch",
              "lepb200_decode_images", "lepb200_decode_upload", "lepb200_decode_launch", "lepb200_decode_fetch",
              "lepb200_device_available"):
        getattr(L, f).restype = ctypes.c_int
    L.lepb200_sync.argtypes = [vp]
    L.lepb200_sync.restype = ctypes.c_int
    L.lepb200_last_kernel_ms.argtypes = [vp]
    L.lepb200_last_kernel_ms.restype = ctypes.c_float
    L.lepb200_last_symbolise_ms.argtypes = [vp]
    L.lepb200_last_symbolise_ms.restype = ctypes.c_float
    L.lepb200_kernel_launches.argtypes = [vp]
    L.lepb200_kernel_launches.restype = ctypes.c_uint64
    L.lepb200_last_algorithmic_bytes.argtypes = [vp]
    L.lepb200_last_algorithmic_bytes.restype = ctypes.c_uint64
    L.lepb200_model_bytes.restype = ctypes.c_size_t
    _LIB = L
    return L


@dataclass
class CoefImage:
    """Quantised DCT coefficients of one JPEG plus the thread-segment split chosen for it."""
    ncmp: int
    mcuv: int
    bch: Sequence[int]
    bcv: Sequence[int]
    qtables_zigzag: Sequence[Sequence[int]]
    planes: List[np.ndarray]                 # per component int16 [bch*bcv, 64], AlignedBlock order
    luma_y_start: Sequence[int] = (0,)
    trunc_bcv: Optional[Sequence[int]] = None
    trunc_bc: Optional[Sequence[int]] = None
    jpeg_bytes: int = 0                       # size of the source JPEG (for MB/s accounting only)
    _keep: list = field(default_factory=list, repr=False)

    @property
    def nseg(self) -> int:
        return len(self.luma_y_start)

    def blocks(self) -> int:
        return int(sum(self.bch[c] * self.bcv[c] for c in range(self.ncmp)))

    def to_c(self) -> _Image:
        im = _Image()
        im.ncmp, im.mcuv, im.nseg = self.ncmp, self.mcuv, self.nseg
        if not (1 <= self.nseg <= MAX_SEGMENTS):
            raise LeptonB200Error("nseg out of range")
        for c in range(self.ncmp):
            p = self.planes[c]
            if p.dtype != np.int16 or not p.flags["C_CONTIGUOUS"] or p.size != self.bch[c] * self.bcv[c] * 64:
                raise LeptonB200Error("plane %d must be C-contiguous int16 of bch*bcv*64 elements" % c)
            im.bch[c], im.bcv[c] = self.bch[c], self.bcv[c]
            im.trunc_bcv[c] = self.trunc_bcv[c] if self.trunc_bcv is not None else self.bcv[c]
            im.trunc_bc[c] = self.trunc_bc[c] if self.trunc_bc is not None else self.bch[c] * self.bcv[c]
            for i in range(64):
                im.qtable_zigzag[c][i] = int(self.qtables_zigzag[c][i])
            im.planes[c] = p.ctypes.data
        for s, y in enumerate(self.luma_y_start):
            im.luma_y_start[s] = int(y)
        return im


@dataclass
class SegmentResult:
    data: bytes
    status: int
    ndecisions: int


class LeptonB200Codec:
    """One context per GPU.  ``encode_images`` / ``decode_images`` are the whole-batch equivalents of the
    reference's per-file ``encode_chunk`` / ``decode_chunk``."""

    def __init__(self, device: int = 0):
        self._L = lib()
        self._ctx = ctypes.c_void_p()
        rc = self._L.lepb200_create(ctypes.byref(self._ctx), device)
        if rc != 0:
            raise LeptonB200Error("lepb200_create(device=%d) failed with %d (no CUDA device? there is no CPU fallback)"
                                  % (device, rc))
        self.device = device

    def close(self):
        if self._ctx:
            self._L.lepb200_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise LeptonB200Error("%s failed (%d): %s" % (what, rc, self._L.lepb200_last_error(self._ctx).decode()))

    # ---- staged API -------------------------------------------------------------------------------
    def _c_images(self, images):
        arr = (_Image * len(images))()
        for i, im in enumerate(images):
            arr[i] = im.to_c()
        return arr

    def encode_upload(self, images):
        self._enc_imgs = images
        self._enc_c = self._c_images(images)
        self._check(self._L.lepb200_encode_upload(self._ctx, self._enc_c, len(images)), "encode_upload")

    def encode_launch(self):
        self._check(self._L.lepb200_encode_launch(self._ctx), "encode_launch")

    def encode_fetch(self, copy=True):
        n = sum(im.nseg for im in self._enc_imgs)
        out = (_Stream * n)()
        self._check(self._L.lepb200_encode_fetch(self._ctx, out), "encode_fetch")
        res, k = [], 0
        for im in self._enc_imgs:
            segs = []
            for _ in range(im.nseg):
                s = out[k]
                data = ctypes.string_at(s.data, s.len) if (copy and s.len) else b""
                segs.append(SegmentResult(data, s.status, s.ndecisions))
                k += 1
            res.append(segs)
        self.last_lens = [out[i].len for i in range(n)]
        return res

    def encode_images(self, images, copy=True):
        self.encode_upload(images)
        self.encode_launch()
        return self.encode_fetch(copy=copy)

    def decode_upload(self, images, streams):
        """streams: per image, a list of per-segment byte strings"""
        n = sum(im.nseg for im in images)
        arr = (_Stream * n)()
        keep, k = [], 0
        for im, segs in zip(images, streams):
            if len(segs) != im.nseg:
                raise LeptonB200Error("stream count != nseg")
            for s in segs:
                buf = np.frombuffer(s, dtype=np.uint8)
                keep.append(buf)
                arr[k].data = buf.ctypes.data if len(buf) else None
                arr[k].len = len(buf)
                k += 1
        self._dec_imgs, self._dec_keep = images, keep
        self._dec_c = self._c_images(images)
        self._check(self._L.lepb200_decode_upload(self._ctx, self._dec_c, len(images), arr), "decode_upload")

    def decode_launch(self):
        self._check(self._L.lepb200_decode_launch(self._ctx), "decode_launch")

    def decode_fetch(self, into=None):
        """Copies the planes of the last decode_launch into the uploaded images' planes and returns per-segment status
        codes.  ``into`` ({image index: list of per-component int16 arrays}) copies only those images, into those arrays."""
        n = sum(im.nseg for im in self._dec_imgs)
        st = (ctypes.c_int32 * n)()
        dst = self._dec_c
        if into is not None:
            dst = (_Image * len(self._dec_imgs))()
            for i in range(len(self._dec_imgs)):
                dst[i] = self._dec_c[i]
                for c in range(dst[i].ncmp):
                    p = into.get(i)
                    if p is not None and (p[c].dtype != np.int16 or not p[c].flags["C_CONTIGUOUS"] or p[c].size != dst[i].bch[c] * dst[i].bcv[c] * 64):
                        raise LeptonB200Error("plane %d of image %d must be C-contiguous int16 of bch*bcv*64 elements" % (c, i))
                    dst[i].planes[c] = p[c].ctypes.data if p is not None else None
        self._check(self._L.lepb200_decode_fetch(self._ctx, dst, len(self._dec_imgs), st), "decode_fetch")
        return list(st)

    def decode_images(self, images, streams):
        """Decodes into ``images[i].planes`` (pre-allocated).  Returns per-segment status codes."""
        self.decode_upload(images, streams)
        self.decode_launch()
        return self.decode_fetch()

    def sync(self):
        self._check(self._L.lepb200_sync(self._ctx), "sync")

    # ---- introspection ----------------------------------------------------------------------------
    @property
    def last_kernel_ms(self) -> float:
        return float(self._L.lepb200_last_kernel_ms(self._ctx))

    @property
    def last_symbolise_ms(self) -> float:
        return float(self._L.lepb200_last_symbolise_ms(self._ctx))

    @property
    def kernel_launches(self) -> int:
        return int(self._L.lepb200_kernel_launches(self._ctx))

    @property
    def last_algorithmic_bytes(self) -> int:
        return int(self._L.lepb200_last_algorithmic_bytes(self._ctx))


# ---------------------------------------------------------------------------------------------------------
# File-level drop-in: what the reference CLI does per file (`lepton in.jpg out.lep`), batched.
# ---------------------------------------------------------------------------------------------------------
class _Buffer(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("len", ctypes.c_size_t)]


class _Result(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("len", ctypes.c_size_t), ("status", ctypes.c_int32)]


def _bind_file_api(L):
    if getattr(L, "_file_api_bound", False):
        return
    vp = ctypes.c_void_p
    L.lepb200_codec_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int]
    L.lepb200_codec_create.restype = ctypes.c_int
    L.lepb200_codec_destroy.argtypes = [vp]
    L.lepb200_codec_destroy.restype = None
    L.lepb200_codec_last_error.argtypes = [vp]
    L.lepb200_codec_last_error.restype = ctypes.c_char_p
    L.lepb200_codec_ctx.argtypes = [vp]
    L.lepb200_codec_ctx.restype = vp
    L.lepb200_codec_last_timing.argtypes = [vp] + [ctypes.POINTER(ctypes.c_double)] * 3
    L.lepb200_codec_last_timing.restype = None
    L.lepb200_codec_kernel_launches.argtypes = [vp]
    L.lepb200_codec_kernel_launches.restype = ctypes.c_uint64
    L.lepb200_codec_set_chunk_images.argtypes = [vp, ctypes.c_int]
    L.lepb200_codec_set_chunk_images.restype = None
    L.lepb200_codec_set_gpu_huffman.argtypes = [vp, ctypes.c_int]
    L.lepb200_codec_set_gpu_huffman.restype = None
    L.lepb200_codec_set_allow_progressive.argtypes = [vp, ctypes.c_int]
    L.lepb200_codec_set_allow_progressive.restype = None
    L.lepb200_codec_set_encode_threads.argtypes = [vp, ctypes.c_int, ctypes.c_int]
    L.lepb200_codec_set_encode_threads.restype = None
    L.lepb200_codec_last_huffman_ms.argtypes = [vp]
    L.lepb200_codec_last_huffman_ms.restype = ctypes.c_double
    L.lepb200_codec_last_gpu_recoded.argtypes = [vp]
    L.lepb200_codec_last_gpu_recoded.restype = ctypes.c_int
    L.lepb200_compress_jpegs.argtypes = [vp, ctypes.POINTER(_Buffer), ctypes.c_int, ctypes.POINTER(_Result)]
    L.lepb200_compress_jpegs.restype = ctypes.c_int
    L.lepb200_host_jpeg_open.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_int32)]
    L.lepb200_host_jpeg_open.restype = ctypes.c_int
    L.lepb200_host_jpeg_open_threads.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_int32)]
    L.lepb200_host_jpeg_open_threads.restype = ctypes.c_int
    L.lepb200_host_jpeg_open_split.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_int32)]
    L.lepb200_host_jpeg_open_split.restype = ctypes.c_int
    L.lepb200_codec_set_even_split.argtypes = [vp, ctypes.c_int]
    L.lepb200_codec_set_even_split.restype = None
    L.lepb200_codec_set_verify.argtypes = [vp, ctypes.c_int]
    L.lepb200_codec_set_verify.restype = None
    L.lepb200_host_jpeg_error.argtypes = [vp]
    L.lepb200_host_jpeg_error.restype = ctypes.c_char_p
    L.lepb200_host_jpeg_image.argtypes = [vp, ctypes.POINTER(_Image)]
    L.lepb200_host_jpeg_image.restype = ctypes.c_int
    L.lepb200_host_jpeg_write_lep.argtypes = [vp, ctypes.POINTER(_Stream), ctypes.c_int, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_size_t)]
    L.lepb200_host_jpeg_write_lep.restype = ctypes.c_int
    L.lepb200_host_jpeg_close.argtypes = [vp]
    L.lepb200_host_jpeg_close.restype = None
    L.lepb200_decompress_leps.argtypes = [vp, ctypes.POINTER(_Buffer), ctypes.c_int, ctypes.POINTER(_Result)]
    L.lepb200_decompress_leps.restype = ctypes.c_int
    L.lepb200_host_lep_open.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_int32)]
    L.lepb200_host_lep_open.restype = ctypes.c_int
    L.lepb200_host_lep_error.argtypes = [vp]
    L.lepb200_host_lep_error.restype = ctypes.c_char_p
    L.lepb200_host_lep_image.argtypes = [vp, ctypes.POINTER(_Image)]
    L.lepb200_host_lep_image.restype = ctypes.c_int
    L.lepb200_host_lep_stream.argtypes = [vp, ctypes.c_int, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_size_t)]
    L.lepb200_host_lep_stream.restype = ctypes.c_int
    L.lepb200_host_lep_recode.argtypes = [vp, ctypes.c_void_p * 3, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_size_t)]
    L.lepb200_host_lep_recode.restype = ctypes.c_int
    L.lepb200_host_lep_close.argtypes = [vp]
    L.lepb200_host_lep_close.restype = None
    L._file_api_bound = True


class HostJpeg:
    """Host stages only (no GPU): parse + Huffman-decode a JPEG, expose it as a CoefImage, assemble a .lep."""

    def __init__(self, data: bytes, min_threads: int = 1, max_threads: int = 8, even_split: bool = False):
        self._L = lib()
        _bind_file_api(self._L)
        self._h = ctypes.c_void_p()
        st = ctypes.c_int32()
        self._data = data
        self._L.lepb200_host_jpeg_open_split(data, len(data), min_threads, max_threads, 1 if even_split else 0, ctypes.byref(self._h), ctypes.byref(st))
        self.status = st.value
        self.error = self._L.lepb200_host_jpeg_error(self._h).decode()

    def close(self):
        if self._h:
            self._L.lepb200_host_jpeg_close(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def coef_image(self) -> CoefImage:
        if self.status:
            raise LeptonB200Error("JPEG front end refused the file: status %d (%s)" % (self.status, self.error))
        im = _Image()
        if self._L.lepb200_host_jpeg_image(self._h, ctypes.byref(im)) != 0:
            raise LeptonB200Error("host_jpeg_image failed")
        planes = []
        for c in range(im.ncmp):
            n = im.bch[c] * im.bcv[c]
            arr = np.ctypeslib.as_array(ctypes.cast(im.planes[c], ctypes.POINTER(ctypes.c_int16)), shape=(n, 64))
            planes.append(arr)          # view into memory owned by this HostJpeg
        return CoefImage(ncmp=im.ncmp, mcuv=im.mcuv, bch=[im.bch[c] for c in range(im.ncmp)],
                         bcv=[im.bcv[c] for c in range(im.ncmp)],
                         qtables_zigzag=[[im.qtable_zigzag[c][i] for i in range(64)] for c in range(im.ncmp)],
                         planes=planes, luma_y_start=[im.luma_y_start[s] for s in range(im.nseg)],
                         jpeg_bytes=len(self._data), _keep=[self])

    def write_lep(self, streams: Sequence[bytes]) -> bytes:
        arr = (_Stream * len(streams))()
        keep = []
        for i, s in enumerate(streams):
            b = np.frombuffer(s, dtype=np.uint8)
            keep.append(b)
            arr[i].data = b.ctypes.data if len(b) else None
            arr[i].len = len(b)
        d, n = ctypes.c_void_p(), ctypes.c_size_t()
        if self._L.lepb200_host_jpeg_write_lep(self._h, arr, len(streams), ctypes.byref(d), ctypes.byref(n)) != 0:
            raise LeptonB200Error("write_lep failed: %s" % self._L.lepb200_host_jpeg_error(self._h).decode())
        return ctypes.string_at(d, n.value)


class HostLep:
    """Decode-side host stages only (no GPU): parse a .lep, expose geometry / splits / segment streams, and
    re-create the JPEG bytes from coefficient planes."""

    def __init__(self, data: bytes):
        self._L = lib()
        _bind_file_api(self._L)
        self._h = ctypes.c_void_p()
        st = ctypes.c_int32()
        self._data = data
        self._L.lepb200_host_lep_open(data, len(data), ctypes.byref(self._h), ctypes.byref(st))
        self.status = st.value
        self.error = self._L.lepb200_host_lep_error(self._h).decode()

    def close(self):
        if self._h:
            self._L.lepb200_host_lep_close(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def coef_image(self) -> CoefImage:
        """Geometry + splits with freshly allocated (zero) planes to decode into."""
        if self.status:
            raise LeptonB200Error(".lep reader refused the file: status %d (%s)" % (self.status, self.error))
        im = _Image()
        if self._L.lepb200_host_lep_image(self._h, ctypes.byref(im)) != 0:
            raise LeptonB200Error("host_lep_image failed")
        planes = [np.zeros((im.bch[c] * im.bcv[c], 64), dtype=np.int16) for c in range(im.ncmp)]
        return CoefImage(ncmp=im.ncmp, mcuv=im.mcuv, bch=[im.bch[c] for c in range(im.ncmp)],
                         bcv=[im.bcv[c] for c in range(im.ncmp)],
                         qtables_zigzag=[[im.qtable_zigzag[c][i] for i in range(64)] for c in range(im.ncmp)],
                         planes=planes, luma_y_start=[im.luma_y_start[s] for s in range(im.nseg)])

    def scan_layout(self):
        """(offset, length) of the entropy-coded scan in the original JPEG, (0, 0) if the host has to re-encode it."""
        off, n = ctypes.c_uint32(), ctypes.c_uint32()
        if self._L.lepb200_host_lep_scan_layout(self._h, ctypes.byref(off), ctypes.byref(n)) != 0:
            raise LeptonB200Error("host_lep_scan_layout failed")
        return off.value, n.value

    def assemble(self, scan: bytes) -> bytes:
        """JPEG bytes around a scan that was Huffman-encoded elsewhere (the device)."""
        d, n = ctypes.c_void_p(), ctypes.c_size_t()
        if self._L.lepb200_host_lep_assemble(self._h, scan, len(scan), ctypes.byref(d), ctypes.byref(n)) != 0:
            raise LeptonB200Error("host_lep_assemble failed: " + self._L.lepb200_host_lep_error(self._h).decode())
        return ctypes.string_at(d, n.value)

    def streams(self, nseg: int):
        out = []
        for s in range(nseg):
            d, n = ctypes.c_void_p(), ctypes.c_size_t()
            if self._L.lepb200_host_lep_stream(self._h, s, ctypes.byref(d), ctypes.byref(n)) != 0:
                raise LeptonB200Error("host_lep_stream failed")
            out.append(ctypes.string_at(d, n.value))
        return out

    def recode(self, planes) -> bytes:
        arr = (ctypes.c_void_p * 3)()
        keep = []
        for i, p in enumerate(planes):
            q = np.ascontiguousarray(p, dtype=np.int16)
            keep.append(q)
            arr[i] = q.ctypes.data
        d, n = ctypes.c_void_p(), ctypes.c_size_t()
        if self._L.lepb200_host_lep_recode(self._h, arr, ctypes.byref(d), ctypes.byref(n)) != 0:
            raise LeptonB200Error("recode failed: %s" % self._L.lepb200_host_lep_error(self._h).decode())
        return ctypes.string_at(d, n.value)


class LeptonB200FileCodec:
    """JPEG bytes -> .lep bytes for a batch of files; host threads + one GPU."""

    def __init__(self, device: int = 0, host_threads: int = 0, chunk_images: int = 0, gpu_huffman: bool = True,
                 allow_progressive: bool = True, min_encode_threads: int = 1, max_encode_threads: int = 8,
                 even_split: bool = False, verify: bool = False):
        self._L = lib()
        _bind_file_api(self._L)
        self._c = ctypes.c_void_p()
        rc = self._L.lepb200_codec_create(ctypes.byref(self._c), device, host_threads)
        if rc != 0:
            raise LeptonB200Error("lepb200_codec_create(device=%d) failed with %d (no CUDA device? there is no CPU fallback)" % (device, rc))
        if chunk_images > 0:
            self._L.lepb200_codec_set_chunk_images(self._c, chunk_images)
        self._L.lepb200_codec_set_gpu_huffman(self._c, 1 if gpu_huffman else 0)
        self._L.lepb200_codec_set_allow_progressive(self._c, 1 if allow_progressive else 0)      # False = -rejectprogressive
        self._L.lepb200_codec_set_encode_threads(self._c, min_encode_threads, max_encode_threads)   # -minencodethreads= / -maxencodethreads=
        self._L.lepb200_codec_set_even_split(self._c, 1 if even_split else 0)                      # -evensplit
        self._L.lepb200_codec_set_verify(self._c, 1 if verify else 0)                              # -verify (reference default) / -skipverify

    def close(self):
        if self._c:
            self._L.lepb200_codec_destroy(self._c)
            self._c = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def prepare(files: Sequence[bytes]):
        """Build the C argument array (pointer + length per file) once, for callers that submit the same host buffers
        repeatedly; the ctypes marshalling of thousands of pointers is harness overhead, not part of the codec."""
        n = len(files)
        bufs = (_Buffer * n)()
        keep = []
        for i, j in enumerate(files):
            b = np.frombuffer(j, dtype=np.uint8)
            keep.append(b)
            bufs[i].data = b.ctypes.data
            bufs[i].len = len(b)
        return (bufs, n, keep, (_Result * n)())

    def compress(self, jpegs, copy: bool = True):
        """-> list of (status, lep_bytes).  `jpegs` is a sequence of bytes objects or a handle from prepare().
        With copy=False only lengths are materialised (benchmarking)."""
        bufs, n, _keep, res = jpegs if isinstance(jpegs, tuple) else self.prepare(jpegs)
        rc = self._L.lepb200_compress_jpegs(self._c, bufs, n, res)
        if rc != 0:
            raise LeptonB200Error("compress_jpegs failed (%d): %s" % (rc, self._L.lepb200_codec_last_error(self._c).decode()))
        if not copy:
            return [(res[i].status, res[i].len) for i in range(n)]
        return [(res[i].status, ctypes.string_at(res[i].data, res[i].len) if res[i].len else b"") for i in range(n)]

    def decompress(self, leps, copy: bool = True):
        """.lep bytes -> JPEG bytes; -> list of (status, jpeg_bytes).  `leps`: bytes objects or a handle from prepare()."""
        bufs, n, _keep, res = leps if isinstance(leps, tuple) else self.prepare(leps)
        rc = self._L.lepb200_decompress_leps(self._c, bufs, n, res)
        if rc != 0:
            raise LeptonB200Error("decompress_leps failed (%d): %s" % (rc, self._L.lepb200_codec_last_error(self._c).decode()))
        if not copy:
            return [(res[i].status, res[i].len) for i in range(n)]
        return [(res[i].status, ctypes.string_at(res[i].data, res[i].len) if res[i].len else b"") for i in range(n)]

    @staticmethod
    def results(handle, indices, copy: bool = True):
        """(status, bytes) of files ``indices`` of the last compress / decompress call made with a prepare() handle, also
        after copy=False (with copy=False: (status, length)).  The bytes belong to the codec that made them and are valid
        until its next call."""
        res = handle[3]
        if not copy:
            return [(res[i].status, res[i].len) for i in indices]
        return [(res[i].status, ctypes.string_at(res[i].data, res[i].len) if res[i].len else b"") for i in indices]

    @property
    def last_gpu_recoded(self):
        return int(self._L.lepb200_codec_last_gpu_recoded(self._c))

    def last_timing(self):
        a, b, c = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
        self._L.lepb200_codec_last_timing(self._c, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
        return {"front_s": a.value, "gpu_s": b.value, "back_s": c.value,
                "huffman_kernel_ms_last_chunk": float(self._L.lepb200_codec_last_huffman_ms(self._c))}

    @property
    def kernel_launches(self) -> int:
        return int(self._L.lepb200_codec_kernel_launches(self._c))


def shard_by_size_native(sizes, world):
    """lepb200_shard_by_size: owner (codec / GPU index) of every file, longest-first by size -- the native twin of
    lepton_b200.sharding.shard_by_size."""
    L = lib()
    n = len(sizes)
    arr = (ctypes.c_size_t * n)(*sizes)
    owner = (ctypes.c_int * n)()
    L.lepb200_shard_by_size.argtypes = [ctypes.POINTER(ctypes.c_size_t), ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
    L.lepb200_shard_by_size.restype = None
    L.lepb200_shard_by_size(arr, n, world, owner)
    return list(owner)


class LeptonB200MultiGpuFileCodec:
    """One process, several GPUs: a LeptonB200FileCodec per device, files dealt to them balanced by bytes
    (lepb200_compress_jpegs_multi / lepb200_decompress_leps_multi); no data crosses between GPUs."""

    def __init__(self, devices, host_threads_per_gpu: int = 0, **kw):
        self.codecs = [LeptonB200FileCodec(d, host_threads=host_threads_per_gpu, **kw) for d in devices]
        self._L = self.codecs[0]._L
        vp = ctypes.c_void_p
        self._arr = (vp * len(self.codecs))(*[c._c for c in self.codecs])
        for f in (self._L.lepb200_compress_jpegs_multi, self._L.lepb200_decompress_leps_multi):
            f.argtypes = [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
            f.restype = ctypes.c_int

    def _run(self, fn, files):
        bufs, n, _keep, res = self.codecs[0].prepare(files)
        rc = fn(self._arr, len(self.codecs), ctypes.cast(bufs, ctypes.c_void_p), n, ctypes.cast(res, ctypes.c_void_p))
        if rc != 0:
            raise LeptonB200Error("multi-GPU call failed (%d)" % rc)
        return [(res[i].status, ctypes.string_at(res[i].data, res[i].len) if res[i].len else b"") for i in range(n)]

    def compress(self, jpegs):
        return self._run(self._L.lepb200_compress_jpegs_multi, jpegs)

    def decompress(self, leps):
        return self._run(self._L.lepb200_decompress_leps_multi, leps)

    def close(self):
        for c in self.codecs:
            c.close()
