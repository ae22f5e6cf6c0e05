"""CPU emulation of the decode kernels (test infrastructure).

The kernel sources compile as host C++ through `cuda_shim.h`, which runs every CUDA thread of a CTA as a fiber and
implements the warp collectives and `__syncthreads` among them, so `lep_decode.cu` (warp per segment) and
`lep_decode_g2.cu` (G lanes per segment, 32 / G segments per warp in lock step) execute with real 32-lane warps, divergence,
votes and shuffles included, and can be pinned to the oracle bit for bit without a GPU.  The GPU parity tests then
confirm the same sources on the device; what the emulator cannot show is timing and memory-system behaviour.
"""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "lepton_b200", "csrc")
OUT = os.path.join(HERE, "_build", "libemu_kernels.so")
SOURCES = [os.path.join(HERE, "emu_kernels.cc"), os.path.join(HERE, "cuda_shim.h"), os.path.join(HERE, "fake", "cuda_runtime.h"),
           os.path.join(CSRC, "lep_encode.cu"), os.path.join(CSRC, "lep_decode.cu"), os.path.join(CSRC, "lep_decode_g2.cu"),
           os.path.join(CSRC, "lep_huff.cu"), os.path.join(CSRC, "lep_huffpar.cu"), os.path.join(CSRC, "lep_mux.cu"), os.path.join(CSRC, "lep_huffenc.cu"), os.path.join(CSRC, "lep_common.cuh"), os.path.join(CSRC, "lep_predict.cuh"), os.path.join(ROOT, "include", "lepton_b200.h")]

KERNEL_WARP = 0


def KERNEL_G2(lanes):
    """lep_decode_g2_kernel<lanes>: `lanes` lanes per thread-segment, 32 / lanes segments per warp in lock step."""
    assert lanes in (1, 2, 4, 8, 16, 32)
    return 200 + lanes


_LIB = None


def build(out=OUT, defines=()):
    if os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in SOURCES):
        return out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    # compile to a private name and rename: parallel test workers may build at once, and none may load a half-written file
    tmp = "%s.%d.tmp" % (out, os.getpid())
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", "-I", os.path.join(HERE, "fake"),
                           "-Wno-unknown-pragmas"] + ["-D" + d for d in defines] + ["-o", tmp, os.path.join(HERE, "emu_kernels.cc")])
    os.replace(tmp, out)
    return out


def use_variant(name, defines):
    """Switches this module to a build of the harness with extra -D defines (e.g. another model layout)."""
    global _LIB
    _LIB = ctypes.CDLL(build(os.path.join(HERE, "_build", "libemu_kernels_%s.so" % name), defines))
    _LIB.emu_decode_images.restype = ctypes.c_int
    _LIB.emu_encode_images.restype = ctypes.c_int


def use_default():
    global _LIB
    _LIB = None


def lib():
    global _LIB
    if _LIB is None:
        # LEPB200_EMU_LIB: another build of the harness, e.g. the AddressSanitizer one of tests/tools_emu_sanitize.py
        _LIB = ctypes.CDLL(os.environ.get("LEPB200_EMU_LIB") or build())
        _LIB.emu_decode_images.restype = ctypes.c_int
        _LIB.emu_encode_images.restype = ctypes.c_int
    return _LIB


def decode_images(kernel, images, streams, grid_cap=0):
    """Same contract as LeptonB200Codec.decode_images: decodes into images[i].planes, returns (status, ndecisions) per segment."""
    from lepton_b200.codec import _Image, _Stream
    n = sum(im.nseg for im in images)
    arr = (_Stream * n)()
    keep, k = [], 0
    for im, segs in zip(images, streams):
        assert len(segs) == im.nseg
        for s in segs:
            buf = np.frombuffer(bytes(s), dtype=np.uint8)
            keep.append(buf)
            arr[k].data = buf.ctypes.data if len(buf) else None
            arr[k].len = len(buf)
            k += 1
    cim = (_Image * len(images))(*[im.to_c() for im in images])
    st = (ctypes.c_int32 * n)()
    nd = (ctypes.c_uint64 * n)()
    rc = lib().emu_decode_images(int(kernel), int(grid_cap), cim, len(images), arr, st, nd)
    if rc != 0:
        raise RuntimeError("emu_decode_images failed with %d" % rc)
    return list(st), list(nd)


ENC_KERNEL_A = 0


def encode_images(images, grid_cap=0, kernel=0):
    """Same contract as LeptonB200Codec.encode_images: per image a list of (status, bytes, ndecisions) per segment."""
    from lepton_b200.codec import _Image, _Stream
    n = sum(im.nseg for im in images)
    cim = (_Image * len(images))(*[im.to_c() for im in images])
    out = (_Stream * n)()
    cap = sum(im.blocks() for im in images) * 64 + 8192 * n
    arena = (ctypes.c_uint8 * cap)()
    rc = lib().emu_encode_images(int(kernel), int(grid_cap), cim, len(images), out, arena, ctypes.c_size_t(cap))
    if rc != 0:
        raise RuntimeError("emu_encode_images failed with %d" % rc)
    res, k = [], 0
    for im in images:
        segs = []
        for _ in range(im.nseg):
            o = out[k]
            segs.append((o.status, ctypes.string_at(o.data, o.len) if o.len else b"", int(o.ndecisions)))
            k += 1
        res.append(segs)
    return res


# ---- baseline Huffman decode kernels (lep_huff.cu, lep_huffpar.cu)
class _HuffTable(ctypes.Structure):
    _fields_ = [("bits", ctypes.c_uint8 * 17), ("vals", ctypes.c_uint8 * 256)]


class _HuffRow(ctypes.Structure):
    _fields_ = [("bitpos", ctypes.c_uint32), ("lastdc", ctypes.c_int16 * 3), ("mcu_y", ctypes.c_int16), ("tokens", ctypes.c_uint32)]


class _Scan(ctypes.Structure):
    _fields_ = [("entropy", ctypes.c_void_p), ("nbytes", ctypes.c_uint32), ("ncmp", ctypes.c_int32), ("mcuh", ctypes.c_int32),
                ("mcuv", ctypes.c_int32), ("rsti", ctypes.c_int32), ("H", ctypes.c_int32 * 3), ("V", ctypes.c_int32 * 3),
                ("nch", ctypes.c_int32 * 3), ("ncv", ctypes.c_int32 * 3), ("dc", _HuffTable * 3), ("ac", _HuffTable * 3),
                ("status", ctypes.c_int32), ("padbit", ctypes.c_int32), ("end_bitpos", ctypes.c_uint32), ("nrows", ctypes.c_int32),
                ("rows", ctypes.POINTER(_HuffRow))]


HUFF_SERIAL, HUFF_SUBSEQ = 0, 1


def huffman_decode(mode, jpegs, sub_bits=4096, iter_cap=62, mutate=None):
    """Huffman-decodes whole JPEG files with the emulated kernels.  mode HUFF_SERIAL: lep_huffdecode_kernel (one warp per
    image); HUFF_SUBSEQ: the sub-sequence kernels of lep_huffpar.cu, then lep_huffdecode_kernel for what they left.
    Returns (results, info): per file None when the host front end does not hand the file to the GPU decoder, else a dict
    with status, padbit, end_bitpos, rows [(bitpos, lastdc, mcu_y, tokens)], planes [ndarray(blocks, 64)], host_planes;
    info = (synchronisation iterations, images the serial kernel had to redo).  `mutate(i, bytearray)` may damage the
    de-stuffed entropy bytes of file i before decoding."""
    from lepton_b200.codec import HostJpeg, lib as product_lib
    L = product_lib()
    L.lepb200_host_jpeg_scan.argtypes = [ctypes.c_void_p, ctypes.POINTER(_Scan)]
    L.lepb200_host_jpeg_scan.restype = ctypes.c_int
    hjs, scans, idx, keep = [], [], [], []
    for i, data in enumerate(jpegs):
        hj = HostJpeg(data)
        hjs.append(hj)
        sc = _Scan()
        if hj.status != 0 or L.lepb200_host_jpeg_scan(hj._h, ctypes.byref(sc)) != 0:
            continue
        if mutate is not None:
            buf = bytearray(ctypes.string_at(sc.entropy, sc.nbytes))
            mutate(i, buf)
            arr = (ctypes.c_uint8 * len(buf)).from_buffer(buf)
            keep.append((buf, arr))
            sc.entropy = ctypes.addressof(arr)
            sc.nbytes = len(buf)
        rows = (_HuffRow * (sc.mcuv + 1))()
        keep.append(rows)
        sc.rows = ctypes.cast(rows, ctypes.POINTER(_HuffRow))
        scans.append(sc)
        idx.append(i)
    n = len(scans)
    res = [None] * len(jpegs)
    if n == 0:
        return res, (0, 0)
    arr = (_Scan * n)(*scans)
    planes, pp = [], (ctypes.POINTER(ctypes.c_int16) * (3 * n))()
    for k, sc in enumerate(scans):
        ps = []
        for c in range(sc.ncmp):
            a = np.zeros((sc.mcuh * sc.H[c] * sc.mcuv * sc.V[c], 64), np.int16)
            ps.append(a)
            pp[3 * k + c] = a.ctypes.data_as(ctypes.POINTER(ctypes.c_int16))
        planes.append(ps)
    info = (ctypes.c_int * 2)()
    f = lib().emu_huffman_decode
    f.restype = ctypes.c_int
    rc = f(int(mode), int(sub_bits), int(iter_cap), arr, n, pp, info)
    if rc != 0:
        raise RuntimeError("emu_huffman_decode failed with %d" % rc)
    for k, i in enumerate(idx):
        sc = arr[k]
        rows = [(sc.rows[r].bitpos, tuple(sc.rows[r].lastdc), sc.rows[r].mcu_y, sc.rows[r].tokens) for r in range(max(0, min(sc.nrows, sc.mcuv + 1)))]
        host = [np.array(p) for p in hjs[i].coef_image().planes] if mutate is None else None
        res[i] = dict(status=sc.status, padbit=sc.padbit, end_bitpos=sc.end_bitpos, nrows=sc.nrows, rows=rows, planes=planes[k], host_planes=host)
    return res, (info[0], info[1])


# ---- device container assembly (lep_mux.cu)
class _MuxPacket(ctypes.Structure):
    _fields_ = [("id", ctypes.c_uint8), ("nhdr", ctypes.c_uint8), ("hdr", ctypes.c_uint8 * 3), ("src_off", ctypes.c_uint32), ("len", ctypes.c_uint32)]


def mux_plan(lens):
    """lepb200_host_mux_plan of the PRODUCT library (host code, no GPU): the MuxWriter schedule for streams of these lengths."""
    import lepton_b200
    L = lepton_b200.lib()
    L.lepb200_host_mux_plan.restype = ctypes.c_int
    L.lepb200_host_mux_plan.argtypes = [ctypes.POINTER(ctypes.c_size_t), ctypes.c_int, ctypes.POINTER(_MuxPacket), ctypes.c_int]
    arr = (ctypes.c_size_t * len(lens))(*lens)
    n = L.lepb200_host_mux_plan(arr, len(lens), None, 0)
    assert n >= 0
    out = (_MuxPacket * max(n, 1))()
    assert L.lepb200_host_mux_plan(arr, len(lens), out, n) == n
    return out, n


def mux_files(files, grid=3):
    """files: list of (header bytes, [stream bytes per segment]).  Returns the assembled .lep files (lep_gather_kernel on the
    emulator over the pieces the C ABI would build)."""
    from lepton_b200.codec import _Stream
    nf = len(files)
    hdrs = [ctypes.create_string_buffer(h, len(h)) for h, _ in files]
    hdr_p = (ctypes.c_void_p * nf)(*[ctypes.cast(h, ctypes.c_void_p) for h in hdrs])
    hlen = (ctypes.c_size_t * nf)(*[len(h) for h, _ in files])
    nseg = (ctypes.c_int * nf)(*[len(ss) for _, ss in files])
    flat = [s for _, ss in files for s in ss]
    keep = [ctypes.create_string_buffer(s, max(len(s), 1)) for s in flat]
    st = (_Stream * max(len(flat), 1))()
    for k, (s, b) in enumerate(zip(flat, keep)):
        st[k].data = ctypes.cast(b, ctypes.c_void_p).value
        st[k].len = len(s)
    plans, first = [], [0]
    for _, ss in files:
        p, n = mux_plan([len(s) for s in ss])
        plans.extend(p[i] for i in range(n))
        first.append(first[-1] + n)
    plan = (_MuxPacket * max(len(plans), 1))(*plans)
    pf = (ctypes.c_uint32 * (nf + 1))(*first)
    cap = sum(len(h) + sum(len(s) for s in ss) for h, ss in files) * 2 + 4096 * nf
    out = (ctypes.c_uint8 * cap)()
    off = (ctypes.c_size_t * nf)()
    ln = (ctypes.c_size_t * nf)()
    L = lib()
    L.emu_mux_files.restype = ctypes.c_int
    rc = L.emu_mux_files(nf, hdr_p, hlen, nseg, st, plan, pf, int(grid), out, ctypes.c_size_t(cap), off, ln)
    if rc != 0:
        raise RuntimeError("emu_mux_files failed with %d" % rc)
    raw = bytes(out)
    return [raw[off[f]:off[f] + ln[f]] for f in range(nf)]


# ---- baseline Huffman encode for the way back (lep_huffenc.cu)
class _HEncSegment(ctypes.Structure):
    _fields_ = [("mcu_row_start", ctypes.c_int32), ("mcu_row_end", ctypes.c_int32), ("last_dc", ctypes.c_int16 * 3),
                ("overhang_bits", ctypes.c_uint8), ("overhang_byte", ctypes.c_uint8), ("expect_bytes", ctypes.c_uint32)]


class _HEncImage(ctypes.Structure):
    _fields_ = [("rsti", ctypes.c_int32), ("padbit", ctypes.c_int32), ("H", ctypes.c_int32 * 3), ("V", ctypes.c_int32 * 3),
                ("dc", _HuffTable * 3), ("ac", _HuffTable * 3), ("nseg", ctypes.c_int32), ("seg", _HEncSegment * 16),
                ("scan_bytes", ctypes.c_uint32), ("data", ctypes.c_void_p), ("status", ctypes.c_int32)]


def henc_job(host_lep):
    """lepb200_host_lep_henc_image of the PRODUCT library (host code): the job the device Huffman encoder gets for this .lep."""
    L = host_lep._L
    L.lepb200_host_lep_henc_image.restype = ctypes.c_int
    L.lepb200_host_lep_henc_image.argtypes = [ctypes.c_void_p, ctypes.POINTER(_HEncImage)]
    job = _HEncImage()
    assert L.lepb200_host_lep_henc_image(host_lep._h, ctypes.byref(job)) == 0
    return job


def huffman_encode(job, img):
    """lep_huffencode_kernel on the emulator: scan bytes, per-segment (status, bytes produced).  img: CoefImage with the planes."""
    assert job.scan_bytes > 0
    planes = [np.ascontiguousarray(p, dtype=np.int16) for p in img.planes]
    pp = (ctypes.c_void_p * 3)(*[p.ctypes.data for p in planes] + [None] * (3 - len(planes)))
    bch = (ctypes.c_int * 3)(*list(img.bch) + [0] * (3 - len(img.bch)))
    out = (ctypes.c_uint8 * job.scan_bytes)()
    st = (ctypes.c_int32 * 16)()
    prod = (ctypes.c_uint32 * 16)()
    L = lib()
    L.emu_huffman_encode.restype = ctypes.c_int
    rc = L.emu_huffman_encode(ctypes.byref(job), img.ncmp, img.mcuv, pp, bch, out, st, prod)
    if rc != 0:
        raise RuntimeError("emu_huffman_encode failed with %d" % rc)
    return bytes(out), [(st[k], prod[k]) for k in range(job.nseg)]
