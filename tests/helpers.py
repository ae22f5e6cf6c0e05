"""Shared helpers for the parity tests (test infrastructure; may use oracle/)."""
import hashlib
import json
import os

import numpy as np

import lepfmt
import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
MANIFEST = json.load(open(os.path.join(GOLDEN, "manifest.json")))


def golden_leps():
    """All committed reference-written .lep files (baseline and progressive)."""
    return sorted(f for f in os.listdir(GOLDEN) if f.endswith(".lep"))


def load_lep(name):
    return lepfmt.parse_container(open(os.path.join(GOLDEN, name), "rb").read())


def geometry_of(lf):
    f = lf.frame
    tbcv, tbc = lepfmt.truncation(lf)
    q = [f.qtables[f.qidx[c]] for c in range(f.ncmp)]
    return oracle.make_geometry(f.ncmp, f.bch, f.bcv, f.mcuv, q, tbcv, tbc), tbcv, tbc


def segments_of(lf):
    hs = lf.handoffs
    return [(h.luma_y_start, h.luma_y_end, i == len(hs) - 1) for i, h in enumerate(hs)]


def oracle_decode_planes(lf):
    """Coefficient planes of a .lep, decoded by the ORACLE from the reference-written streams."""
    f = lf.frame
    g, _, _ = geometry_of(lf)
    streams = lepfmt.demux(lf.payload, lf.version)
    planes = [np.zeros((f.bch[c] * f.bcv[c], 64), dtype=np.int16) for c in range(f.ncmp)]
    for i, (y0, y1, last) in enumerate(segments_of(lf)):
        rc, _ = oracle.decode_segment(g, planes, y0, y1, last, streams[i])
        assert rc == 0, (i, rc)
    return planes, streams


def plane_hashes(planes):
    return [hashlib.sha256(np.ascontiguousarray(p).tobytes()).hexdigest() for p in planes]


def coef_image_from_lep(lf, planes):
    """lepton_b200.CoefImage carrying the same geometry / splits as a parsed reference .lep."""
    from lepton_b200 import CoefImage
    f = lf.frame
    tbcv, tbc = lepfmt.truncation(lf)
    q = [f.qtables[f.qidx[c]] for c in range(f.ncmp)]
    return CoefImage(ncmp=f.ncmp, mcuv=f.mcuv, bch=f.bch[:f.ncmp], bcv=f.bcv[:f.ncmp], qtables_zigzag=q,
                     planes=[np.ascontiguousarray(p) for p in planes],
                     luma_y_start=[h.luma_y_start for h in lf.handoffs], trunc_bcv=tbcv, trunc_bc=tbc,
                     jpeg_bytes=lf.jpeg_size)


def random_coef_image(rng, ncmp=3, mcuh=5, mcuv=4, sf=((2, 2), (1, 1), (1, 1)), density=0.25, amp=60, nseg=1,
                      qscale=1):
    """Synthetic coefficient planes with JPEG-like statistics (sparse, decaying with frequency)."""
    from lepton_b200 import CoefImage
    bch = [mcuh * sf[c][0] for c in range(ncmp)]
    bcv = [mcuv * sf[c][1] for c in range(ncmp)]
    planes = []
    for c in range(ncmp):
        n = bch[c] * bcv[c]
        mag = rng.geometric(0.15, size=(n, 64)).astype(np.int32) * amp // 8
        decay = np.ones(64)
        decay[:49] = np.linspace(1.0, 0.05, 49)       # aligned order == zig-zag order for the 7x7 part
        keep = rng.random((n, 64)) < (density * decay + 0.02)
        sign = rng.integers(0, 2, size=(n, 64)) * 2 - 1
        p = (mag * keep * sign).astype(np.int16)
        p[:, 49] = np.clip(np.cumsum(rng.integers(-20, 21, size=n)), -1000, 1000).astype(np.int16)  # smooth DC
        p = np.clip(p, -2047, 2047).astype(np.int16)
        planes.append(np.ascontiguousarray(p))
    q = [[max(1, min(255, int((3 + i // 4) * qscale))) for i in range(64)] for _ in range(ncmp)]
    v0 = bcv[0] // mcuv
    starts = sorted({(k * mcuv // nseg) * v0 for k in range(nseg)})
    return CoefImage(ncmp=ncmp, mcuv=mcuv, bch=bch, bcv=bcv, qtables_zigzag=q, planes=planes, luma_y_start=starts)


def oracle_encode_image(img):
    """Oracle streams + decision counts for a CoefImage -> list of (rc, bytes, ndecisions) per segment."""
    g = oracle.make_geometry(img.ncmp, list(img.bch), list(img.bcv), img.mcuv, img.qtables_zigzag,
                             list(img.trunc_bcv) if img.trunc_bcv is not None else None,
                             list(img.trunc_bc) if img.trunc_bc is not None else None)
    out = []
    starts = list(img.luma_y_start)
    for i, y0 in enumerate(starts):
        last = i == len(starts) - 1
        y1 = img.bcv[0] if last else starts[i + 1]
        out.append(oracle.encode_segment(g, img.planes, y0, y1, last))
    return out


def synth_jpeg(w, h, quality, subsampling, progressive=False, seed=0):
    """A photo-sized JPEG generated on the spot (stands in for test images too large to keep in the repository).  The
    pixels come from integer arithmetic only, so they are the same on every machine; Pillow's libjpeg writes the file."""
    import io
    from PIL import Image, ImageFile
    ImageFile.MAXBLOCK = 1 << 26
    rng = np.random.default_rng(seed)
    img = np.full((h, w, 3), 96, np.int32)
    for scale, amp in ((256, 96), (64, 48), (16, 24), (4, 12), (1, 6)):
        n = rng.integers(0, amp, (h // scale + 1, w // scale + 1, 3), dtype=np.int32)
        img += np.repeat(np.repeat(n, scale, 0), scale, 1)[:h, :w]
    b = io.BytesIO()
    Image.fromarray(np.clip(img - 93, 0, 255).astype(np.uint8), "RGB").save(
        b, "JPEG", quality=quality, subsampling=subsampling, progressive=progressive, optimize=False)
    return b.getvalue()


def mixed_corpus_jpegs():
    """36 small JPEGs of mixed size (incl. odd sizes), chroma subsampling, quality, with and without restart markers, some
    progressive, some grey (BASELINE config 3 in miniature)."""
    import io
    from PIL import Image, ImageFile
    ImageFile.MAXBLOCK = 1 << 24
    rng = np.random.default_rng(20240917)
    jpegs = []
    for k in range(36):
        w, h = int(rng.integers(9, 700)), int(rng.integers(9, 500))
        y, x = np.mgrid[0:h, 0:w]
        base = (128 + 70 * np.sin(x / (5.0 + k)) + 50 * np.cos(y / (3.0 + 0.5 * k)))[..., None] + rng.normal(0, 6 + 3 * (k % 7), (h, w, 3))
        im = Image.fromarray(np.clip(base, 0, 255).astype(np.uint8))
        kw = dict(quality=[60, 75, 85, 95, 100][k % 5])
        if k % 9 == 8:
            im = im.convert("L")
        else:
            kw["subsampling"] = k % 3
        if k % 4 == 3:
            kw["restart_marker_blocks"] = 1 + k % 5
        if k % 6 == 5:
            kw["progressive"] = True
        if k % 10 == 7:
            kw["optimize"] = True
        b = io.BytesIO()
        im.save(b, "JPEG", **kw)
        jpegs.append(b.getvalue())
    return jpegs
