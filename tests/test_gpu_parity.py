"""GPU parity: the sm_100a kernels, called through the C ABI, against the pinned oracle and the reference's own
.lep files.  Bit-exact (integer / byte work): streams must be identical, decoded planes identical."""
import os

import numpy as np
import pytest

import lepfmt
from helpers import (GOLDEN, MANIFEST, coef_image_from_lep, golden_leps, load_lep, oracle_decode_planes, oracle_encode_image,
                     random_coef_image)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def codec():
    from lepton_b200 import LeptonB200Codec
    c = LeptonB200Codec(0)
    yield c
    c.close()


def test_golden_batch_encode_matches_reference_streams(codec):
    """All committed reference-written .lep files in ONE batch: GPU streams == the reference's streams."""
    imgs, want = [], []
    for name in golden_leps():
        lf = load_lep(name)
        planes, streams = oracle_decode_planes(lf)
        imgs.append(coef_image_from_lep(lf, planes))
        want.append(streams[:lf.nseg])
    got = codec.encode_images(imgs)
    for name, g, w in zip(golden_leps(), got, want):
        for i, (seg, ref) in enumerate(zip(g, w)):
            assert seg.status == 0, (name, i, seg.status)
            assert seg.data == ref, "%s segment %d differs from the reference stream" % (name, i)


def test_golden_batch_decode_matches_reference_planes(codec):
    imgs, streams_all, want = [], [], []
    for name in golden_leps():
        lf = load_lep(name)
        planes, streams = oracle_decode_planes(lf)
        img = coef_image_from_lep(lf, [np.full_like(p, 77) for p in planes])
        imgs.append(img)
        streams_all.append(streams[:lf.nseg])
        want.append((lf, planes))
    st = codec.decode_images(imgs, streams_all)
    assert all(s == 0 for s in st), st
    for name, img, (lf, planes) in zip(golden_leps(), imgs, want):
        for c in range(img.ncmp):
            assert np.array_equal(img.planes[c], planes[c]), "%s component %d" % (name, c)


@pytest.mark.parametrize("lanes", ["4", "8", "32"])
def test_golden_batch_decode_group_kernel(monkeypatch, lanes):
    """lep_decode_g2_kernel<G> (the decode kernel of large batches; forced here with LEPB200_DEC_MODE=2): G lanes per
    thread-segment, 32 / G segments per warp in lock step; every group size the library ships must give the reference
    planes.  LEPB200_DEC_THREADS=32 forces several launches / a shared queue."""
    from lepton_b200 import LeptonB200Codec
    monkeypatch.setenv("LEPB200_DEC_MODE", "2")
    monkeypatch.setenv("LEPB200_DEC_LANES", lanes)
    if lanes == "4":
        monkeypatch.setenv("LEPB200_DEC_THREADS", "32")
    c = LeptonB200Codec(0)
    try:
        test_golden_batch_decode_matches_reference_planes(c)
    finally:
        c.close()


def test_random_planes_through_both_decode_kernels(monkeypatch):
    """The same coded batch through the warp-per-segment kernel (LEPB200_DEC_MODE=1) and the group kernel (mode 2): both
    must return the planes that were encoded."""
    from lepton_b200 import CoefImage, LeptonB200Codec
    rng = np.random.default_rng(4242)
    imgs = [random_coef_image(rng, ncmp=3, mcuh=3 + k % 5, mcuv=3 + k % 4, sf=((2, 2), (1, 1), (1, 1)) if k % 2 else ((1, 1), (1, 1), (1, 1)), nseg=1 + k % 4)
            for k in range(40)]
    for mode in ("1", "2"):
        monkeypatch.setenv("LEPB200_DEC_MODE", mode)
        c = LeptonB200Codec(0)
        try:
            got = c.encode_images(imgs)
            outs = [CoefImage(ncmp=im.ncmp, mcuv=im.mcuv, bch=im.bch, bcv=im.bcv, qtables_zigzag=im.qtables_zigzag,
                              planes=[np.full_like(p, 3) for p in im.planes], luma_y_start=im.luma_y_start) for im in imgs]
            st = c.decode_images(outs, [[g.data for g in r] for r in got])
            assert all(s == 0 for s in st), (mode, st)
            for im, o in zip(imgs, outs):
                for a, b in zip(im.planes, o.planes):
                    assert np.array_equal(a, b), mode
        finally:
            c.close()


@pytest.mark.parametrize("cfg", [
    dict(ncmp=3, mcuh=5, mcuv=4, sf=((2, 2), (1, 1), (1, 1)), nseg=1),
    dict(ncmp=3, mcuh=7, mcuv=6, sf=((2, 2), (1, 1), (1, 1)), nseg=3),
    dict(ncmp=3, mcuh=9, mcuv=5, sf=((1, 1), (1, 1), (1, 1)), nseg=2),
    dict(ncmp=3, mcuh=6, mcuv=4, sf=((2, 1), (1, 1), (1, 1)), nseg=2),
    dict(ncmp=1, mcuh=11, mcuv=7, sf=((1, 1),), nseg=4),
    dict(ncmp=1, mcuh=1, mcuv=1, sf=((1, 1),), nseg=1),        # single block
    dict(ncmp=1, mcuh=1, mcuv=9, sf=((1, 1),), nseg=2),        # one block wide (width_one model)
    dict(ncmp=3, mcuh=1, mcuv=3, sf=((2, 2), (1, 1), (1, 1)), nseg=1),
    dict(ncmp=3, mcuh=12, mcuv=8, sf=((2, 2), (1, 1), (1, 1)), nseg=8, density=0.9, amp=100, qscale=0.3),   # dense, large coefficients
    dict(ncmp=3, mcuh=8, mcuv=8, sf=((2, 2), (1, 1), (1, 1)), nseg=1, density=0.0, amp=1),     # (almost) empty blocks
])
def test_random_planes_encode_decode_vs_oracle(codec, cfg):
    rng = np.random.default_rng(1234)
    img = random_coef_image(rng, **cfg)
    ref = oracle_encode_image(img)
    got = codec.encode_images([img])[0]
    assert len(got) == len(ref)
    for i, (g, (rc, s, nd)) in enumerate(zip(got, ref)):
        assert g.status == rc == 0
        assert g.data == s, "segment %d" % i
        assert g.ndecisions == nd
    # decode what we encoded
    from lepton_b200 import CoefImage
    out = CoefImage(ncmp=img.ncmp, mcuv=img.mcuv, bch=img.bch, bcv=img.bcv, qtables_zigzag=img.qtables_zigzag,
                    planes=[np.full_like(p, -5) for p in img.planes], luma_y_start=img.luma_y_start)
    st = codec.decode_images([out], [[g.data for g in got]])
    assert all(s == 0 for s in st)
    for c in range(img.ncmp):
        assert np.array_equal(out.planes[c], img.planes[c])


def test_out_of_range_coefficient_status(codec):
    """COEFFICIENT_OUT_OF_RANGE (reference exit code 6, src/vp8/encoder/encoder.cc:124,265,343)."""
    rng = np.random.default_rng(5)
    img = random_coef_image(rng, ncmp=1, mcuh=4, mcuv=4, sf=((1, 1),), nseg=2)
    img.planes[0][3, 7] = 4096          # 13-bit magnitude in the first segment only
    ref = oracle_encode_image(img)
    got = codec.encode_images([img])[0]
    assert [g.status for g in got] == [r[0] for r in ref] == [6, 0]
    assert got[1].data == ref[1][1]


def test_branch_saturation_long_run(codec):
    """Long constant runs drive branch counts through the 255 overflow / 'neverseen' paths (branch.hh:82-100)."""
    from lepton_b200 import CoefImage
    n = 40 * 40
    p = np.zeros((n, 64), dtype=np.int16)
    p[:, 0] = 1
    p[::7, 1] = -3
    p[:, 49] = 5
    img = CoefImage(ncmp=1, mcuv=40, bch=[40], bcv=[40], qtables_zigzag=[[8] * 64], planes=[p], luma_y_start=[0])
    (rc, s, nd), = oracle_encode_image(img)
    got = codec.encode_images([img])[0][0]
    assert rc == 0 and got.status == 0 and got.data == s and got.ndecisions == nd
    out = CoefImage(ncmp=1, mcuv=40, bch=[40], bcv=[40], qtables_zigzag=[[8] * 64], planes=[np.zeros_like(p)], luma_y_start=[0])
    assert codec.decode_images([out], [[got.data]]) == [0]
    assert np.array_equal(out.planes[0], p)


def test_mixed_batch_many_images(codec):
    """A batch of different geometries in one launch: per-image results must not depend on batching."""
    rng = np.random.default_rng(99)
    imgs = []
    for k in range(24):
        ncmp = 1 if k % 5 == 0 else 3
        sf = ((1, 1),) if ncmp == 1 else (((2, 2), (1, 1), (1, 1)) if k % 2 else ((1, 1), (1, 1), (1, 1)))
        imgs.append(random_coef_image(rng, ncmp=ncmp, mcuh=2 + k % 7, mcuv=2 + (k * 3) % 5, sf=sf, nseg=1 + k % 3))
    got = codec.encode_images(imgs)
    for img, g in zip(imgs, got):
        ref = oracle_encode_image(img)
        assert [x.data for x in g] == [r[1] for r in ref]


@pytest.mark.parametrize("device_mux", ["1", "0"])
def test_file_level_compress_matches_reference_lep_bytes(device_mux, monkeypatch):
    """JPEG bytes -> .lep bytes through the file-level C ABI (host front end + CUDA coder + container) must equal
    the file the unmodified reference CLI wrote for the same JPEG -- with the container assembled on the device
    (lep_gather_kernel, the default) and by the host MuxWriter (LEPB200_DEVICE_MUX=0)."""
    import os
    monkeypatch.setenv("LEPB200_DEVICE_MUX", device_mux)
    from helpers import GOLDEN
    from lepton_b200 import LeptonB200FileCodec
    names = ["android.jpg", "androidcrop.jpg", "androidcropoptions.jpg", "androidtrail.jpg", "colorswap.jpg",
             "grayscale.jpg", "iphonecrop2.jpg", "trailingrst.jpg", "trailingrst2.jpg",
             "androidprogressive.jpg", "iphoneprogressive.jpg", "iphoneprogressive2.jpg"]     # incl. progressive (flag 'X')
    jpegs = [open(os.path.join(GOLDEN, n), "rb").read() for n in names]
    fc = LeptonB200FileCodec(0, host_threads=4)
    res = fc.compress(jpegs)
    for n, (st, lep) in zip(names, res):
        assert st == 0, (n, st)
        assert lep == open(os.path.join(GOLDEN, n[:-4] + ".lep"), "rb").read(), n
    fc.close()


def test_file_level_roundtrip_jpeg_lep_jpeg():
    """jpg -> lep -> jpg through the file-level C ABI: .lep equals the reference's, JPEG equals the input; and
    reference-written multi-segment .lep files decode to the original JPEG."""
    import os
    from helpers import GOLDEN, MANIFEST
    from lepton_b200 import LeptonB200FileCodec
    names = ["android.jpg", "androidcrop.jpg", "androidcropoptions.jpg", "androidtrail.jpg", "colorswap.jpg",
             "grayscale.jpg", "iphonecrop2.jpg", "trailingrst.jpg", "trailingrst2.jpg",
             "gray2sf.jpg", "narrowrst.jpg", "nofsync.jpg", "singlerowtrunc.jpg", "truncatedzerorun.jpg",     # truncated files
             "androidprogressive.jpg", "iphoneprogressive.jpg", "iphoneprogressive2.jpg"]                        # progressive
    jpegs = [open(os.path.join(GOLDEN, n), "rb").read() for n in names]
    fc = LeptonB200FileCodec(0, host_threads=4, chunk_images=4)
    leps = fc.compress(jpegs)
    assert all(st == 0 for st, _ in leps)
    for n, (_, lep) in zip(names, leps):
        assert lep == open(os.path.join(GOLDEN, n[:-4] + ".lep"), "rb").read(), n
    back = fc.decompress([l for _, l in leps])
    for n, j, (st, out) in zip(names, jpegs, back):
        assert st == 0 and out == j, n
    # most complete baseline files (restart markers / grey / 4:2:0 included) are re-encoded on the device; truncated and
    # progressive ones, and scans whose component order differs from the frame's, by the host
    assert 6 <= fc.last_gpu_recoded <= 9, fc.last_gpu_recoded
    ref = ["android_t4.lep", "iphonecrop2_t8.lep", "androidcrop_t2.lep"]
    back = fc.decompress([open(os.path.join(GOLDEN, n), "rb").read() for n in ref])
    for n, (st, out) in zip(ref, back):
        assert st == 0 and out == open(os.path.join(GOLDEN, MANIFEST[n]["source"]), "rb").read(), n
    fc.close()


@pytest.mark.timeout(600, method="thread")        # added without a GPU at hand: a hang must cost this test, not the box
@pytest.mark.parametrize("parts", ["", "1", "7"])
def test_decompress_large_batch_device_reencode_in_parts(parts, monkeypatch):
    """A batch large enough (>= 256 files) for the device Huffman encode to run in several launches whose D2H copies and
    JPEG assembly overlap the next launch (lepb200_huffman_encode_resident_parts): device-re-encoded files, files the host
    re-encodes (truncated / progressive) and a damaged .lep in ONE call; 1 part and an odd number of parts give the same bytes."""
    import os
    from helpers import GOLDEN
    from lepton_b200 import LeptonB200FileCodec
    if parts:
        monkeypatch.setenv("LEPB200_HENC_PARTS", parts)
    names = ["android.jpg", "androidcrop.jpg", "grayscale.jpg", "iphonecrop2.jpg", "trailingrst.jpg", "colorswap.jpg",
             "gray2sf.jpg", "iphoneprogressive.jpg", "androidtrail.jpg", "narrowrst.jpg"]
    jpegs = [open(os.path.join(GOLDEN, n), "rb").read() for n in names]
    leps = [open(os.path.join(GOLDEN, n[:-4] + ".lep"), "rb").read() for n in names]
    order = [(7 * k + k // 10) % len(names) for k in range(300)]
    batch = [leps[i] for i in order]
    bad = bytearray(leps[0])
    for q in range(len(bad) // 2, len(bad) // 2 + 40):
        bad[q] ^= 0x5a
    batch[123] = bytes(bad)
    fc = LeptonB200FileCodec(0, host_threads=8)
    back = fc.decompress(batch)
    n_dev = fc.last_gpu_recoded
    fc.close()
    for k, (i, (st, out)) in enumerate(zip(order, back)):
        if k == 123:
            assert st != 0 or out != jpegs[i]
            continue
        assert st == 0 and out == jpegs[i], (k, names[i], st)
    assert n_dev >= 150, n_dev


@pytest.mark.parametrize("gpu_huffman", [True, False])
def test_file_level_compress_both_huffman_paths(gpu_huffman):
    """Huffman decode on the GPU (one thread per image) and on host threads must give the same, reference-identical
    .lep files (restart markers, grey, 4:2:0 and multi-segment images included)."""
    import os
    from helpers import GOLDEN
    from lepton_b200 import LeptonB200FileCodec
    names = ["android.jpg", "androidcrop.jpg", "androidcropoptions.jpg", "androidtrail.jpg", "colorswap.jpg",
             "grayscale.jpg", "iphonecrop2.jpg", "trailingrst.jpg", "trailingrst2.jpg"]
    jpegs = [open(os.path.join(GOLDEN, n), "rb").read() for n in names] * 3
    fc = LeptonB200FileCodec(0, host_threads=4, chunk_images=8, gpu_huffman=gpu_huffman)
    res = fc.compress(jpegs)
    for k, (st, lep) in enumerate(res):
        n = names[k % len(names)]
        assert st == 0, (n, st)
        assert lep == open(os.path.join(GOLDEN, n[:-4] + ".lep"), "rb").read(), n
    fc.close()


@pytest.mark.parametrize("par,bits", [("0", "4096"), ("1", "4096"), ("1", "512")])
def test_huffman_decode_kernels_serial_and_subsequence(par, bits, monkeypatch):
    """lep_huffdecode_kernel alone (LEPB200_HUFF_PAR=0) and the sub-sequence kernels of lep_huffpar.cu in front of it must
    both lead to the reference's .lep bytes; synthetic 4:2:0 / 4:4:4 files large enough for hundreds of sub-sequences
    are checked against each other and by a round trip."""
    import io
    import os
    import numpy as np
    from PIL import Image
    from helpers import GOLDEN
    from lepton_b200 import LeptonB200FileCodec
    monkeypatch.setenv("LEPB200_HUFF_PAR", par)
    monkeypatch.setenv("LEPB200_HUFF_SUBSEQ_BITS", bits)
    names = ["android.jpg", "androidcrop.jpg", "androidcropoptions.jpg", "androidtrail.jpg", "grayscale.jpg", "iphonecrop2.jpg", "trailingrst.jpg"]
    jpegs = [open(os.path.join(GOLDEN, n), "rb").read() for n in names]
    rng = np.random.default_rng(11)
    for k, (w, h, q, sub) in enumerate([(1920, 1080, 85, 2), (801, 603, 95, 0), (2048, 64, 70, 1), (1280, 720, 85, 2)]):
        yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
        img = np.stack([128 + 70 * np.sin(xx / (9.0 + c) + yy / (17.0 - c) + k) for c in range(3)], -1) + rng.normal(0, 16, (h, w, 3))
        b = io.BytesIO()
        Image.fromarray(np.clip(img, 0, 255).astype(np.uint8), "RGB").save(b, "JPEG", quality=q, subsampling=sub)
        jpegs.append(b.getvalue())
    fc = LeptonB200FileCodec(0, host_threads=4)
    res = fc.compress(jpegs)
    host = LeptonB200FileCodec(0, host_threads=4, gpu_huffman=False)
    want = host.compress(jpegs)
    host.close()
    for k, ((st, lep), (st2, lep2)) in enumerate(zip(res, want)):
        assert st == 0 and st2 == 0, k
        assert lep == lep2, "file %d: GPU Huffman decode and host Huffman decode lead to different .lep bytes" % k
        if k < len(names):
            assert lep == open(os.path.join(GOLDEN, names[k][:-4] + ".lep"), "rb").read(), names[k]
    back = fc.decompress([lep for _, lep in res])
    fc.close()
    for k, (j, (st, out)) in enumerate(zip(jpegs, back)):
        assert st == 0 and out == j, k


def test_cli_jpg_to_lep_and_back(tmp_path):
    """`lepton-b200 in.jpg out.lep` writes the reference CLI's bytes; `lepton-b200 out.lep back.jpg` restores the input
    (the north_star's `lepton` command-line surface, src/lepton/jpgcoder.cc:988-1219,1528)."""
    import os
    import subprocess
    from helpers import GOLDEN
    exe = os.path.join(os.path.dirname(GOLDEN), "..", "lepton_b200", "bin", "lepton-b200")
    assert os.path.exists(exe), "build() did not produce the CLI"
    for name in ("androidcrop.jpg", "iphoneprogressive.jpg", "gray2sf.jpg"):
        src = os.path.join(GOLDEN, name)
        lep, back = str(tmp_path / "o.lep"), str(tmp_path / "o.jpg")
        r = subprocess.run([exe, "-skipverify", src, lep], capture_output=True)
        assert r.returncode == 0, r.stderr
        assert open(lep, "rb").read() == open(os.path.join(GOLDEN, name[:-4] + ".lep"), "rb").read(), name
        r = subprocess.run([exe, lep, back], capture_output=True)
        assert r.returncode == 0, r.stderr
        assert open(back, "rb").read() == open(src, "rb").read(), name
    r = subprocess.run([exe, "-socket", os.path.join(GOLDEN, "androidcrop.jpg")], capture_output=True)
    assert r.returncode == 13                     # service modes are outside this build: refused, not ignored


def test_mixed_corpus_matches_reference_cli_and_round_trips():
    """BASELINE config 3 in miniature: JPEGs of mixed size (incl. odd sizes), chroma subsampling, quality, with and without
    restart markers, some progressive, some grey -- one batch through the file API.  Every .lep must equal what the
    unmodified reference CLI writes (md5s in tests/golden/mixed_corpus.json, by tests/golden/make_refimages.py), and
    decompress must restore every input."""
    import hashlib
    import json
    from helpers import GOLDEN, mixed_corpus_jpegs
    from lepton_b200 import LeptonB200FileCodec
    jpegs = mixed_corpus_jpegs()
    ref = json.load(open(os.path.join(GOLDEN, "mixed_corpus.json")))
    assert [hashlib.md5(j).hexdigest() for j in jpegs] == ref["jpg_md5"], "not the JPEGs the reference was given"
    fc = LeptonB200FileCodec(0, host_threads=4)
    leps = fc.compress(jpegs)
    assert all(st == 0 for st, _ in leps), [st for st, _ in leps]
    for k, (_, lep) in enumerate(leps):
        assert hashlib.md5(lep).hexdigest() == ref["lep_md5"][k], "file %d: .lep differs from the reference CLI's" % k
    back = fc.decompress([l for _, l in leps])
    for k, (j, (st, out)) in enumerate(zip(jpegs, back)):
        assert st == 0 and out == j, k
    assert fc.last_gpu_recoded >= 20          # the complete baseline files took the device Huffman encoder
    fc.close()


def test_corrupt_files_fail_alone_inside_a_batch():
    """Damaged inputs (scan bytes of a JPEG, coded payload / header bytes of a .lep) travel in one batch with intact files:
    the kernels must stay inside their buffers, every damaged file ends with either a status or some output, and the
    intact files of the batch still come out byte-exact."""
    import os
    import random
    from helpers import GOLDEN
    from lepton_b200 import LeptonB200FileCodec
    rnd = random.Random(99)
    good = ["android.jpg", "grayscale.jpg", "trailingrst.jpg", "iphonecrop2.jpg"]
    good_jpg = [open(os.path.join(GOLDEN, n), "rb").read() for n in good]
    good_lep = [open(os.path.join(GOLDEN, n[:-4] + ".lep"), "rb").read() for n in good]
    bad_jpg, bad_lep = [], []
    for k in range(24):
        j = bytearray(good_jpg[k % 4])
        sos = j.rfind(b"\xff\xda")
        for _ in range(1 + k % 5):
            j[rnd.randrange(sos + 14, len(j) - 2)] = rnd.randrange(256)
        bad_jpg.append(bytes(j))
        l = bytearray(good_lep[k % 4])
        lo = 28 if k % 3 == 0 else len(l) // 3                 # header blob (zlib) or the arithmetic-coded payload
        for _ in range(1 + k % 4):
            l[rnd.randrange(lo, len(l) - 4)] = rnd.randrange(256)
        bad_lep.append(bytes(l))
    fc = LeptonB200FileCodec(0, host_threads=4)
    res = fc.compress(good_jpg + bad_jpg)
    for n, (st, lep), ref in zip(good, res[:4], good_lep):
        assert st == 0 and lep == ref, n
    assert all(st != 0 or len(lep) > 0 for st, lep in res[4:])
    back = fc.decompress(good_lep + bad_lep)
    for n, (st, out), ref in zip(good, back[:4], good_jpg):
        assert st == 0 and out == ref, n
    assert all(st != 0 or len(out) > 0 for st, out in back[4:])
    # files that still compress must also restore exactly (a damaged scan is just another JPEG to the coder)
    again = [lep for st, lep in res[4:] if st == 0]
    src = [j for j, (st, _) in zip(bad_jpg, res[4:]) if st == 0]
    if again:
        for j, (st, out) in zip(src, fc.decompress(again)):
            assert st == 0 and out == j
    fc.close()


@pytest.mark.timeout(600, method="thread")        # added without a GPU at hand: a hang must cost this test, not the box
def test_reference_legacy_golden_vector_decompress():
    """The reference repository's golden vector images/gold-legacy.lep (tests/golden/legacy/; test_suite/test_legacy.sh
    pins the md5 of its decoding): a legacy container without a handoff table, four thread-segments.  The product's
    file-level decode must produce the golden md5, and compressing the result again must round-trip."""
    import hashlib
    from lepton_b200 import LeptonB200FileCodec
    data = open(os.path.join(GOLDEN, "legacy", "gold-legacy.lep"), "rb").read()
    fc = LeptonB200FileCodec(0, host_threads=4)
    (st, jpg), = fc.decompress([data])
    assert st == 0 and hashlib.md5(jpg).hexdigest() == "9ffbfc24d1157d0b1ed7a9b53bef4c23"
    (st, lep), = fc.compress([jpg])
    assert st == 0
    (st, back), = fc.decompress([lep])
    assert st == 0 and back == jpg
    fc.close()


@pytest.mark.timeout(600, method="thread")        # added without a GPU at hand: a hang must cost this test, not the box
def test_cli_batch_mode(tmp_path):
    """`lepton-b200 -outdir=DIR inputs...`: JPEGs and .lep files in one invocation, one library call per direction;
    outputs equal the reference's files, a damaged input fails alone with its exit code."""
    import subprocess
    from helpers import GOLDEN
    exe = os.path.join(os.path.dirname(GOLDEN), "..", "lepton_b200", "bin", "lepton-b200")
    names = ["androidcrop.jpg", "grayscale.jpg", "iphoneprogressive.jpg", "trailingrst.jpg"]
    leps = ["android.lep", "gray2sf.lep", "iphonecrop2_t8.lep"]
    bad = tmp_path / "broken.lep"
    bad.write_bytes(open(os.path.join(GOLDEN, "android.lep"), "rb").read()[:40])          # cut inside the header: SHORT_READ
    out = tmp_path / "out"
    out.mkdir()
    args = [os.path.join(GOLDEN, n) for n in names + leps] + [str(bad)]
    r = subprocess.run([exe, "-skipverify", "-outdir=" + str(out)] + args, capture_output=True)
    assert r.returncode != 0 and b"broken.lep" in r.stderr, r.stderr            # the damaged file reports, the rest is written
    for n in names:
        assert (out / (n[:-4] + ".lep")).read_bytes() == open(os.path.join(GOLDEN, n[:-4] + ".lep"), "rb").read(), n
    from helpers import MANIFEST
    for n in leps:
        src = MANIFEST[n]["source"] if "source" in MANIFEST.get(n, {}) else n[:-4] + ".jpg"
        assert (out / (n[:-4] + ".jpg")).read_bytes() == open(os.path.join(GOLDEN, src), "rb").read(), n
    assert not (out / "broken.jpg").exists()


@pytest.mark.timeout(600, method="thread")        # added without a GPU at hand: a hang must cost this test, not the box
def test_rejectprogressive_exit_code():
    """-rejectprogressive (src/lepton/jpgcoder.cc:1056-1058, :2911-2925): progressive files leave with the reference's
    exit code 8 (PROGRESSIVE_UNSUPPORTED); baseline files of the same batch are coded as usual."""
    from helpers import GOLDEN
    from lepton_b200 import LeptonB200FileCodec
    names = ["androidcrop.jpg", "iphoneprogressive.jpg", "grayscale.jpg", "androidprogressive.jpg"]
    fc = LeptonB200FileCodec(0, host_threads=2, allow_progressive=False)
    res = fc.compress([open(os.path.join(GOLDEN, n), "rb").read() for n in names])
    fc.close()
    assert [st for st, _ in res] == [0, 8, 0, 8]
    for n, (st, lep) in zip(names, res):
        if st == 0:
            assert lep == open(os.path.join(GOLDEN, n[:-4] + ".lep"), "rb").read(), n


@pytest.mark.timeout(600, method="thread")        # added without a GPU at hand: a hang must cost this test, not the box
def test_minencodethreads_files_match_reference():
    """-minencodethreads=N through the file API: the .lep bytes of the reference CLI run with the same flag."""
    from helpers import GOLDEN, MANIFEST
    from lepton_b200 import LeptonB200FileCodec
    for lep_name, n in (("android_t4.lep", 4), ("androidcrop_t2.lep", 2), ("iphonecrop2_t8.lep", 8)):
        fc = LeptonB200FileCodec(0, host_threads=2, min_encode_threads=n)
        (st, lep), = fc.compress([open(os.path.join(GOLDEN, MANIFEST[lep_name]["source"]), "rb").read()])
        fc.close()
        assert st == 0 and lep == open(os.path.join(GOLDEN, lep_name), "rb").read(), lep_name


@pytest.mark.timeout(600, method="thread")        # added without a GPU at hand: a hang must cost this test, not the box
def test_multi_gpu_single_process_codec():
    """lepb200_compress_jpegs_multi / _decompress_leps_multi: one process, every visible GPU (the same GPU twice when
    there is only one -- two codecs, two pipelines, same device), files dealt by size; bytes == the reference's."""
    import torch
    from helpers import GOLDEN
    from lepton_b200 import LeptonB200MultiGpuFileCodec
    ngpu = torch.cuda.device_count()
    devices = list(range(ngpu)) if ngpu > 1 else [0, 0]
    names = ["android.jpg", "androidcrop.jpg", "grayscale.jpg", "iphonecrop2.jpg", "trailingrst.jpg", "iphoneprogressive.jpg",
             "gray2sf.jpg", "colorswap.jpg", "androidtrail.jpg"]
    jpegs = [open(os.path.join(GOLDEN, n), "rb").read() for n in names]
    mc = LeptonB200MultiGpuFileCodec(devices, host_threads_per_gpu=2)
    leps = mc.compress(jpegs)
    for n, (st, lep) in zip(names, leps):
        assert st == 0 and lep == open(os.path.join(GOLDEN, n[:-4] + ".lep"), "rb").read(), n
    back = mc.decompress([l for _, l in leps])
    for n, j, (st, out) in zip(names, jpegs, back):
        assert st == 0 and out == j, n
    mc.close()


@pytest.mark.timeout(600, method="thread")        # added without a GPU at hand: a hang must cost this test, not the box
def test_verify_mode_withholds_files_that_do_not_round_trip(tmp_path):
    """-verify (the reference CLI's default): the reference's images/roundtripfail.jpg (tests/golden/legacy/) is coded by
    the reference only with -skipverify -- its .lep decodes to a JPEG that differs from the input -- and exits with
    41 (ROUNDTRIP_FAILURE) otherwise.  Same here: with verify on the file is withheld with status 41 while the other
    files of the batch are written as usual; with verify off the bytes equal what the reference writes under -skipverify."""
    import subprocess
    from helpers import GOLDEN
    from lepton_b200 import LeptonB200FileCodec
    bad = open(os.path.join(GOLDEN, "legacy", "roundtripfail.jpg"), "rb").read()
    names = ["androidcrop.jpg", "grayscale.jpg", "iphoneprogressive.jpg", "gray2sf.jpg"]
    jpegs = [open(os.path.join(GOLDEN, n), "rb").read() for n in names]
    fc = LeptonB200FileCodec(0, host_threads=2, verify=True)
    res = fc.compress(jpegs[:2] + [bad] + jpegs[2:])
    fc.close()
    assert [st for st, _ in res] == [0, 0, 41, 0, 0] and res[2][1] == b""
    for n, (st, lep) in zip(names, res[:2] + res[3:]):
        assert lep == open(os.path.join(GOLDEN, n[:-4] + ".lep"), "rb").read(), n
    fc = LeptonB200FileCodec(0, host_threads=2)
    (st, lep), = fc.compress([bad])
    (st2, back), = fc.decompress([lep])
    fc.close()
    assert st == 0 and lep == open(os.path.join(GOLDEN, "legacy", "roundtripfail_skipverify.lep"), "rb").read()
    assert st2 == 0 and back != bad and len(back) == len(bad)
    exe = os.path.join(os.path.dirname(GOLDEN), "..", "lepton_b200", "bin", "lepton-b200")
    r = subprocess.run([exe, os.path.join(GOLDEN, "legacy", "roundtripfail.jpg"), str(tmp_path / "o.lep")], capture_output=True)
    assert r.returncode == 41 and not (tmp_path / "o.lep").exists()
    r = subprocess.run([exe, os.path.join(GOLDEN, "androidcrop.jpg"), str(tmp_path / "a.lep")], capture_output=True)
    assert r.returncode == 0 and (tmp_path / "a.lep").read_bytes() == open(os.path.join(GOLDEN, "androidcrop.lep"), "rb").read()


@pytest.mark.timeout(600, method="thread")
def test_reference_cli_with_b200_adapters(tmp_path):
    """oracle/_ref/lepton-b200plug = the reference's own CLI, built from its sources with B200ComponentEncoder /
    B200ComponentDecoder (lepton_b200/adapter/) in its two factory lines: `lepton in.jpg out.lep` must write the bytes
    the unmodified reference writes, and `lepton out.lep back.jpg` must restore the input through both decoder entries."""
    import subprocess
    from helpers import GOLDEN
    exe = os.path.join(os.path.dirname(GOLDEN), "..", "oracle", "_ref", "lepton-b200plug")
    assert os.path.exists(exe), "oracle/_ref/lepton-b200plug missing: __graft_entry__.build() makes it where /root/reference exists (it travels with the snapshot)"
    for name in ("androidcrop.jpg", "grayscale.jpg", "iphonecrop2.jpg"):
        src = os.path.join(GOLDEN, name)
        lep, back = str(tmp_path / "o.lep"), str(tmp_path / "o.jpg")
        r = subprocess.run([exe, "-unjailed", "-skipverify", src, lep], capture_output=True)
        assert r.returncode == 0, r.stderr[-2000:]
        assert open(lep, "rb").read() == open(os.path.join(GOLDEN, name[:-4] + ".lep"), "rb").read(), name
        for flags in (["-forceprogressive"], [], ["-singlethread"]):        # full-plane entry, row entry threaded / single-threaded
            r = subprocess.run([exe, "-unjailed"] + flags + [lep, back], capture_output=True)
            assert r.returncode == 0, (flags, r.stderr[-2000:])
            assert open(back, "rb").read() == open(src, "rb").read(), (name, flags)
