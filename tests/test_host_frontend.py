"""Host (CPU) halves of the drop-in, no GPU needed: the JPEG front end must reproduce the reference's coefficient
planes and thread-segment splits, and the container writer must reproduce the reference's .lep bytes when fed the
reference's own segment streams (so header blob, zlib stream, handoffs, mux packets and trailer are all pinned)."""
import hashlib
import os

import numpy as np
import pytest

import lepfmt
from helpers import GOLDEN, MANIFEST, load_lep

BASELINE_COMPLETE = ["android.jpg", "androidcrop.jpg", "androidcropoptions.jpg", "androidtrail.jpg", "colorswap.jpg",
                     "grayscale.jpg", "iphonecrop2.jpg", "trailingrst.jpg", "trailingrst2.jpg"]
# truncated files (early EOF inside the scan): EEE truncation bounds, eof fix-up of the last block, 2-byte garbage tail
BASELINE_TRUNCATED = ["gray2sf.jpg", "narrowrst.jpg", "nofsync.jpg", "singlerowtrunc.jpg", "truncatedzerorun.jpg"]
# progressive (spectral selection + successive approximation, end-of-band runs, correction bits): container flag 'X'
PROGRESSIVE = ["androidprogressive.jpg", "iphoneprogressive.jpg", "iphoneprogressive2.jpg"]


@pytest.mark.parametrize("name", BASELINE_COMPLETE + BASELINE_TRUNCATED + PROGRESSIVE)
def test_jpeg_front_end_and_container_match_reference(name):
    from lepton_b200 import HostJpeg
    data = open(os.path.join(GOLDEN, name), "rb").read()
    hj = HostJpeg(data)
    assert hj.status == 0, hj.error
    img = hj.coef_image()
    m = MANIFEST[name]
    got = [hashlib.sha256(np.ascontiguousarray(p).tobytes()).hexdigest() for p in img.planes]
    assert got == m["plane_sha256"], "Huffman-decoded planes differ from the reference's -ujg dump"
    assert list(img.luma_y_start) == m["splits"]
    lf = load_lep(name[:-4] + ".lep")
    streams = lepfmt.demux(lf.payload)[:lf.nseg]
    lep = hj.write_lep(streams)
    ref = open(os.path.join(GOLDEN, name[:-4] + ".lep"), "rb").read()
    assert lep == ref, "assembled .lep differs from the reference's file"


def test_unhandled_inputs_are_refused_not_miscoded():
    """Inputs outside what the host halves cover are refused with a status, never mis-coded: here a CMYK-style
    4-component frame (reference: UNSUPPORTED_4_COLORS) and a file that is not a JPEG at all."""
    from lepton_b200 import HostJpeg
    hj = HostJpeg(b"\x89PNG\r\n\x1a\n" + b"\0" * 64)
    assert hj.status != 0 and hj.error


def test_c_abi_exports_every_declared_symbol():
    """Every function declared in include/lepton_b200.h must be exported by the built library."""
    import re
    import ctypes
    from lepton_b200 import library_path
    hdr = open(os.path.join(os.path.dirname(GOLDEN), "..", "include", "lepton_b200.h")).read()
    names = set(re.findall(r"\b(lepb200_[a-z0-9_]+)\s*\(", hdr))
    L = ctypes.CDLL(library_path())
    missing = [n for n in sorted(names) if not hasattr(L, n)]
    assert not missing, missing
    assert len(names) >= 25


def test_no_cpu_fallback_without_device():
    import torch
    from lepton_b200 import LeptonB200Codec, LeptonB200Error
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(LeptonB200Error):
        LeptonB200Codec(0)


@pytest.mark.parametrize("name", BASELINE_COMPLETE + BASELINE_TRUNCATED + ["android_t4.lep", "iphonecrop2_t8.lep", "androidcrop_t2.lep"])
def test_lep_reader_and_jpeg_recode_match_original(name):
    """Decode-side host halves without a GPU: our .lep reader must demux exactly the reference's streams, and the
    Huffman re-encoder must re-create the original JPEG byte for byte from the (oracle-decoded) coefficient planes."""
    from lepton_b200 import HostLep
    from helpers import oracle_decode_planes
    lep_name = name if name.endswith(".lep") else name[:-4] + ".lep"
    src_jpg = MANIFEST[lep_name]["source"] if lep_name in MANIFEST else name
    data = open(os.path.join(GOLDEN, lep_name), "rb").read()
    hl = HostLep(data)
    assert hl.status == 0, hl.error
    lf = load_lep(lep_name)
    img = hl.coef_image()
    assert list(img.luma_y_start) == [h.luma_y_start for h in lf.handoffs]
    assert hl.streams(img.nseg) == lepfmt.demux(lf.payload)[:lf.nseg]
    planes, _ = oracle_decode_planes(lf)
    jpg = hl.recode(planes)
    assert jpg == open(os.path.join(GOLDEN, src_jpg), "rb").read(), "re-created JPEG differs from the original"


@pytest.mark.parametrize("name", BASELINE_COMPLETE + BASELINE_TRUNCATED + PROGRESSIVE)
def test_device_reencode_layout_and_assembly(name):
    """Host half of the device Huffman re-encode path: for the files it accepts, the scan it asks the GPU for is exactly
    the byte range of the original scan, and the JPEG assembled around those bytes is the original; truncated,
    progressive and out-of-order scans are left to the host re-encoder."""
    from lepton_b200 import HostLep
    jpg = open(os.path.join(GOLDEN, name), "rb").read()
    hl = HostLep(open(os.path.join(GOLDEN, name[:-4] + ".lep"), "rb").read())
    assert hl.status == 0, hl.error
    off, n = hl.scan_layout()
    if name in BASELINE_TRUNCATED or name in PROGRESSIVE:
        assert (off, n) == (0, 0)
        return
    if n == 0:
        assert name == "colorswap.jpg"            # scan order differs from the frame's: host path
        return
    sos = jpg.rfind(b"\xff\xda", 0, off)
    assert sos >= 0 and off == sos + 2 + int.from_bytes(jpg[sos + 2:sos + 4], "big")     # right behind the SOS segment
    assert hl.assemble(jpg[off:off + n]) == jpg


@pytest.mark.timeout(60)
def test_progressive_reencode_rejects_coefficients_its_tables_cannot_express():
    """prog8x8.jpg (one 8x8 block, optimised progressive tables) has AC tables without any end-of-band code.  The real
    coefficients re-encode to the original bytes; coefficients that would need an end-of-band run must come back as an
    error, not spin in the run-length flush (EOB run handling: jpgcoder.cc encode_eobrun :5345-5377)."""
    from lepton_b200 import HostJpeg, HostLep, LeptonB200Error
    jpg = open(os.path.join(GOLDEN, "prog8x8.jpg"), "rb").read()
    hj = HostJpeg(jpg)
    assert hj.status == 0, hj.error
    planes = hj.coef_image().planes
    hl = HostLep(open(os.path.join(GOLDEN, "prog8x8.lep"), "rb").read())
    assert hl.status == 0, hl.error
    assert hl.recode(planes) == jpg
    flat = [np.full_like(np.asarray(p), i + 1) for i, p in enumerate(planes)]
    try:
        out = hl.recode(flat)
    except LeptonB200Error:
        return
    assert out != jpg


def test_legacy_container_golden_vector():
    """images/gold-legacy.lep of the reference repository (committed under tests/golden/legacy/): its test
    test_suite/test_legacy.sh expects md5 9ffbfc24d1157d0b1ed7a9b53bef4c23 after decoding.  A version-1 file from
    before the handoff table existed: segment rows come from the payload (vp8_decoder.cc:337-369) and the scan can
    only be re-created front to back.  Host halves: reader demuxes the four streams, the oracle decodes them, the
    re-encoder must produce the golden md5."""
    from lepton_b200 import HostLep
    from helpers import oracle_decode_planes
    data = open(os.path.join(GOLDEN, "legacy", "gold-legacy.lep"), "rb").read()
    hl = HostLep(data)
    assert hl.status == 0, hl.error
    lf = lepfmt.parse_container(data)
    img = hl.coef_image()
    assert img.nseg == 4 and list(img.luma_y_start) == [h.luma_y_start for h in lf.handoffs] == [0, 94, 182, 284]
    assert hl.streams(img.nseg) == lepfmt.demux(lf.payload)[:4]
    planes, _ = oracle_decode_planes(lf)
    jpg = hl.recode(planes)
    assert len(jpg) == lf.jpeg_size and hashlib.md5(jpg).hexdigest() == "9ffbfc24d1157d0b1ed7a9b53bef4c23"


def brotli_available():
    import ctypes
    from lepton_b200 import lib
    L = lib()
    L.lepb200_host_brotli_available.restype = ctypes.c_int
    return L.lepb200_host_brotli_available() == 1


def test_future_compat_golden_vector_brotli_header():
    """images/narrowrst.lep of the reference repository (committed under tests/golden/future/): container version 4, header
    blob brotli-coded, EOF marker behind the mux packets; test_suite/test_future_compat.sh expects md5
    07e9021d35114bd69f44f5bc1c3788e3 after decoding.  Host halves: the reader (system libbrotlidec for the blob) must find
    the same JPEG header, truncation bounds, handoff and segment stream as in the version-1 container the reference writes
    for narrowrst.jpg today; oracle-decoded planes through the re-encoder give the golden md5."""
    from lepton_b200 import HostLep
    from helpers import oracle_decode_planes
    if not brotli_available():
        pytest.skip("no libbrotlidec on this system: version 2 / 4 containers are refused (test below)")
    v4 = HostLep(open(os.path.join(GOLDEN, "future", "narrowrst.lep"), "rb").read())
    assert v4.status == 0, v4.error
    lf1 = load_lep("narrowrst.lep")
    v1 = HostLep(open(os.path.join(GOLDEN, "narrowrst.lep"), "rb").read())
    i4, i1 = v4.coef_image(), v1.coef_image()
    assert (i4.ncmp, list(i4.bch), list(i4.bcv), i4.mcuv, list(i4.luma_y_start)) == (i1.ncmp, list(i1.bch), list(i1.bcv), i1.mcuv, list(i1.luma_y_start))
    assert i4.qtables_zigzag == i1.qtables_zigzag
    assert v4.streams(i4.nseg) == v1.streams(i1.nseg) == lepfmt.demux(lf1.payload)[:lf1.nseg]
    planes, _ = oracle_decode_planes(lf1)
    jpg = v4.recode(planes)
    assert hashlib.md5(jpg).hexdigest() == "07e9021d35114bd69f44f5bc1c3788e3"
    assert jpg == open(os.path.join(GOLDEN, "narrowrst.jpg"), "rb").read() == v1.recode(planes)


def test_container_reader_modes_agree():
    """The batch decoder reads containers with the mux packets recorded in place (gathered into the pinned staging buffer by
    lepb200_decode_upload_gather); the host API copies the streams out.  Both modes must agree on every golden .lep (1 to 8
    segments, legacy, version 4 with its EOF marker) and on damaged files (status, and streams where there are any)."""
    import ctypes
    import glob
    import random
    from lepton_b200 import lib
    L = lib()
    L.lepb200_host_lep_lazy_equal.restype = ctypes.c_int
    L.lepb200_host_lep_lazy_equal.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
    files = sorted(glob.glob(os.path.join(GOLDEN, "*.lep")) + glob.glob(os.path.join(GOLDEN, "legacy", "*.lep")) + glob.glob(os.path.join(GOLDEN, "future", "*.lep")))
    assert len(files) >= 20
    rnd = random.Random(5)
    for f in files:
        raw = open(f, "rb").read()
        assert L.lepb200_host_lep_lazy_equal(raw, len(raw)) == 0, f
        for _ in range(6):
            bad = bytearray(raw)
            for _ in range(rnd.randrange(1, 4)):
                bad[rnd.randrange(2, len(bad))] = rnd.randrange(256)
            if rnd.random() < 0.3:
                bad = bad[:rnd.randrange(8, len(bad))]
            assert L.lepb200_host_lep_lazy_equal(bytes(bad), len(bad)) == 0, f


def test_container_versions():
    """Version 3 is the ANS coder (another codec behind the same boundary, jpgcoder.cc:1727): always refused with the 'not
    handled' status.  Versions 2 and 4 carry a brotli header blob: a zlib blob under that version byte is 'not properly brotli
    coded' (ASSERTION_FAILURE, like the reference's always_assert), or 'not handled' where libbrotlidec is missing; a damaged
    brotli blob fails the same way -- never bytes."""
    from lepton_b200 import HostLep
    data = bytearray(open(os.path.join(GOLDEN, "android.lep"), "rb").read())
    data[2] = 3
    hl = HostLep(bytes(data))
    assert hl.status == 200 and hl.error
    for v in (2, 4):
        data[2] = v
        hl = HostLep(bytes(data))
        assert hl.status == (1 if brotli_available() else 200) and hl.error, (v, hl.status)
    data[2] = 5
    assert HostLep(bytes(data)).status == 200
    if brotli_available():
        good = bytearray(open(os.path.join(GOLDEN, "future", "narrowrst.lep"), "rb").read())
        two = bytearray(good)
        two[2] = 2                                   # version 2 = the same layout (brotli header, EOF marker)
        assert HostLep(bytes(two)).status == 0
        zlen = int.from_bytes(good[24:28], "little")
        bad = bytearray(good)
        bad[28:28 + zlen] = bytes([0xFF]) * zlen     # not a brotli stream (brotli itself carries no checksum: a flipped literal may still parse)
        assert HostLep(bytes(bad)).status == 1
        cut = bytearray(good)
        cut[24:28] = (zlen // 2).to_bytes(4, "little")          # blob ends early
        assert HostLep(bytes(cut)).status != 0


def test_cli_without_a_device_fails_loudly(tmp_path):
    """The CLI (single-file and batch mode) has no CPU coder to fall back to."""
    import subprocess
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    exe = os.path.join(os.path.dirname(GOLDEN), "..", "lepton_b200", "bin", "lepton-b200")
    assert os.path.exists(exe), "build() did not produce the CLI"
    src = os.path.join(GOLDEN, "androidcrop.jpg")
    for args in ([src, str(tmp_path / "o.lep")], ["-outdir=" + str(tmp_path), src]):
        r = subprocess.run([exe] + args, capture_output=True)
        assert r.returncode == 33 and b"no CPU coder" in r.stderr
        assert not (tmp_path / "o.lep").exists() and not (tmp_path / "androidcrop.lep").exists()
    assert subprocess.run([exe], capture_output=True).returncode == 1            # usage
    assert subprocess.run([exe, "-socket", src], capture_output=True).returncode == 13


@pytest.mark.parametrize("lep_name,min_threads", [("android_t4.lep", 4), ("androidcrop_t2.lep", 2), ("iphonecrop2_t8.lep", 8)])
def test_minencodethreads_reproduces_reference_containers(lep_name, min_threads):
    """-minencodethreads=N (src/lepton/jpgcoder.cc:1086-1089, :3862-3874): the thread-segment selection with a lower bound
    must give the splits -- and, fed the reference's streams, the container bytes -- of the files the reference wrote
    with that flag."""
    from lepton_b200 import HostJpeg
    src = MANIFEST[lep_name]["source"]
    hj = HostJpeg(open(os.path.join(GOLDEN, src), "rb").read(), min_threads=min_threads)
    assert hj.status == 0, hj.error
    lf = load_lep(lep_name)
    assert list(hj.coef_image().luma_y_start) == [h.luma_y_start for h in lf.handoffs]
    assert lf.nseg >= min(min_threads, 2)
    ref = open(os.path.join(GOLDEN, lep_name), "rb").read()
    assert hj.write_lep(lepfmt.demux(lf.payload)[:lf.nseg]) == ref


@pytest.mark.parametrize("flags", [["-maxencodethreads=1"], ["-maxencodethreads=2"], ["-maxencodethreads=3", "-minencodethreads=3"],
                                   ["-minencodethreads=8"], ["-minencodethreads=5", "-maxencodethreads=6"],
                                   ["-evensplit"], ["-evensplit", "-minencodethreads=8"]])
def test_encode_thread_flags_against_live_reference(flags):
    """Splits chosen under -minencodethreads / -maxencodethreads / -evensplit == the unmodified reference CLI's, on files of
    three sizes (the largest a 24 MP tests/helpers.synth_jpeg one); the container around the oracle's streams for those
    splits == the reference's file (md5).  The reference's results: tests/golden/reference_cpu.json."""
    import hashlib
    import json
    from helpers import oracle_encode_image, synth_jpeg
    from lepton_b200 import HostJpeg
    ref = json.load(open(os.path.join(GOLDEN, "reference_cpu.json")))["thread_flags"][" ".join(flags)]
    lo = max([int(f.split("=")[1]) for f in flags if f.startswith("-min")] + [1])
    hi = min([int(f.split("=")[1]) for f in flags if f.startswith("-max")] + [8])
    assert sorted(ref) == ["androidcrop.jpg", "iphonecrop2.jpg", "synth_6000x4000_q95_444.jpg"]
    for name, want in sorted(ref.items()):
        jpg = open(os.path.join(GOLDEN, want["fixture"]), "rb").read() if "fixture" in want else synth_jpeg(**want["synth"])
        hj = HostJpeg(jpg, min_threads=lo, max_threads=hi, even_split="-evensplit" in flags)
        assert hj.status == 0, hj.error
        img = hj.coef_image()
        assert list(img.luma_y_start) == want["luma_y_start"], (name, flags)
        enc = oracle_encode_image(img)
        assert [rc for rc, _, _ in enc] == [0] * len(enc), (name, flags)
        assert hashlib.md5(hj.write_lep([s for _, s, _ in enc])).hexdigest() == want["lep_md5"], (name, flags)


def test_roundtripfail_fixture_host_halves():
    """images/roundtripfail.jpg of the reference repository (tests/golden/legacy/): the reference codes it only under
    -skipverify (exit code 41, ROUNDTRIP_FAILURE, otherwise) because the .lep does not decode back to the input.  The
    host halves reproduce both facts: the container equals the reference's -skipverify output, and re-creating the JPEG
    from the decoded planes gives a file of the same length that differs from the input -- what lepb200_codec_set_verify
    catches on the GPU path."""
    from lepton_b200 import HostJpeg, HostLep
    from helpers import oracle_decode_planes
    d = open(os.path.join(GOLDEN, "legacy", "roundtripfail.jpg"), "rb").read()
    ref = open(os.path.join(GOLDEN, "legacy", "roundtripfail_skipverify.lep"), "rb").read()
    hj = HostJpeg(d)
    assert hj.status == 0, hj.error
    lf = lepfmt.parse_container(ref)
    assert hj.write_lep(lepfmt.demux(lf.payload)[:lf.nseg]) == ref
    hl = HostLep(ref)
    assert hl.status == 0, hl.error
    planes, _ = oracle_decode_planes(lf)
    back = hl.recode(planes)
    assert len(back) == len(d) and back != d
