"""Pins the CPU oracle (oracle/lepton_oracle.c) against files written by the UNMODIFIED reference.

tests/golden/*.lep were written by oracle/_ref/lepton (the reference CLI compiled from /root/reference by
oracle/Makefile.ref); manifest.json holds sha256s of the coefficient planes from the reference's own -ujg dump.
 * oracle decode of the reference's segment streams must reproduce the reference's coefficient planes;
 * oracle encode of those planes must reproduce the reference's segment streams byte for byte.
The reference repository's own golden vector images/iphone16.lep (test_suite/test_16threads.sh) is checked where the
reference's images/ directory is present; the other checks against the reference use what it wrote, kept in
tests/golden/reference_cpu.json (tests/golden/make_refimages.py).
"""
import json
import os

import numpy as np
import pytest

import lepfmt
import oracle
from helpers import GOLDEN, MANIFEST, geometry_of, golden_leps, load_lep, oracle_decode_planes, plane_hashes, segments_of

REFERENCE = json.load(open(os.path.join(GOLDEN, "reference_cpu.json")))


@pytest.mark.parametrize("name", golden_leps())
def test_oracle_roundtrips_reference_streams(name):
    lf = load_lep(name)
    planes, streams = oracle_decode_planes(lf)
    src = MANIFEST.get(name[:-4] + ".jpg") or MANIFEST.get(MANIFEST.get(name, {}).get("source", ""), {})
    if "plane_sha256" in src:
        assert plane_hashes(planes) == src["plane_sha256"], "oracle decode != reference -ujg coefficient dump"
    g, _, _ = geometry_of(lf)
    for i, (y0, y1, last) in enumerate(segments_of(lf)):
        rc, s, nd = oracle.encode_segment(g, planes, y0, y1, last)
        assert rc == 0
        assert s == streams[i], "oracle encode != reference stream for segment %d" % i
        assert nd > 0


@pytest.mark.skipif(not os.path.isdir("/root/reference/images"), reason="reference tree only exists in the build container")
@pytest.mark.slow
def test_reference_repo_golden_vector_iphone16(tmp_path):
    """images/iphone16.lep (16 thread segments) is the reference's own golden vector: test_suite/test_16threads.sh
    expects it to decode to iphone.jpg (md5 8ea9fcf1b2c24877aa838dd6ac1df413).  The oracle must decode its 16
    streams to exactly the coefficient planes the reference dumps for iphone.jpg, and re-encode them bit-exactly."""
    import hashlib
    import subprocess
    from conftest import REF_LEPTON
    jpg = "/root/reference/images/iphone.jpg"
    assert hashlib.md5(open(jpg, "rb").read()).hexdigest() == "8ea9fcf1b2c24877aa838dd6ac1df413"
    lf = lepfmt.parse_container(open("/root/reference/images/iphone16.lep", "rb").read())
    assert lf.nseg == 16
    planes, streams = oracle_decode_planes(lf)
    ujg = str(tmp_path / "a.ujg")
    assert subprocess.run([REF_LEPTON, "-ujg", "-skipverify", jpg, ujg], capture_output=True).returncode == 0
    _, ref_planes = lepfmt.parse_ujg_planes(open(ujg, "rb").read())
    for a, b in zip(planes, ref_planes):
        assert np.array_equal(a, b)
    g, _, _ = geometry_of(lf)
    for i, (y0, y1, last) in enumerate(segments_of(lf)):
        rc, s, _ = oracle.encode_segment(g, planes, y0, y1, last)
        assert rc == 0 and s == streams[i]


def _pin_against_reference_lep(lf, ref_plane_sha256, nseg, streams=None):
    """Oracle decode of the container's streams == planes the reference dumps (-ujg) for the JPEG (their sha256s);
    oracle re-encode == streams.  ``streams``: decode these instead of lf's own (a golden container whose header blob
    this image cannot read)."""
    assert len(lf.handoffs) == nseg
    if streams is None:
        streams = lepfmt.demux(lf.payload, lf.version)
    f = lf.frame
    g, _, _ = geometry_of(lf)
    planes = [np.zeros((f.bch[c] * f.bcv[c], 64), dtype=np.int16) for c in range(f.ncmp)]
    for i, (y0, y1, last) in enumerate(segments_of(lf)):
        rc, _ = oracle.decode_segment(g, planes, y0, y1, last, streams[i])
        assert rc == 0, (i, rc)
    assert plane_hashes(planes) == ref_plane_sha256, "oracle decode != reference -ujg coefficient dump"
    for i, (y0, y1, last) in enumerate(segments_of(lf)):
        rc, s, _ = oracle.encode_segment(g, planes, y0, y1, last)
        assert rc == 0 and s == streams[i], i


@pytest.mark.slow
def test_reference_repo_golden_vector_gold_legacy():
    """images/gold-legacy.lep of the reference repository (tests/golden/legacy/; test_suite/test_legacy.sh expects md5
    9ffbfc24d1157d0b1ed7a9b53bef4c23 after decoding): a version-1 file from before the handoff table existed -- the
    payload opens with the segment count and the luma split rows (src/lepton/vp8_decoder.cc:337-369).  The planes are
    pinned to the reference's -ujg dump of the JPEG it decodes to."""
    lf = lepfmt.parse_container(open(os.path.join(GOLDEN, "legacy", "gold-legacy.lep"), "rb").read())
    _pin_against_reference_lep(lf, REFERENCE["gold_legacy_plane_sha256"], nseg=4)


def test_reference_repo_golden_vector_narrowrst():
    """images/narrowrst.lep (tests/golden/future/; test_suite/test_future_compat.sh expects md5
    07e9021d35114bd69f44f5bc1c3788e3 = the md5 of images/narrowrst.jpg): container version 4, brotli header blob (no
    brotli decoder needed here), one thread-segment, a truncated JPEG with restart markers.  The blob is skipped by its
    length field; the frame and the truncation bounds come from the version-1 container the reference writes for
    narrowrst.jpg today (tests/golden/narrowrst.lep), whose coefficient stream must be byte-identical with the golden
    file's.  The oracle then has to decode the GOLDEN stream to the reference's planes and re-create it."""
    import hashlib
    data = open(os.path.join(GOLDEN, "narrowrst.jpg"), "rb").read()
    assert hashlib.md5(data).hexdigest() == "07e9021d35114bd69f44f5bc1c3788e3"
    lf4 = lepfmt.parse_container(open(os.path.join(GOLDEN, "future", "narrowrst.lep"), "rb").read(), data)
    assert lf4.version == 4 and lf4.nseg == 1 and lf4.jpeg_size == len(data)
    golden_streams = lepfmt.demux(lf4.payload, lf4.version)
    v1 = open(os.path.join(GOLDEN, "narrowrst.lep"), "rb").read()
    assert hashlib.md5(v1).hexdigest() == MANIFEST["narrowrst.jpg"]["lep_md5"]
    lf1 = lepfmt.parse_container(v1)
    assert lf1.version == 1 and "EEE" in lf1.sections
    assert lepfmt.demux(lf1.payload, 1) == golden_streams
    _pin_against_reference_lep(lf1, MANIFEST["narrowrst.jpg"]["plane_sha256"], nseg=1, streams=golden_streams)


def test_branch_update_matches_reference_semantics():
    """Branch::record_obs_and_update corner cases (src/vp8/model/branch.hh:82-100) through a tiny stream."""
    # An all-zero 1x1-block grayscale image exercises the identity priors; encode/decode must agree.
    q = [[16] * 64]
    g = oracle.make_geometry(1, [1], [1], 1, q)
    planes = [np.zeros((1, 64), dtype=np.int16)]
    rc, s, nd = oracle.encode_segment(g, planes, 0, 1, True)
    assert rc == 0 and nd == 6 + 3 + 3 + 1
    out = [np.ones((1, 64), dtype=np.int16)]
    rc, nd2 = oracle.decode_segment(g, out, 0, 1, True, s)
    assert rc == 0 and nd2 == nd and not out[0].any()


def test_out_of_range_coefficient_is_rejected():
    """COEFFICIENT_OUT_OF_RANGE (exit code 6): src/vp8/encoder/encoder.cc:124,265,343."""
    q = [[16] * 64]
    g = oracle.make_geometry(1, [1], [1], 1, q)
    planes = [np.zeros((1, 64), dtype=np.int16)]
    planes[0][0, 3] = 4096
    rc, _, _ = oracle.encode_segment(g, planes, 0, 1, True)
    assert rc == 6


@pytest.mark.slow
def test_oracle_vs_live_reference_on_a_large_fixture():
    """A photo-sized JPEG (tests/helpers.synth_jpeg, 12 MP, 8 thread-segments): the host front end's planes == the
    reference's -ujg dump, the reference's segment starts, and oracle encode == the reference's streams (md5s)."""
    import hashlib
    from helpers import oracle_encode_image, synth_jpeg
    from lepton_b200 import HostJpeg
    ref = REFERENCE["large"]
    hj = HostJpeg(synth_jpeg(**ref["synth"]))
    assert hj.status == 0, hj.error
    img = hj.coef_image()
    assert plane_hashes(img.planes) == ref["plane_sha256"], "front end planes != reference -ujg coefficient dump"
    assert list(img.luma_y_start) == ref["luma_y_start"] and len(ref["luma_y_start"]) == 8
    enc = oracle_encode_image(img)
    assert [rc for rc, _, _ in enc] == [0] * len(enc)
    assert [hashlib.md5(s).hexdigest() for _, s, _ in enc] == ref["stream_md5"]
    assert hashlib.md5(hj.write_lep([s for _, s, _ in enc])).hexdigest() == ref["lep_md5"]
