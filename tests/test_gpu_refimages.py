"""GPU parity over the files of the reference's images/ directory (BASELINE.json: "bit-exact .jpg<->.lep round-trip on
every file in images/"; the reference's Makefile.am:238-362 are its own tests over these files).

tests/golden/refimages.json (written by tests/golden/make_refimages.py) holds what the UNMODIFIED reference CLI did with
each file: the images small enough to keep are under tests/golden/, arithmetic.jpg is kept as its first 4 KB, and the
photo-sized ones are stood in for by JPEGs of the same kinds that tests/helpers.synth_jpeg generates here.  All files go
through the CUDA path by the file-level C ABI; comparison is by md5 of whole files (bit-exact)."""
import hashlib
import json
import os

import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")


def md5(b):
    return hashlib.md5(b).hexdigest()


@pytest.fixture(scope="module")
def expected():
    return json.load(open(os.path.join(GOLDEN, "refimages.json")))


@pytest.fixture(scope="module")
def files(expected):
    """name -> the bytes the reference was given: a fixture under tests/golden/ or a generated JPEG."""
    from helpers import synth_jpeg
    out = {}
    for n, e in expected.items():
        if "fixture" in e:
            out[n] = open(os.path.join(GOLDEN, e["fixture"]), "rb").read()
        else:
            a = dict(e["synth"])
            keep = a.pop("truncate", 1.0)
            j = synth_jpeg(**a)
            out[n] = j[:int(len(j) * keep)]
        assert md5(out[n]) == e.get("jpg_md5", e.get("lep_md5")), "%s: not the input the reference was given" % n
    return out


@pytest.fixture(scope="module")
def compressed(expected, files):
    """All JPEGs (good and expected-failure ones alike) in ONE batch through lepb200_compress_jpegs."""
    from lepton_b200 import LeptonB200FileCodec
    names = sorted(n for n in expected if n.endswith(".jpg"))
    jpegs = [files[n] for n in names]
    fc = LeptonB200FileCodec(0, host_threads=8)
    res = fc.compress(jpegs)
    launches = fc.kernel_launches
    fc.close()
    assert launches > 0
    return names, jpegs, res


def test_every_reference_image_compresses_to_the_reference_lep(expected, compressed):
    names, jpegs, res = compressed
    good = 0
    for n, j, (st, lep) in zip(names, jpegs, res):
        e = expected[n]
        assert md5(j) == e["jpg_md5"], n
        assert st == e["status_want"], (n, st, e["status_want"])
        if e["status_want"] == 0:
            assert len(lep) == e["lep_size"] and md5(lep) == e["lep_md5"], "%s: .lep differs from the reference CLI's" % n
            good += 1
        else:
            assert lep == b"", n
    assert good == 22          # the photo-sized stand-ins (8 thread-segments, 4:4:4 q95, progressive, truncated) included


def test_expected_failure_exit_codes(expected, compressed):
    """Makefile.am:302-304 (arithmetic: EXPECT_FAILURE) and :357-359 (badzerorun: EXPECT_FAILURE): the reference process
    that meets the error leaves with UNSUPPORTED_JPEG (42) / ASSERTION_FAILURE (1, the assert at jpgcoder.cc:4951)."""
    names, _, res = compressed
    st = {n: s for n, (s, _) in zip(names, res)}
    assert st["arithmetic_head.jpg"] == 42
    assert st["badzerorun.jpg"] == 1
    # what the live reference CLI said in the build container.  Its process status is not a stable witness (custom_exit
    # ends ONE thread with SYS_exit, memory.cc:246-247: 42 or 0 depending on which thread leaves last), the name it
    # writes first (memory.cc:238-245) and the empty output are
    assert expected["arithmetic_head.jpg"]["exit_name"] == "UNSUPPORTED_JPEG" and "lep_md5" not in expected["arithmetic_head.jpg"]
    assert expected["badzerorun.jpg"]["rc_skipverify"] != 0 and "lep_md5" not in expected["badzerorun.jpg"]


def test_every_reference_image_round_trips(expected, compressed):
    """.lep -> .jpg through lepb200_decompress_leps (GPU arithmetic decode, GPU or host Huffman re-encode): equal to the
    input for every file the reference round-trips, equal to the REFERENCE's (different) decoding for roundtripfail.jpg."""
    from lepton_b200 import LeptonB200FileCodec
    names, jpegs, res = compressed
    ok = [(n, j, lep) for n, j, (st, lep) in zip(names, jpegs, res) if st == 0]
    fc = LeptonB200FileCodec(0, host_threads=8)
    back = fc.decompress([lep for _, _, lep in ok])
    fc.close()
    for (n, j, _), (st, out) in zip(ok, back):
        assert st == 0, (n, st)
        assert md5(out) == expected[n]["back_md5"], "%s: restored JPEG differs from the reference's decoding" % n
        if n != "roundtripfail.jpg":
            assert out == j, n


def test_roundtripfail_with_verify_is_withheld(expected, files):
    """test_suite/test_roundtrip.sh territory: with validation on (the reference CLI's default) the file exits 41."""
    from lepton_b200 import LeptonB200FileCodec
    assert expected["roundtripfail.jpg"]["rc_verify"] == 41 or expected["roundtripfail.jpg"]["exit_name_verify"] == "ROUNDTRIP_FAILURE"
    fc = LeptonB200FileCodec(0, host_threads=4, verify=True)
    names = ("iphonecrop2.jpg", "roundtripfail.jpg", "synth_3264x2448_q92_trunc.jpg")
    res = fc.compress([files[n] for n in names])
    fc.close()
    assert [st for st, _ in res] == [0, 41, 0]
    assert md5(res[0][1]) == expected[names[0]]["lep_md5"] and md5(res[2][1]) == expected[names[2]]["lep_md5"]


def test_reference_golden_lep_vectors_decode_to_the_pinned_md5(expected, files):
    """The reference repository's own golden vectors: gold-legacy.lep (test_suite/test_legacy.sh) must decode to the md5
    that script pins; so must narrowrst.lep
    (test_suite/test_future_compat.sh), a version-4 container whose header blob is brotli-coded (read through the system's
    libbrotlidec; where that library is missing the file must be REFUSED with status 200 -- never produce bytes for it)."""
    import ctypes
    from lepton_b200 import lib
    from lepton_b200 import LeptonB200FileCodec
    names = ["gold-legacy.lep", "narrowrst.lep"]
    fc = LeptonB200FileCodec(0, host_threads=4)
    back = fc.decompress([files[n] for n in names])
    fc.close()
    st, out = back[0]
    assert st == 0, (names[0], st)
    assert md5(out) == expected[names[0]]["decoded_md5"], names[0]
    L = lib()
    L.lepb200_host_brotli_available.restype = ctypes.c_int
    if L.lepb200_host_brotli_available() == 1:
        assert back[1][0] == 0 and md5(back[1][1]) == expected["narrowrst.lep"]["decoded_md5"] == "07e9021d35114bd69f44f5bc1c3788e3"
    else:
        assert back[1][0] == 200 and back[1][1] == b""
