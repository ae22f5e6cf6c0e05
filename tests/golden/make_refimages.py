#!/usr/bin/env python
"""Record what the UNMODIFIED reference CLI does with every file of the reference repository's images/ directory, as
tests/golden/refimages.json (tests/test_gpu_refimages.py compares the CUDA path with it).

    python tests/golden/make_refimages.py <reference checkout>/images

needs oracle/_ref/lepton (`make -C oracle REF=<reference checkout>`).  The repository keeps the images that are small
enough to keep (tests/golden/, copied verbatim; a missing one is copied from the images directory), the first 4 KB of
arithmetic.jpg (its headers already make the reference refuse the file) and, for the photo-sized images it cannot keep
(hq, iphone, iphonecity, slr*, trunc), JPEGs of the same kinds that tests/helpers.synth_jpeg generates on the spot.
Per file the JSON holds:

  fixture / synth          where the input comes from: a path under tests/golden/, or synth_jpeg's arguments (+ truncate:
                           the share of the file kept, for a truncated JPEG)
  jpg_md5 / jpg_size       the input
  rc_skipverify            exit code of `lepton -unjailed -skipverify -allowprogressive in.jpg out.lep`
  rc_verify                exit code of the same without -skipverify (41 = ROUNDTRIP_FAILURE, roundtripfail.jpg)
  exit_name                the ExitCode name the reference wrote to stderr when it left through custom_exit with an error
                           (src/vp8/util/memory.cc:238-245).  The NUMBER the shell sees is not stable across kernels:
                           custom_exit ends with syscall(SYS_exit) (memory.cc:246-247), which ends one thread, so the
                           process status is that of whichever thread leaves last -- the name is
  lep_md5 / lep_size       the .lep the reference wrote (only when rc_skipverify == 0 and the file is non-empty)
  back_md5                 md5 of what the reference decodes that .lep to (== jpg_md5 unless the file does not round-trip)
  status_want              the status the LIBRARY must report for the file: 0, or the ExitCode of the reference process
                           that meets the error (src/vp8/util/memory.hh:13-39): arithmetic 42 UNSUPPORTED_JPEG
                           (jpgcoder.cc:2911-2925 "image is coded arithm."), badzerorun.jpg 1 ASSERTION_FAILURE
                           (jpgcoder.cc:4951) -- Makefile.am:302-304,357-359 expect them to fail
and for the reference repository's golden .lep vectors that the repository keeps (gold-legacy.lep, narrowrst.lep) the md5
its own test scripts pin for the decoded JPEG (test_suite/test_legacy.sh, test_future_compat.sh).

tests/golden/mixed_corpus.json: md5s of the JPEGs of tests/helpers.mixed_corpus_jpegs and of the .lep files the reference
writes for them (`lepton -unjailed -skipverify -allowprogressive`; tests/test_gpu_parity.py).

tests/golden/reference_cpu.json, for the CPU tests (tests/test_oracle_golden.py, tests/test_host_frontend.py):
  gold_legacy_plane_sha256   sha256 of each coefficient plane the reference dumps (-ujg) for the JPEG gold-legacy.lep decodes to
  large                      a photo-sized JPEG (synth_jpeg arguments): the reference's .lep md5, its thread-segment starts,
                             the md5 of each segment's coded stream, and the sha256 of the planes of its -ujg dump
  thread_flags               per set of -minencodethreads / -maxencodethreads / -evensplit flags and per JPEG (kept fixtures
                             and a photo-sized synth_jpeg one): the thread-segment starts and the md5 of the .lep it writes
"""
import hashlib
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
LEPTON = os.path.join(ROOT, "oracle", "_ref", "lepton")
OUT = os.path.join(HERE, "refimages.json")

# name in images/ -> fixture under tests/golden/
KEPT = {n: n for n in (
    "android.jpg", "androidcrop.jpg", "androidcropoptions.jpg", "androidprogressive.jpg", "androidtrail.jpg", "badzerorun.jpg",
    "colorswap.jpg", "gray2sf.jpg", "grayscale.jpg", "iphonecrop2.jpg", "iphoneprogressive.jpg", "iphoneprogressive2.jpg",
    "narrowrst.jpg", "nofsync.jpg", "singlerowtrunc.jpg", "trailingrst.jpg", "trailingrst2.jpg", "truncatedzerorun.jpg")}
KEPT.update({"roundtripfail.jpg": "legacy/roundtripfail.jpg", "gold-legacy.lep": "legacy/gold-legacy.lep",
             "narrowrst.lep": "future/narrowrst.lep"})
HEADS = {"arithmetic_head.jpg": ("arithmetic.jpg", 4096)}
SYNTH = {
    "synth_4032x3024_q90.jpg": dict(w=4032, h=3024, quality=90, subsampling=2, seed=1),                       # iphone, iphonecity
    "synth_6000x4000_q95_444.jpg": dict(w=6000, h=4000, quality=95, subsampling=0, seed=2),                   # hq, slr*
    "synth_2592x1944_q85_progressive.jpg": dict(w=2592, h=1944, quality=85, subsampling=2, progressive=True, seed=3),
    "synth_3264x2448_q92_trunc.jpg": dict(w=3264, h=2448, quality=92, subsampling=2, seed=4, truncate=0.6),    # trunc
}
STATUS_WANT = {"arithmetic_head.jpg": 42, "badzerorun.jpg": 1}
GOLDEN_LEP_MD5 = {"gold-legacy.lep": "9ffbfc24d1157d0b1ed7a9b53bef4c23", "narrowrst.lep": "07e9021d35114bd69f44f5bc1c3788e3"}


def md5(b):
    return hashlib.md5(b).hexdigest()


def synth(args):
    from helpers import synth_jpeg
    a = dict(args)
    keep = a.pop("truncate", 1.0)
    j = synth_jpeg(**a)
    return j[:int(len(j) * keep)]


def inputs(images):
    """name -> (where, bytes); copies kept fixtures that are missing and checks the others against images/."""
    out = {}
    for name, rel in KEPT.items():
        dst = os.path.join(HERE, rel)
        src = open(os.path.join(images, name), "rb").read()
        if not os.path.exists(dst):
            shutil.copyfile(os.path.join(images, name), dst)
            os.chmod(dst, 0o644)
        assert open(dst, "rb").read() == src, "%s differs from %s in images/" % (rel, name)
        out[name] = ({"fixture": rel}, src)
    for name, (src, n) in HEADS.items():
        head = open(os.path.join(images, src), "rb").read()[:n]
        with open(os.path.join(HERE, name), "wb") as f:
            f.write(head)
        out[name] = ({"fixture": name}, head)
    for name, args in SYNTH.items():
        j = synth(args)
        assert j == synth(args), "%s: the generator is not deterministic" % name
        out[name] = ({"synth": args}, j)
    return out


def main(images):
    expected = {}
    with tempfile.TemporaryDirectory() as td:
        for name, (where, data) in sorted(inputs(images).items()):
            src = os.path.join(td, "in")
            with open(src, "wb") as f:
                f.write(data)
            if name.endswith(".lep"):
                back = os.path.join(td, "g.jpg")
                rc = subprocess.run([LEPTON, "-unjailed", src, back], capture_output=True).returncode
                got = md5(open(back, "rb").read()) if rc == 0 else None
                assert got == GOLDEN_LEP_MD5[name], (name, rc, got)          # the reference still meets its own golden md5
                expected[name] = dict(where, lep_md5=md5(data), lep_size=len(data), decoded_md5=GOLDEN_LEP_MD5[name])
                continue
            e = dict(where, jpg_md5=md5(data), jpg_size=len(data))
            lep = os.path.join(td, "o.lep")
            for key, flags in (("rc_skipverify", ["-skipverify"]), ("rc_verify", [])):
                if os.path.exists(lep):
                    os.unlink(lep)
                run = subprocess.run([LEPTON, "-unjailed", "-allowprogressive"] + flags + [src, lep], capture_output=True)
                e[key] = run.returncode
                names = re.findall(rb"^([A-Z][A-Z0-9_]{3,})$", run.stderr, re.M)
                e["exit_name" if key == "rc_skipverify" else "exit_name_verify"] = names[-1].decode() if names else None
                if key == "rc_skipverify" and e[key] == 0 and os.path.getsize(lep) > 0:
                    ld = open(lep, "rb").read()
                    e.update(lep_md5=md5(ld), lep_size=len(ld))
                    back = os.path.join(td, "b.jpg")
                    rc = subprocess.run([LEPTON, "-unjailed", lep, back], capture_output=True).returncode
                    e["back_md5"] = md5(open(back, "rb").read()) if rc == 0 else None
            e["status_want"] = STATUS_WANT.get(name, 0)
            assert (e["status_want"] == 0) == ("lep_md5" in e), (name, e)
            expected[name] = e
            print(name, e.get("lep_size"), e["rc_skipverify"], e["rc_verify"], e["exit_name"], flush=True)
    with open(OUT, "w") as f:
        json.dump(expected, f, indent=1, sort_keys=True)
        f.write("\n")
    from helpers import mixed_corpus_jpegs
    mixed = {"jpg_md5": [], "lep_md5": []}
    with tempfile.TemporaryDirectory() as td:
        src, lep = os.path.join(td, "in.jpg"), os.path.join(td, "o.lep")
        for j in mixed_corpus_jpegs():
            with open(src, "wb") as f:
                f.write(j)
            subprocess.run([LEPTON, "-unjailed", "-skipverify", "-allowprogressive", src, lep], capture_output=True, check=True)
            mixed["jpg_md5"].append(md5(j))
            mixed["lep_md5"].append(md5(open(lep, "rb").read()))
    with open(os.path.join(HERE, "mixed_corpus.json"), "w") as f:
        json.dump(mixed, f, indent=1)
        f.write("\n")
    reference_cpu()


LARGE = dict(w=4032, h=3024, quality=90, subsampling=2, seed=6)
THREAD_FLAGS = [["-maxencodethreads=1"], ["-maxencodethreads=2"], ["-maxencodethreads=3", "-minencodethreads=3"], ["-minencodethreads=8"],
                ["-minencodethreads=5", "-maxencodethreads=6"], ["-evensplit"], ["-evensplit", "-minencodethreads=8"]]
THREAD_FILES = {"androidcrop.jpg": {"fixture": "androidcrop.jpg"}, "iphonecrop2.jpg": {"fixture": "iphonecrop2.jpg"},
                "synth_6000x4000_q95_444.jpg": {"synth": SYNTH["synth_6000x4000_q95_444.jpg"]}}


def reference_cpu():
    import hashlib as hl
    import lepfmt

    def planes_sha(jpg, td):
        ujg = os.path.join(td, "a.ujg")
        subprocess.run([LEPTON, "-unjailed", "-ujg", "-skipverify", jpg, ujg], capture_output=True, check=True)
        _, planes = lepfmt.parse_ujg_planes(open(ujg, "rb").read())
        return [hl.sha256(p.tobytes()).hexdigest() for p in planes]

    out = {}
    with tempfile.TemporaryDirectory() as td:
        jpg, lep = os.path.join(td, "in.jpg"), os.path.join(td, "o.lep")
        subprocess.run([LEPTON, "-unjailed", os.path.join(HERE, "legacy", "gold-legacy.lep"), jpg], capture_output=True, check=True)
        assert md5(open(jpg, "rb").read()) == GOLDEN_LEP_MD5["gold-legacy.lep"]
        out["gold_legacy_plane_sha256"] = planes_sha(jpg, td)
        with open(jpg, "wb") as f:
            f.write(synth(LARGE))
        subprocess.run([LEPTON, "-unjailed", "-skipverify", jpg, lep], capture_output=True, check=True)
        ld = open(lep, "rb").read()
        lf = lepfmt.parse_container(ld)
        out["large"] = {"synth": LARGE, "lep_md5": md5(ld), "luma_y_start": [h.luma_y_start for h in lf.handoffs],
                        "stream_md5": [md5(s) for s in lepfmt.demux(lf.payload, lf.version)[:lf.nseg]],
                        "plane_sha256": planes_sha(jpg, td)}
        tf = {}
        for flags in THREAD_FLAGS:
            per = tf[" ".join(flags)] = {}
            for name, where in THREAD_FILES.items():
                with open(jpg, "wb") as f:
                    f.write(open(os.path.join(HERE, where["fixture"]), "rb").read() if "fixture" in where else synth(where["synth"]))
                subprocess.run([LEPTON, "-skipverify", "-unjailed"] + flags + [jpg, lep], capture_output=True, check=True)
                ld = open(lep, "rb").read()
                per[name] = dict(where, luma_y_start=[h.luma_y_start for h in lepfmt.parse_container(ld).handoffs], lep_md5=md5(ld))
        out["thread_flags"] = tf
    with open(os.path.join(HERE, "reference_cpu.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
