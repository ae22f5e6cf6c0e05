#!/usr/bin/env python
"""bench.py -- Lepton arithmetic-coding hot path on B200: JPEG MB/s encode+decode, roofline fractions, CPU baseline.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line.

Metric (BASELINE.json): "JPEG MB/s encode+decode; bit-exact round-trip pass rate".  A "step" is one ROUND TRIP of the hot
path over one batch of synthetic input: encode (coefficient planes -> per-segment bool-coder streams) followed by decode
(streams -> coefficient planes).  The default workload is BASELINE.json configs[1]: 4096 x synthetic 1920x1080 4:2:0 q=85
baseline JPEGs per GPU (weak scaling: every rank codes its own batch, no collective on the data path).
  value    = JPEG MB/s through BOTH directions = input-JPEG bytes / (encode kernel time + decode kernel time), planes /
             streams resident in HBM, CUDA events; `encode` and `decode` carry the per-direction rates and rooflines
  e2e      = the same metric through the file-level C ABI with HOST buffers: JPEG bytes in host memory -> .lep bytes in
             host memory (lepb200_compress_jpegs) and back (lepb200_decompress_leps), wall clock; e2e.encode / e2e.decode
  parity_vs_reference = the .lep files of the e2e leg compared byte for byte with what the UNMODIFIED reference CLI
             writes for the same JPEGs (the cpu_baseline leg keeps them), and the restored JPEGs with the inputs.  The line
             is refused (exit 3) when any file differs: a fast path with different bytes is not a result.
  --impl reference : the unmodified reference CLI (oracle/_ref/lepton) on the box's host cores, encode + decode of a
             bounded sample per step.
  --config 3|4|5 : the other BASELINE.json workloads through the file-level API (mixed sizes enc+dec; 4K 4:4:4
             progressive encode; decode-only thumbnails with p50 latency).
"""
import argparse
import hashlib
import io
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    2: "4096x synthetic 1920x1080 4:2:0 q=85 baseline JPEGs, encode + decode round trip",
    3: "65536x mixed 256^2-4096^2 baseline JPEGs ({4:2:0,4:4:4} x q{75,85,95}), encode+decode sharded across 8 GPUs (8192 per GPU)",
    4: "1024x 3840x2160 4:4:4 progressive JPEGs (-allowprogressive), encode, 128 per GPU",
    5: "decode-only .lep->.jpg stream, 640x480 4:2:0 q=85 thumbnails (1M across 8 GPUs), p50 per-image latency",
}
DEFAULT_IMAGES = {2: 4096, 3: 8192, 4: 128, 5: 131072}
DEFAULT_DISTINCT = {2: 256, 3: 96, 4: 16, 5: 256}


# ---------------------------------------------------------------------------------------------- synthetic corpus
def synth_pixels(seed, w, h):
    """Deterministic photo-like content: low-frequency gradients + band-limited noise (seed = image index)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    img = np.zeros((h, w, 3), np.float32)
    for c in range(3):
        a = rng.uniform(-1, 1, 6)
        img[..., c] = 128 + 60 * (a[0] * xx / w + a[1] * yy / h) + 40 * np.sin(
            2 * np.pi * (a[2] * 3 * xx / w + a[3] * 2 * yy / h) + a[4] * 6)
    for scale, amp in ((16, 28.0), (4, 12.0), (1, 4.0)):
        n = rng.normal(0, 1, (h // scale + 2, w // scale + 2)).astype(np.float32)
        if scale > 1:
            n = np.kron(n, np.ones((scale, scale), np.float32))[:h, :w]
            s2 = scale // 2
            n = (n + np.roll(n, s2, 0) + np.roll(n, s2, 1) + np.roll(np.roll(n, s2, 0), s2, 1)) / 4
        else:
            n = n[:h, :w]
        img += amp * n[..., None] * rng.uniform(0.6, 1.0, 3).astype(np.float32)
    return np.clip(img, 0, 255).astype(np.uint8)


def image_spec(config, seed):
    """(width, height, quality, subsampling, progressive) of synthetic image `seed` of a BASELINE config (SURVEY 8(d))."""
    import numpy as np
    if config == 2:
        return 1920, 1080, 85, 2, False
    if config == 3:
        rng = np.random.default_rng(1_000_003 * 3 + seed)
        side = int(rng.integers(256, 4097))
        return side, side, (75, 85, 95)[int(rng.integers(0, 3))], (2, 0)[int(rng.integers(0, 2))], False
    if config == 4:
        return 3840, 2160, 85, 0, True
    return 640, 480, 85, 2, False


def synth_jpeg(arg):
    from PIL import Image, ImageFile
    ImageFile.MAXBLOCK = 1 << 26
    config, seed = arg
    w, h, q, sub, prog = image_spec(config, seed)
    b = io.BytesIO()
    Image.fromarray(synth_pixels(seed, w, h), "RGB").save(b, "JPEG", quality=q, subsampling=sub, optimize=False, progressive=prog)
    return b.getvalue()


def make_corpus(config, distinct, seed0=0):
    """`distinct` different JPEGs of the config's shape (generated in parallel processes)."""
    from concurrent.futures import ProcessPoolExecutor
    workers = max(1, min(distinct, effective_cores(), 32))
    with ProcessPoolExecutor(workers) as ex:
        return list(ex.map(synth_jpeg, [(config, s) for s in range(seed0, seed0 + distinct)]))


def pin_to_gpu_numa_node(local_rank, world, want_threads):
    """Ranks of a multi-GPU run: keep this rank's threads (and the pinned staging buffers they first touch) on the NUMA node
    its GPU hangs on (/sys/bus/pci/devices/<id>/local_cpulist).  Returns the note that goes into the JSON line.  Does nothing
    when the node cannot be read, is the whole machine, or is too small for the threads of all the ranks whose GPUs share it
    (2 or 4 ranks on the GPUs of one socket keep the whole machine)."""
    try:
        import torch

        def cpulist(i):
            pr = torch.cuda.get_device_properties(i)
            dev = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            return dev, open("/sys/bus/pci/devices/%s/local_cpulist" % dev).read().strip()

        dev, cl = cpulist(local_rank)
        sharing = sum(1 for i in range(world) if cpulist(i)[1] == cl)
        cpus = set()
        for part in cl.split(","):
            if part:
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        now = os.sched_getaffinity(0)
        use = cpus & now
        if not use or use == now or len(use) < max(1, want_threads) * sharing:
            return "not pinned (GPU %s: local cpus %s, %d usable of %d allowed, %d ranks on this node)" % (dev, cl or "?", len(use), len(now), sharing)
        os.sched_setaffinity(0, use)
        return "pinned to the %d cores of GPU %s's NUMA node (%s), shared by %d ranks" % (len(use), dev, cl, sharing)
    except Exception as ex:          # no sysfs entry, no permission: run unpinned
        return "not pinned (%s)" % type(ex).__name__


def effective_cores():
    """CPU cores this process may actually use: affinity mask and cgroup quota, whichever is smaller."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p))))
    except Exception:
        pass
    return max(1, n)


# ---------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self.reasons = set()
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                self.samples.append((float(f[0]), float(f[1])))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(s[0] for s in self.samples)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.samples[0][1] if self.samples else None,
                "reasons": sorted(self.reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- reference arm / cpu baseline
REF_LEPTON = os.path.join(ROOT, "oracle", "_ref", "lepton")


def run_reference_sample(jpegs, workers, decode=True, keep=None, flags=()):
    """Round trip of every JPEG through the UNMODIFIED reference CLI, `workers` concurrent processes ("backfill" mode
    of src/lepton/benchmark.cc:388-423): in.jpg -> .lep, then .lep -> .jpg.  Returns (encode_s, decode_s, bytes,
    restored_equal).  `keep` (dict) receives md5 -> the .lep bytes the reference wrote for each distinct input."""
    from concurrent.futures import ThreadPoolExecutor
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as td:
        paths = []
        for i, j in enumerate(jpegs):
            p = os.path.join(td, "i%05d.jpg" % i)
            with open(p, "wb") as f:
                f.write(j)
            paths.append(p)

        def enc(p):
            return subprocess.run([REF_LEPTON, "-skipverify", "-unjailed"] + list(flags) + [p, p[:-4] + ".lep"], stdout=subprocess.DEVNULL,
                                  stderr=subprocess.DEVNULL).returncode

        def dec(p):
            return subprocess.run([REF_LEPTON, "-unjailed"] + list(flags) + [p[:-4] + ".lep", p[:-4] + ".out.jpg"], stdout=subprocess.DEVNULL,
                                  stderr=subprocess.DEVNULL).returncode
        t0 = time.perf_counter()
        with ThreadPoolExecutor(workers) as ex:
            rcs = list(ex.map(enc, paths))
        t_enc = time.perf_counter() - t0
        if any(rcs):
            raise RuntimeError("reference CLI failed to encode the sample: %r" % rcs[:8])
        t_dec, equal = 0.0, None
        if decode:
            t0 = time.perf_counter()
            with ThreadPoolExecutor(workers) as ex:
                rcs = list(ex.map(dec, paths))
            t_dec = time.perf_counter() - t0
            if any(rcs):
                raise RuntimeError("reference CLI failed to decode the sample: %r" % rcs[:8])
            equal = sum(int(open(p[:-4] + ".out.jpg", "rb").read() == j) for p, j in zip(paths, jpegs))
        if keep is not None:
            for p, j in zip(paths, jpegs):
                k = hashlib.md5(j).hexdigest()
                if k not in keep:
                    keep[k] = open(p[:-4] + ".lep", "rb").read()
    return t_enc, t_dec, sum(len(j) for j in jpegs), equal


def cpu_baseline(distinct_jpegs, sample_files, decode=True, keep=None, flags=()):
    cores = effective_cores()
    n = max(sample_files, len(distinct_jpegs)) if keep is not None else sample_files     # parity needs every distinct file once
    jp = [distinct_jpegs[i % len(distinct_jpegs)] for i in range(n)]
    t_enc, t_dec, nbytes, equal = run_reference_sample(jp, cores, decode=decode, keep=keep, flags=flags)
    out = {"value": nbytes / (t_enc + t_dec) / 1e6, "unit": "MB/s", "cores": cores, "kind": "reference",
           "encode": {"value": nbytes / t_enc / 1e6, "unit": "MB/s"},
           "sample": "%d files (%.1f MB JPEG) of the workload through oracle/_ref/lepton (-skipverify -unjailed; then .lep -> .jpg), %d "
                     "concurrent processes, wall clock incl. process spawn; value = bytes / (encode s + decode s)" % (n, nbytes / 1e6, cores)}
    if decode:
        out["decode"] = {"value": nbytes / t_dec / 1e6, "unit": "MB/s", "restored_equal": equal, "files": n}
    return out


def md5(b):
    return hashlib.md5(b).hexdigest()


# ---------------------------------------------------------------------------------------------- --dump-outputs
DUMP_LIMIT = 64 << 20


class OutputDump:
    """What the timed path returned in its last step, as DIR/<name>.npy (float32 / float64), so that two builds run with the
    same arguments (hence the same inputs) can be compared output for output.  Byte strings (coded streams, files) are
    kept whole for a fixed, seeded sample of them; all files together stay under DUMP_LIMIT bytes."""

    def __init__(self, directory):
        self.dir = directory
        self.arrays = {}

    def add(self, name, values, dtype="float64"):
        import numpy as np
        self.arrays[name] = np.asarray(values, dtype=dtype)

    def add_bytes(self, name, lengths, fetch, budget):
        """Byte strings of the given lengths, `fetch(indices)` -> their bytes.  <name>_lengths: every length;
        <name>_index: a seeded sample of whole strings that fits `budget` bytes as float32; <name>: their bytes, in order."""
        import numpy as np
        keep, used = [], 0
        for i in np.random.default_rng(0).permutation(len(lengths)):
            if used + 4 * lengths[i] <= budget:
                keep.append(int(i))
                used += 4 * lengths[i]
        keep.sort()
        self.add(name + "_lengths", lengths)
        self.add(name + "_index", keep)
        self.add(name, np.frombuffer(b"".join(fetch(keep)), np.uint8), "float32")

    def write(self):
        import numpy as np
        total = sum(a.nbytes + 256 for a in self.arrays.values())          # 256: more than a .npy header takes
        assert total <= DUMP_LIMIT, "output dump of %d bytes exceeds %d" % (total, DUMP_LIMIT)
        os.makedirs(self.dir, exist_ok=True)
        for name, a in self.arrays.items():
            np.save(os.path.join(self.dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--images", type=int, default=0, help="images per GPU per step (0 = the config's share per GPU)")
    ap.add_argument("--distinct", type=int, default=0, help="distinct synthetic images replicated to --images (0 = per config)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed steps of the file-level legs (0 = --steps)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-only", action="store_true", help="diagnostic: skip the device-resident legs (the line then has no `value`)")
    ap.add_argument("--no-decode", action="store_true")
    ap.add_argument("--host-threads", type=int, default=0, help="host threads for the e2e stage (0 = effective cores / ranks)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=512)
    ap.add_argument("--batch", type=int, default=1024, help="config 5: files per decode call (latency = time of a call)")
    ap.add_argument("--streams", type=int, default=4, help="config 5: decode calls in flight (one codec + one submitting thread each), like a server that keeps several requests going")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed legs returned in their last step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    cfg = args.config
    if args.e2e_steps <= 0:
        args.e2e_steps = args.steps
    if args.images <= 0:
        args.images = DEFAULT_IMAGES[cfg]
    if args.distinct <= 0:
        args.distinct = DEFAULT_DISTINCT[cfg]
    args.distinct = min(args.distinct, args.images)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != max(args.gpus, 1) and world > 1:
        args.gpus = world

    config = {"workload": WORKLOADS[cfg], "baseline_config": cfg, "images_per_gpu": args.images, "distinct_images": args.distinct,
              "parallelism": "independent per-GPU batches x%d (no collective on the data path)" % max(world, 1)}
    if cfg == 2:
        config.update(width=1920, height=1080, subsampling="4:2:0", quality=85,
                      l2="inputs (%.1f GB of coefficient planes per GPU) far exceed the 126 MB L2" % (args.images * 6266880 / 1e9))
    metric = "JPEG MB/s encode+decode" if cfg in (2, 3) else ("JPEG MB/s encode" if cfg == 4 else "JPEG MB/s decode")
    ref_flags = ("-allowprogressive",) if cfg == 4 else ()

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        if not os.path.exists(REF_LEPTON):
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/lepton not built (run __graft_entry__.build() where /root/reference exists)"}))
            return 0
        distinct = make_corpus(cfg, min(args.distinct, 64))
        cores = effective_cores()
        nsample = args.cpu_sample if cfg == 2 else max(cores, min(args.cpu_sample, 64 if cfg == 3 else (16 if cfg == 4 else 2048)))
        sample = [distinct[i % len(distinct)] for i in range(nsample)]
        for _ in range(max(args.warmup, 0)):
            run_reference_sample(sample[:max(8, cores // 4)], cores, flags=ref_flags)
        te = td = 0.0
        tot_b = 0
        for _ in range(args.steps):
            a, b, nb, _eq = run_reference_sample(sample, cores, decode=cfg != 4, flags=ref_flags)
            te += a
            td += b
            tot_b += nb
        tot_t = td if cfg == 5 else te + td
        v = tot_b / tot_t / 1e6
        line = {"impl": "reference", "metric": metric, "value": v, "unit": "MB/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "int16 coefficients / u8 probabilities (integer)",
                "data": "synthetic", "config": config,
                "encode": {"value": tot_b / te / 1e6, "unit": "MB/s"},
                "cpu_baseline": {"value": v, "unit": "MB/s", "cores": cores, "kind": "reference",
                                 "sample": "%d files per step through oracle/_ref/lepton (-skipverify -unjailed, then .lep -> .jpg), %d concurrent "
                                           "processes; value = bytes / (encode s + decode s)" % (len(sample), cores)},
                "e2e": {"value": v, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        if td > 0:
            line["decode"] = {"value": tot_b / td / 1e6, "unit": "MB/s"}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from lepton_b200 import HostJpeg, LeptonB200Codec, LeptonB200FileCodec
    from lepton_b200.sharding import reduce_job_throughput

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def rmax(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def rsum(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t[0])

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    peak_source = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)"
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))
    except Exception:
        pass

    distinct = make_corpus(cfg, args.distinct, seed0=100000 * rank)
    jpegs = [distinct[i % len(distinct)] for i in range(args.images)]
    jpeg_bytes = sum(len(j) for j in jpegs)
    threads = args.host_threads or max(1, effective_cores() // max(world, 1))
    numa_note = pin_to_gpu_numa_node(local_rank, world, threads) if world > 1 and not os.environ.get("LEPB200_BENCH_NO_PIN") else None

    line = {"metric": metric, "unit": "MB/s", "n_gpus": max(world, 1), "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int16 coefficients / u8 probabilities (integer)", "data": "synthetic", "config": config}
    dump = OutputDump(args.dump_outputs) if args.dump_outputs and rank == 0 else None

    # ================================================================== device-resident legs (config 2 only)
    sampler = ClockSampler(local_rank)
    if cfg == 2 and not args.e2e_only:
        hjs = [HostJpeg(j) for j in distinct]
        for h in hjs:
            assert h.status == 0, h.error
        base_imgs = [h.coef_image() for h in hjs]
        imgs = [base_imgs[i % len(base_imgs)] for i in range(args.images)]
        nseg = sum(im.nseg for im in imgs)
        blocks = sum(im.blocks() for im in imgs)

        codec = LeptonB200Codec(local_rank)
        codec.encode_upload(imgs)            # H2D: planes become resident in HBM
        codec.encode_launch()
        res = codec.encode_fetch(copy=False)
        assert all(s.status == 0 for r in res for s in r), "encode failed"
        stream_bytes = sum(codec.last_lens)
        ndecisions = sum(s.ndecisions for r in res for s in r)
        alg_bytes = codec.last_algorithmic_bytes
        for _ in range(max(args.warmup - 1, 0)):
            codec.encode_launch()
            codec.sync()
        barrier()
        sampler.start()
        launches0 = codec.kernel_launches
        t_wall0 = time.perf_counter()
        kernel_ms, sym_ms = [], []
        for _ in range(args.steps):
            codec.encode_launch()
            codec.sync()
            kernel_ms.append(codec.last_kernel_ms)
            sym_ms.append(codec.last_symbolise_ms)
        barrier()
        t_wall = time.perf_counter() - t_wall0
        launches = codec.kernel_launches - launches0
        enc_s = rmax(sum(kernel_ms) / 1e3)                     # max over ranks of the device time of all timed steps
        total_jpeg = rsum(jpeg_bytes)
        avg_step_s = (sum(kernel_ms) / len(kernel_ms)) / 1e3          # kernel A + kernel B
        avg_a_s = (sum(sym_ms) / len(sym_ms)) / 1e3                  # kernel A (symbolise + model update)
        enc = {"value": total_jpeg * args.steps / enc_s / 1e6, "unit": "MB/s", "ms_per_step": 1e3 * enc_s / args.steps,
               "roofline": {"bound": "hbm", "achieved": alg_bytes / avg_a_s / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": alg_bytes / avg_a_s / 1e9 / peak, "traffic": traffic.get("lep_encode_kernel"),
                            "peak_source": peak_source, "algorithmic_bytes_per_launch": int(alg_bytes),
                            "kernel": "lep_encode_kernel (symbolise + model update); lep_rangecode_kernel is the remainder of the step",
                            "kernel_ms": 1e3 * avg_a_s, "rangecode_kernel_ms": 1e3 * (avg_step_s - avg_a_s),
                            "step_frac": alg_bytes / avg_step_s / 1e9 / peak,
                            "decisions_per_s": ndecisions / avg_step_s, "decisions_per_launch": int(ndecisions)}}

        # ---------------------------------------------------------------- decode direction + round trip (same batch)
        res = codec.encode_fetch(copy=True)                       # streams of the last launch, on the host
        streams = [[s.data for s in r] for r in res]
        if dump:
            segs = [s for r in res for s in r]
            dump.add("encode_status", [s.status for s in segs])
            dump.add("encode_ndecisions", [s.ndecisions for s in segs])
            dump.add_bytes("encode_streams", [len(s.data) for s in segs], lambda ix: [segs[i].data for i in ix], 16 << 20)
        from lepton_b200 import CoefImage
        outs = [CoefImage(ncmp=im.ncmp, mcuv=im.mcuv, bch=im.bch, bcv=im.bcv, qtables_zigzag=im.qtables_zigzag,
                          planes=[np.full_like(p, 1) for p in im.planes], luma_y_start=im.luma_y_start) for im in base_imgs]
        st = codec.decode_images(outs, streams[:len(outs)])
        ok = k = 0
        for im, o in zip(base_imgs, outs):
            good = all(s == 0 for s in st[k:k + im.nseg]) and all(np.array_equal(a, b) for a, b in zip(im.planes, o.planes))
            ok += int(good)
            k += im.nseg
        del outs
        codec.decode_upload(imgs, streams)
        for _ in range(max(args.warmup, 3) - 1):
            codec.decode_launch()
            codec.sync()
        barrier()
        l0 = codec.kernel_launches
        dms = []
        for _ in range(args.steps):
            codec.decode_launch()
            codec.sync()
            dms.append(codec.last_kernel_ms)
        barrier()
        launches += codec.kernel_launches - l0
        clocks = sampler.stop()
        if dump:
            # planes of a seeded sample of 4 images, and of those a seeded sample of blocks: (image, block index over the
            # image's components in order) -> 64 coefficients
            pick = sorted(int(i) for i in np.random.default_rng(0).choice(len(imgs), size=min(4, len(imgs)), replace=False))
            into = {i: [np.empty_like(p) for p in imgs[i].planes] for i in pick}
            dump.add("decode_status", codec.decode_fetch(into))
            rows, index = [], []
            for i in pick:
                allb = np.concatenate([p.reshape(-1, 64) for p in into[i]])
                sel = np.sort(np.random.default_rng(i).choice(len(allb), size=min(4096, len(allb)), replace=False))
                rows.append(allb[sel])
                index += [(i, int(b)) for b in sel]
            dump.add("decode_blocks", np.concatenate(rows), "float32")
            dump.add("decode_block_index", index)
        dec_s = rmax(sum(dms) / 1e3)
        avg_d_s = (sum(dms) / len(dms)) / 1e3
        dmode = int(os.environ.get("LEPB200_DEC_MODE", "0"))
        group = dmode == 2 or (dmode == 0 and nseg >= int(os.environ.get("LEPB200_DEC_GROUP_MIN", "10240")))
        dec_kernel = ("lep_decode_g2_kernel<%s> (group kernel: %s lanes per thread-segment, lock step)" % ((os.environ.get("LEPB200_DEC_LANES", "4"),) * 2)
                      if group else "lep_decode_kernel (one warp per thread-segment)")
        dec = {"value": total_jpeg * args.steps / dec_s / 1e6, "unit": "MB/s", "ms_per_step": 1e3 * dec_s / args.steps,
               "roundtrip_pass_rate": ok / len(base_imgs), "roundtrip_images": len(base_imgs),
               "roofline": {"bound": "hbm", "achieved": alg_bytes / avg_d_s / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": alg_bytes / avg_d_s / 1e9 / peak, "traffic": traffic.get("decode_kernel"), "peak_source": peak_source,
                            "algorithmic_bytes_per_launch": int(alg_bytes), "kernel": dec_kernel, "kernel_ms": 1e3 * avg_d_s,
                            "decisions_per_s": ndecisions / avg_d_s, "decisions_per_launch": int(ndecisions)}}
        codec.close()
        codec = None
        rt_s = enc_s + dec_s
        dominant = dec if avg_d_s >= avg_a_s else enc
        line.update(value=total_jpeg * args.steps / rt_s / 1e6, ms_per_step=1e3 * rt_s / args.steps, clocks=clocks,
                    gpu_launches=int(launches), roofline=dict(dominant["roofline"]), encode=enc, decode=dec,
                    roundtrip_pass_rate=dec["roundtrip_pass_rate"],
                    wall_ms_per_step_encode=1e3 * rmax(t_wall) / args.steps,
                    batch={"jpeg_bytes": int(jpeg_bytes), "segments": int(nseg), "blocks": int(blocks), "stream_bytes": int(stream_bytes)})
        line["roofline"]["note"] = "dominant kernel of the round trip (the longer of kernel A and the decode kernel); per-direction rooflines under encode / decode"
        del imgs, base_imgs, hjs, streams, res

    # ================================================================== file-level legs (host buffers in, host buffers out)
    ref_leps = {}
    parity = None
    if not args.no_e2e or cfg != 2:
        fc = LeptonB200FileCodec(local_rank, host_threads=threads)
        if cfg == 5:
            # decode-only stream: the .lep files are produced once (untimed), then decoded in calls of --batch files
            r = fc.compress(fc.prepare(distinct), copy=True)
            assert all(st == 0 for st, _ in r)
            dleps = [b for _, b in r]
            leps = [dleps[i % len(dleps)] for i in range(args.images)]
            nb = max(1, min(args.batch, args.images))
            handles = [fc.prepare(leps[i:i + nb]) for i in range(0, args.images, nb)]
            back = fc.decompress(handles[0], copy=True)          # warm-up + check
            exact = sum(int(st == 0 and b == jpegs[i]) for i, (st, b) in enumerate(back))
            assert exact == len(back), "thumbnail decode differs from the input"
            barrier()
            if not sampler.samples and sampler.proc is None:
                sampler.start()
            # K calls in flight: K codecs (own contexts / streams), K submitting threads taking calls from one queue.  A call
            # of 1024 one-segment thumbnails is 1024 serial chains -- a fraction of the machine -- so calls overlap on the
            # device; ctypes releases the GIL for the duration of a call
            K = max(1, min(args.streams, len(handles)))
            codecs = [fc] + [LeptonB200FileCodec(local_rank, host_threads=max(1, threads // K)) for _ in range(K - 1)]
            for cdc in codecs[1:]:
                cdc.decompress(handles[0], copy=False)           # warm-up of every codec (arenas)
            barrier()
            lat = []
            l0 = sum(cdc.kernel_launches for cdc in codecs)
            import queue
            # a step is one pass over the calls; every pass has its own result arrays, so that no two calls in flight
            # write to the same one
            passes = [handles] + [[fc.prepare(leps[i:i + nb]) for i in range(0, args.images, nb)] for _ in range(args.steps - 1)]
            q = queue.Queue()
            for p in range(args.steps):
                for h in range(len(handles)):
                    q.put((p, h))
            lock = threading.Lock()
            last_call = {}

            def serve(cdc):
                while True:
                    try:
                        p, h = q.get_nowait()
                    except queue.Empty:
                        return
                    t1 = time.perf_counter()
                    cdc.decompress(passes[p][h], copy=False)
                    d1 = time.perf_counter() - t1
                    with lock:
                        lat.append(d1)
                    last_call[id(cdc)] = (p, h)
            t0 = time.perf_counter()
            ths = [threading.Thread(target=serve, args=(cdc,)) for cdc in codecs]
            for t in ths:
                t.start()
            for t in ths:
                t.join()
            barrier()
            dt = rmax(time.perf_counter() - t0)
            nlaunch = sum(cdc.kernel_launches for cdc in codecs) - l0
            if dump:
                # the last call of every codec still holds its output: of those in the last pass, file h * nb + k of call h
                last = passes[-1]
                files = [(h, k) for p, h in sorted(last_call.values()) if p == args.steps - 1 for k in range(last[h][1])]
                got = [fc.results(last[h], [k], copy=False)[0] for h, k in files]
                dump.add("decompress_files", [h * nb + k for h, k in files])
                dump.add("decompress_status", [st for st, _ in got])
                dump.add_bytes("decompress_jpeg", [n for _, n in got],
                               lambda ix: [fc.results(last[files[i][0]], [files[i][1]])[0][1] for i in ix], 48 << 20)
            for cdc in codecs[1:]:
                cdc.close()
            lat.sort()
            total_jpeg = rsum(jpeg_bytes)
            v = total_jpeg * args.steps / dt / 1e6
            line.update(value=v, ms_per_step=1e3 * dt / args.steps, clocks=sampler.stop(), gpu_launches=int(nlaunch),
                        images_per_s=rsum(args.images) * args.steps / dt,
                        latency={"p50_ms": 1e3 * lat[len(lat) // 2], "p90_ms": 1e3 * lat[(len(lat) * 9) // 10], "max_ms": 1e3 * lat[-1],
                                 "files_per_call": nb, "calls": len(lat), "calls_in_flight": K,
                                 "note": "per-image latency = latency of the call that carries the image (one serial chain per thumbnail)"},
                        e2e={"value": v, "unit": "MB/s", "h2d_bytes_per_step": int(sum(len(b) for b in leps)), "d2h_bytes_per_step": int(jpeg_bytes),
                             "api": "lepb200_decompress_leps (.lep bytes -> JPEG bytes, host memory)", "host_threads": threads},
                        roundtrip_pass_rate=exact / len(back))
        else:
            handle = fc.prepare(jpegs)
            r = fc.compress(handle, copy=True)          # warm-up (allocates pinned arenas); keep the .lep files for the way back
            assert all(st == 0 for st, _ in r), [st for st, _ in r if st][:8]
            leps = [b for _, b in r]
            lep_bytes = sum(len(b) for b in leps)
            barrier()
            if cfg != 2 or args.e2e_only:
                sampler.start()
            l0 = fc.kernel_launches
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                last = fc.compress(handle, copy=False)
            barrier()
            e_s = rmax(time.perf_counter() - t0)
            if dump:
                dump.add("compress_status", [st for st, _ in last])
                dump.add_bytes("compress_lep", [n for _, n in last], lambda ix: [b for _, b in fc.results(handle, ix)], 16 << 20)
            total_jpeg = rsum(jpeg_bytes)
            e2e = {"unit": "MB/s", "h2d_bytes_per_step": int(jpeg_bytes), "d2h_bytes_per_step": int(lep_bytes),
                   "h2d_note": "entropy-coded scan bytes (Huffman decode happens on the GPU); files the host has to decode upload 128 B per block instead",
                   "steps": args.e2e_steps, "host_threads": threads, "host_affinity": numa_note, "gpu_launches": fc.kernel_launches - l0,
                   "encode": {"value": total_jpeg * args.e2e_steps / e_s / 1e6, "unit": "MB/s", "ms_per_step": 1e3 * e_s / args.e2e_steps,
                              "api": "lepb200_compress_jpegs (JPEG bytes -> .lep bytes, host memory)", "stage_seconds_last_step": fc.last_timing()}}
            d_s = None
            if cfg != 4 and not args.no_decode:
                lhandle = fc.prepare(leps)
                back = fc.decompress(lhandle, copy=True)       # warm-up + round-trip check of every file
                exact = sum(int(st == 0 and b == j) for (st, b), j in zip(back, jpegs))
                del back
                barrier()
                l0 = fc.kernel_launches
                t0 = time.perf_counter()
                for _ in range(args.e2e_steps):
                    last = fc.decompress(lhandle, copy=False)
                barrier()
                d_s = rmax(time.perf_counter() - t0)
                if dump:
                    dump.add("decompress_status", [st for st, _ in last])
                    dump.add_bytes("decompress_jpeg", [n for _, n in last], lambda ix: [b for _, b in fc.results(lhandle, ix)], 16 << 20)
                e2e["gpu_launches"] += fc.kernel_launches - l0
                e2e["d2h_bytes_per_step"] += int(jpeg_bytes)
                e2e["h2d_bytes_per_step"] += int(lep_bytes)
                e2e["decode"] = {"value": total_jpeg * args.e2e_steps / d_s / 1e6, "unit": "MB/s", "ms_per_step": 1e3 * d_s / args.e2e_steps,
                                 "api": "lepb200_decompress_leps (.lep bytes -> JPEG bytes, host memory)",
                                 "roundtrip_pass_rate": exact / len(jpegs), "roundtrip_files": len(jpegs), "stage_seconds_last_step": fc.last_timing()}
            e2e["value"] = total_jpeg * args.e2e_steps / (e_s + (d_s or 0.0)) / 1e6
            line["e2e"] = e2e
            if cfg != 2 or args.e2e_only:
                line.update(value=e2e["value"], ms_per_step=1e3 * (e_s + (d_s or 0.0)) / args.e2e_steps, clocks=sampler.stop(),
                            gpu_launches=int(e2e["gpu_launches"]), value_note="file-level API only for this config (value == e2e.value)")
                if "decode" in e2e:
                    line["roundtrip_pass_rate"] = e2e["decode"]["roundtrip_pass_rate"]
            # ---- parity against the reference CLI on every distinct file (rank 0; BASELINE.md section 3: a gate before timing counts)
            if rank == 0 and os.path.exists(REF_LEPTON) and not args.no_cpu_baseline:
                line["cpu_baseline"] = cpu_baseline(distinct, args.cpu_sample if cfg == 2 else len(distinct), decode=cfg != 4, keep=ref_leps, flags=ref_flags)
                equal = sum(int(ref_leps.get(md5(j)) == lep) for j, lep in zip(distinct, leps[:len(distinct)]))
                parity = {"files": len(distinct), "lep_equal": equal, "checked_against": "oracle/_ref/lepton (unmodified reference CLI), same run"}
                if "decode" in e2e:
                    parity["jpeg_restored_equal"] = int(round(e2e["decode"]["roundtrip_pass_rate"] * len(jpegs)))
                    parity["jpeg_restored_files"] = len(jpegs)
                line["parity_vs_reference"] = parity
        fc.close()
    if cfg == 5 and rank == 0 and os.path.exists(REF_LEPTON) and not args.no_cpu_baseline:
        cb = cpu_baseline(distinct, min(2048, args.images), decode=True, flags=ref_flags)
        cb["value"] = cb["decode"]["value"]
        line["cpu_baseline"] = cb
    if rank == 0 and "cpu_baseline" not in line and not args.no_cpu_baseline:
        if os.path.exists(REF_LEPTON):
            line["cpu_baseline"] = cpu_baseline(distinct, args.cpu_sample, decode=cfg != 4, flags=ref_flags)
        else:
            line["cpu_baseline"] = {"value": None, "unit": "MB/s", "cores": 0, "kind": "reference", "sample": "oracle/_ref/lepton missing"}

    if dist is not None:
        dist.barrier()
        if rank != 0:
            dist.destroy_process_group()
    if rank != 0:
        return 0
    rc = 0
    if parity is not None and (parity["lep_equal"] != parity["files"] or parity.get("jpeg_restored_equal", 0) != parity.get("jpeg_restored_files", 0)):
        line["invalid"] = "parity gate failed: outputs differ from the reference's -- no throughput is reported"
        for k in ("value", "e2e"):
            line.pop(k, None)
        rc = 3
    if dump:
        dump.write()
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return rc


if __name__ == "__main__":
    sys.exit(main())
