#!/usr/bin/env python3
"""bench.py -- decoded channel-samples/s of the B200 Vorbis decode path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE config 4 -- 4,096 concurrent streams per GPU replicated /
offset from the four TestFiles, full entropy + floor + residue + coupling + IMDCT + window/OLA
decode.  Streams are independent, so ranks shard them with no collective ("scaling": "weak": each
GPU gets its own 4,096 streams; `--scaling strong` splits 4,096 over the ranks instead).

A step = one pass of the hot path (K1 entropy/floor/coupling + K3 IMDCT/OLA) over the whole batch.
  value : whole-job channel-samples/s with packets and tables already resident in HBM, timed with
          CUDA events on the library's stream, max over ranks.
  e2e   : the same metric through the reference-facing C ABI with HOST buffers
          (vpz_decode_files: Ogg images in host memory -> page scan + CRC + header/packet walk on the
          host -> H2D -> K1 -> K3 -> D2H into pinned host PCM), wall clock, max over ranks.
  roofline / roofline_k3 : algorithmic bytes (DESIGN.md) / event-timed kernel duration vs the
          measured HBM copy peak in MEASURED_PEAKS.json.
  cpu_baseline : the CPU oracle (C restatement of the reference .NET path; .NET is not available
          here) on all host cores, one stream per thread, bounded sample.  N=1, rank 0 only.
  config3 / config5 : sub-objects of the default line -- BASELINE config 3 (kernel-only IMDCT + window + OLA
          on 65,536 synthetic stereo blocks: value, roofline incl. ncu DRAM traffic) and config 5 (16,384
          random-access excerpts through vpz_decode_excerpts: value, excerpts/s, its own cpu_baseline = the
          oracle's SeekTo + read on all host cores).  `--workload config3|config5` runs them alone.
  e2e.link_gbs_measured / frac_of_link : copy-only pinned device-to-host bandwidth of this box measured in the
          same process (all ranks at once) and the share of it the e2e step's D2H traffic reaches.
`--impl reference` times that same oracle as the reference arm on the SAME workload: the 4,096 streams of
config 4 per step, whole files, all host cores (both oracle builds: portable -O2 and -O3 -march=native built on
the box; the faster one is the line's value).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
FILES = ["1test", "2test", "3test", "issue6test"]
METRIC = "decoded channel-samples/sec"
UNIT = "channel-samples/s"


def load_files():
    out = []
    for n in FILES:
        with open(os.path.join(ROOT, "tests", "data", n + ".ogg"), "rb") as f:
            out.append(f.read())
    return out


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = "/tmp/vpz_clocks_%d_%d.csv" % (os.getpid(), index)

    def start(self):
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.fh,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()  # the exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 8:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                    power.append(float(f[3]))
                except ValueError:
                    continue
                for nme, v in zip(names, f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm), "power_w_max": max(power) if power else None}
        return out


def stream_assignment(streams, rank, world, scaling):
    """Streams are independent units: rank r decodes `count` streams starting at global stream index
    `first`; no rank ever needs another rank's data (no collective on the data path).
    weak: every rank gets `streams` of its own; strong: `streams` in total are split."""
    if scaling == "weak":
        return rank * streams, streams
    base, extra = divmod(streams, world)
    first = rank * base + min(rank, extra)
    return first, base + (1 if rank < extra else 0)


def stream_file_and_start(g, n_files, n_packets):
    """Global stream g decodes file g % n_files; replica r = g // n_files starts at audio packet
    (7 r) mod count (SURVEY 8(d) config 4: replicated / offset)."""
    f = g % n_files
    return f, (7 * (g // n_files)) % n_packets[f]


def pinned_array(lib, nfloats):
    p = lib.vpz_host_alloc(int(nfloats) * 4)
    if not p:
        raise MemoryError("vpz_host_alloc(%d floats)" % nfloats)
    arr = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=(int(nfloats),))
    return arr, p


def dump_outputs(batch, n_runs, out_dir, window=1024, budget_bytes=48 << 20):
    """Writes what a caller of the timed path receives -- the fp32 PCM of every run of the batch as the last
    decode left it -- so that two builds can be compared output for output.  All of it is ~8 GB per GPU, so:
      pcm_windows.npy  float32: a window of `window` floats (fewer when `budget_bytes` or the run is smaller) of
                       every run, at a seeded offset aligned to whole samples, the windows back to back;
      run_samples.npy  float64: samples per channel of every run;
      run_sums.npy     float64: the sum of every run's PCM, which every decoded value enters."""
    os.makedirs(out_dir, exist_ok=True)
    window = max(1, min(window, budget_bytes // (4 * max(n_runs, 1))))
    rng = np.random.default_rng(0x5EED0004)
    windows, samples, sums = [], np.zeros(n_runs), np.zeros(n_runs)
    for run in range(n_runs):
        pcm = batch.read_run(run)
        flat = pcm.reshape(-1)
        w = min(window, flat.size)
        start = int(rng.integers(0, flat.size - w + 1))
        start -= start % pcm.shape[1]
        windows.append(flat[start:start + w])
        samples[run] = pcm.shape[0]
        sums[run] = flat.sum(dtype=np.float64)
    np.save(os.path.join(out_dir, "pcm_windows.npy"), np.concatenate(windows).astype(np.float32))
    np.save(os.path.join(out_dir, "run_samples.npy"), samples)
    np.save(os.path.join(out_dir, "run_sums.npy"), sums)


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU implementation of the path on the host cores.  The
    reference is C# and cannot be built here, so this is the oracle port (cpu_baseline.kind "port")."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as ob
    files = load_files()
    if args.workload == "config1":
        # BASELINE config 1: TestApp-style decode of TestFiles/1test.ogg to float PCM on the CPU, ONE stream on
        # ONE thread (48,000-float reads until 0, TestApp/Program.cs:42,155); a step = 1,000 whole decodes
        reps = 1000
        for _ in range(max(1, args.warmup)):
            ob.bench_decode(files[:1], reps // 10, 1)
        total, sec = 0, 0.0
        for _ in range(args.steps):
            n, s = ob.bench_decode(files[:1], reps, 1)
            total += n
            sec += s
        v = total / sec
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": 0, "steps": args.steps,
            "warmup": max(1, args.warmup), "ms_per_step": 1e3 * sec / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "TestFiles/1test.ogg",
            "config": {"workload": "config1: TestApp decode of TestFiles/1test.ogg to float PCM on CPU, single stream, "
                                   "single thread (%d whole decodes per step)" % reps,
                       "x_realtime": v / 44100.0, "ms_per_decode": 1e3 * sec / (args.steps * reps),
                       "note": "C restatement of the reference .NET decoder (oracle/); no .NET runtime in this image"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
                             "sample": "%d decodes of 1test.ogg (17,318 samples, mono) per step" % reps},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return
    cores = os.cpu_count() or 1
    if args.workload == "config5":
        # BASELINE config 5 on the CPU: the same 16,384 excerpts (same seed) as the GPU arm, SeekTo + read
        file_of, start, count, nread = config5_excerpts(0)
        builds = {}
        for name, native in (("O2", False), ("O3_march_native", True)):
            if ob.bench_lib(native) is None:
                continue
            for _ in range(max(1, args.warmup)):
                ob.bench_excerpts(files[1:], file_of[:2048], start[:2048], count[:2048], cores, native)
            tot, sec = 0, 0.0
            for _ in range(args.steps):
                n, s = ob.bench_excerpts(files[1:], file_of, start, count, cores, native)
                tot += n
                sec += s
            builds[name] = {"value": tot / sec, "ms_per_step": 1e3 * sec / args.steps}
        best = max(builds, key=lambda k: builds[k]["value"])
        v = builds[best]["value"]
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": max(1, args.warmup), "ms_per_step": builds[best]["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded excerpts of TestFiles)",
            "config": {"workload": "config5: %d random-access excerpts (SeekTo + %d samples per channel on {2,3,issue6}test.ogg), "
                                   "one open reader per (thread, file)" % (file_of.size, nread),
                       "threads": cores, "excerpts_per_s": file_of.size / (builds[best]["ms_per_step"] * 1e-3),
                       "note": "C restatement of the reference .NET decoder (oracle/); no .NET runtime in this image"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "builds": builds, "build": best,
                             "sample": "all %d excerpts per step" % file_of.size},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return
    # the SAME workload as the GPU arm's e2e: stream g of args.streams decodes the whole file g % 4
    njobs = args.streams
    builds = {}
    for name, native in (("O2", False), ("O3_march_native", True)):
        if ob.bench_lib(native) is None:
            continue
        for _ in range(args.warmup):
            ob.bench_decode(files, max(4, njobs // 8), cores, native)
        total, sec = 0, 0.0
        for _ in range(args.steps):
            n, s = ob.bench_decode(files, njobs, cores, native)
            total += n
            sec += s
        builds[name] = {"value": total / sec, "ms_per_step": 1e3 * sec / args.steps}
    best = max(builds, key=lambda k: builds[k]["value"])
    v = builds[best]["value"]
    sample = "all %d streams per step (whole files, stream g = TestFile g %% 4, handed to %d threads by a shared cursor)" % (
        njobs, cores)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": builds[best]["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (TestFiles replicated/offset)",
        "config": {"workload": "config4: %d concurrent streams per GPU replicated/offset from TestFiles/{1,2,3,issue6}test.ogg, "
                               "full entropy+floor+residue+IMDCT decode, stream-sharded" % njobs,
                   "streams_per_gpu": njobs, "threads": cores,
                   "note": "C restatement of the reference .NET decoder (oracle/); no .NET runtime in this image; whole "
                           "files (the GPU arm's e2e decodes exactly these streams)"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "builds": builds, "build": best,
                         "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def config5_excerpts(rank, world=1, scaling="weak", n=16384):
    """The excerpt list of BASELINE config 5 (SURVEY 8(d)): rng(0x5EED0005 + rank), file uniform in {2test, 3test,
    issue6test}, start uniform in [0, total - 4096); totals are the decodable sample counts of the files.
    weak: every rank draws its own n excerpts; strong ("16,384 excerpts across N GPUs"): rank 0's list is THE
    list and rank r takes the contiguous slice stream_assignment gives it."""
    totals = [315790, 288094, 548160]
    nread = 4096
    rng = np.random.default_rng(0x5EED0005 + (rank if scaling == "weak" else 0))
    file_of = rng.integers(0, len(totals), n).astype(np.uint32)
    start = np.array([int(rng.integers(0, totals[f] - nread)) for f in file_of], np.int64)
    count = np.full(n, nread, np.int32)
    if scaling == "strong":
        first, cnt = stream_assignment(n, rank, world, "strong")
        file_of, start, count = file_of[first:first + cnt].copy(), start[first:first + cnt].copy(), count[first:first + cnt].copy()
    return file_of, start, count, nread


def d2h_probe(lib, local_rank, barrier, max_over_ranks, sum_over_ranks, seconds=1.0):
    """Copy-only ceiling of the device-to-host path: a 1 GiB device buffer copied into pinned host memory back
    to back for about `seconds`, on every rank at once (the ranks of one box share its host side).  Returns the
    box-wide GB/s (sum of the ranks' bytes / slowest rank's time)."""
    import torch
    n = 1 << 30
    src = torch.empty(n, dtype=torch.uint8, device="cuda")
    p = lib.vpz_host_alloc(n)
    if not p:
        return None
    dst = torch.frombuffer((C.c_uint8 * n).from_address(p), dtype=torch.uint8)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        dst.copy_(src, non_blocking=True)   # warm-up (first touch of the pinned pages)
        st.synchronize()
        reps = 3
        barrier()
        while True:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(reps):
                dst.copy_(src, non_blocking=True)
            e1.record(st)
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            if ms >= 1e3 * seconds * 0.5 or reps >= 96:
                break
            reps *= 2
    barrier()
    t = max_over_ranks(ms * 1e-3)
    total = sum_over_ranks(float(n) * reps)
    del dst
    lib.vpz_host_free(p)
    return total / t / 1e9


def load_traffic():
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def run_config3(args, ctx, rank, world, barrier, max_over_ranks, sum_over_ranks, local_rank, quick=False):
    """BASELINE config 3: kernel-only batched IMDCT + window + overlap-add on synthetic spectra, 65,536
    stereo blocks per GPU (64 streams x 1,024 blocks, long runs with short transitions: the Markov flag
    sequence and roll-off spectra of SURVEY 8(d), same generator as tests/cases.py).  Returns the JSON line
    (rank 0) -- printed as is by `--workload config3`, embedded as "config3" in the default line."""
    from vorbispizza_b200 import SynthBatch
    lib = ctx.lib
    n_streams, n_blocks, ch = 64, 1024, 2
    rng = np.random.default_rng(0x5EED0001 + rank)
    flags = np.zeros((n_streams, n_blocks), np.uint8)
    for s in range(n_streams):
        cur = 1
        u = rng.random(n_blocks)
        for i in range(n_blocks):
            flags[s, i] = cur
            cur = (0 if u[i] < 1 / 16 else 1) if cur else (1 if u[i] < 1 / 4 else 0)
    if args.all_long:
        flags[:] = 1
    sizes = np.where(flags.reshape(-1) & 1, 1024, 128)
    total = int(sizes.sum()) * ch
    k = np.concatenate([np.tile(np.arange(m, dtype=np.float32), ch) for m in sizes])
    spectra = (rng.standard_normal(total).astype(np.float32) * np.exp2(-k / 128.0) * np.float32(0.02)).astype(np.float32)
    batch = SynthBatch(ctx, ch, 8, 11, flags, spectra)
    samples_rank = batch.total_floats
    clocks = ClockSampler(local_rank)
    clocks.start()
    warm = args.warmup
    for _ in range(warm):
        batch.decode(clip=True, sync=False)
    batch.sync()
    barrier()
    launches0 = lib.vpz_ctx_kernel_launches(ctx._h)
    steps = args.steps
    lib.vpz_ctx_mark(ctx._h, 0)
    for _ in range(steps):
        batch.decode(clip=True, sync=False)
    lib.vpz_ctx_mark(ctx._h, 1)
    ms = lib.vpz_ctx_elapsed_ms(ctx._h, 0, 1)
    batch.sync()
    barrier()
    launches = lib.vpz_ctx_kernel_launches(ctx._h) - launches0
    clk = clocks.stop()
    ms_max = max_over_ranks(ms)
    total_samples = sum_over_ranks(float(samples_rank))
    value = total_samples * steps / (ms_max * 1e-3)
    peak, peak_src = measured_peak()
    k3_ms = ms_max / steps
    a = 8.0 * samples_rank / (k3_ms * 1e-3) / 1e9
    batch.close()
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        # the oracle's Mdct.Reverse + OverlapBuffers + interleaved store on the same synthetic streams, all host cores
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_binding as ob
        cores = os.cpu_count() or 1
        builds = {}
        for name, native in (("O2", False), ("O3_march_native", True)):
            if ob.bench_lib(native) is None:
                continue
            ob.bench_imdct_ola(spectra, flags, ch, 256, 2048, cores, native)
            nn, ss, _ = ob.bench_imdct_ola(spectra, flags, ch, 256, 2048, cores, native)
            assert nn == samples_rank, (nn, samples_rank)
            builds[name] = nn / ss
        if builds:
            best = max(builds, key=lambda k: builds[k])
            cpu = {"value": builds[best], "unit": UNIT, "cores": cores, "kind": "port", "build": best, "builds": builds,
                   "sample": "all 65,536 blocks: Mdct.Reverse + OverlapBuffers + interleaved clipped store, one stream per thread"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warm,
        "ms_per_step": k3_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic spectra (seeded)",
        "config": {"workload": "config3: kernel-only IMDCT+window+OLA, 65,536 stereo blocks per GPU "
                               "(64 streams x 1,024 blocks, %s)" % ("all n=2048 (the all-long variant)" if args.all_long else
                                                                     "n=2048 long runs with n=256 short transitions"),
                   "channel_samples_per_gpu": int(samples_rank), "short_block_fraction": float(1.0 - flags.mean()),
                   "l2": "inputs larger than L2: %.2f GB spectra + %.2f GB PCM per step vs 126 MB L2"
                         % (4.0 * samples_rank / 1e9, 4.0 * samples_rank / 1e9)},
        "clocks": clk, "gpu_launches": int(launches),
        "roofline": {"kernel": "vpz_k3_streams", "bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s",
                     "frac": a / peak, "traffic": load_traffic().get("config3:vpz_k3_streams"), "peak_source": peak_src,
                     "ms_per_launch": k3_ms, "algorithmic_bytes_per_launch": 8.0 * samples_rank},
    }
    if cpu:
        line["cpu_baseline"] = cpu
        line["vs_cpu_baseline"] = value / cpu["value"]
    return line


def run_config5(args, ctx, rank, world, barrier, max_over_ranks, sum_over_ranks, local_rank, with_cpu=True):
    """BASELINE config 5: random-access batch -- 16,384 short excerpts per GPU, each = SeekTo(start) + read
    4,096 samples per channel on one of {2test, 3test, issue6test} (SURVEY 8(d): rng(0x5EED0005), start
    uniform in [0, total - 4096)), through the host API vpz_decode_excerpts (host Ogg images in, host
    PCM out: provider side of SeekTo on the host, windows of many excerpts in one GPU batch, D2H).
    Excerpts shard over the ranks like streams do: every rank takes its own 16,384, no collective."""
    lib = ctx.lib
    files = load_files()[1:]
    chans = [1, 2, 2]
    file_of, start, count, nread = config5_excerpts(rank, world, args.scaling)
    n = int(file_of.size)
    keep = [np.frombuffer(f, np.uint8) for f in files]
    ptrs = (C.c_void_p * len(files))(*[k.ctypes.data for k in keep])
    lens = (C.c_size_t * len(files))(*[k.size for k in keep])
    offsets = np.zeros(n, np.int64)
    got = np.zeros(n, np.int32)
    a = (ctx._h, len(files), ptrs, lens, n, file_of.ctypes.data, start.ctypes.data, count.ctypes.data, 1)
    total = ctx.check(lib.vpz_decode_excerpts(*a, None, 0, offsets.ctypes.data, got.ctypes.data))
    dst, dst_p = pinned_array(lib, total)
    clocks = ClockSampler(local_rank)
    clocks.start()
    for _ in range(max(1, min(args.warmup, 3))):
        ctx.check(lib.vpz_decode_excerpts(*a, dst.ctypes.data, dst.size, offsets.ctypes.data, got.ctypes.data))
    # issue6test.ogg's last page advertises 63 samples more than the reference can decode (SURVEY quirk Q4):
    # excerpts that reach into them come back a little short; everything delivered is counted as delivered
    assert (got >= 0).all() and (got >= nread - 64).all(), "every excerpt lies inside its file"
    total_delivered = int(sum(int(g) * chans[int(f)] for g, f in zip(got, file_of)))
    h0, d0 = lib.vpz_transfer_bytes(0), lib.vpz_transfer_bytes(1)
    launches0 = lib.vpz_ctx_kernel_launches(ctx._h)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ctx.check(lib.vpz_decode_excerpts(*a, dst.ctypes.data, dst.size, offsets.ctypes.data, got.ctypes.data))
    barrier()
    t = max_over_ranks(time.perf_counter() - t0)
    clk = clocks.stop()
    launches = lib.vpz_ctx_kernel_launches(ctx._h) - launches0
    delivered = sum_over_ranks(float(total_delivered))
    v = delivered * args.steps / t
    line = {
        "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": min(args.warmup, 3),
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic (seeded excerpts of TestFiles)",
        "config": {"workload": "config5: %s (SeekTo + %d samples per channel on "
                               "{2,3,issue6}test.ogg), host Ogg images -> host PCM through vpz_decode_excerpts" % (
                                   "%d random-access excerpts per GPU" % n if args.scaling == "weak" else
                                   "16384 random-access excerpts across %d GPU(s)" % world, nread),
                   "excerpts_per_gpu": n, "delivered_channel_samples_per_gpu": total_delivered,
                   "excerpts_per_s": sum_over_ranks(float(n)) * args.steps / t, "parallelism": "excerpt-sharded, no collective",
                   "note": "value counts the delivered samples only; every excerpt also decodes its pre-roll packet "
                           "and the unused parts of its first and last packets"},
        "clocks": clk, "gpu_launches": int(launches),
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": (lib.vpz_transfer_bytes(0) - h0) // args.steps,
                "d2h_bytes_per_step": (lib.vpz_transfer_bytes(1) - d0) // args.steps,
                "ms_per_step": 1e3 * t / args.steps, "api": "vpz_decode_excerpts"},
    }
    lib.vpz_host_free(dst_p)
    if with_cpu and rank == 0 and world == 1 and not args.no_cpu:
        # the oracle's SeekTo + read on all host cores (one open reader per thread and file), same excerpts
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_binding as ob
        cores = os.cpu_count() or 1
        allf = load_files()
        builds = {}
        for name, native in (("O2", False), ("O3_march_native", True)):
            if ob.bench_lib(native) is None:
                continue
            ob.bench_excerpts(allf[1:], file_of[:2048], start[:2048], count[:2048], cores, native)
            nn, ss = ob.bench_excerpts(allf[1:], file_of, start, count, cores, native)
            builds[name] = nn / ss
        best = max(builds, key=lambda k: builds[k])
        line["cpu_baseline"] = {"value": builds[best], "unit": UNIT, "cores": cores, "kind": "port", "build": best,
                                "builds": builds, "sample": "all %d excerpts, SeekTo + read, one open reader per (thread, file)" % n}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # one config3 step is ~0.3 ms: alone it defaults to 200 timed steps after ~0.4 s of warm-up (which also lets the
    # clock sampler collect samples under load); the config3 sub-object of the default line uses the line's counts
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 5; 200 for --workload config3)")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up steps (default 3; 1500 for --workload config3)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=4096, help="streams per GPU (weak) / in total (strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU work of the cpu_baseline sample")
    ap.add_argument("--workload", default="config4", choices=["config4", "config3", "config5", "config1"],
                    help="config4 (default, the headline): 4,096 streams full decode; config3: kernel-only "
                         "IMDCT+window+OLA on 65,536 synthetic stereo blocks; config5: 16,384 random-access "
                         "excerpts (SeekTo + 4,096 samples) per GPU through vpz_decode_excerpts; config1 (with --impl "
                         "reference): single-stream CPU decode of 1test.ogg")
    ap.add_argument("--all-long", action="store_true", help="config3 only: pure n=2048 blocks (no short transitions)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the config3 / config5 sub-objects of the default line")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="config4 only: after the timed steps, write a fixed sample of the PCM the last of them decoded "
                         "on rank 0 as DIR/*.npy (see dump_outputs)")
    ap.add_argument("--l1-bits", type=int, default=0, help=argparse.SUPPRESS)  # tuning: first-level Huffman table width
    ap.add_argument("--set", action="append", default=[], metavar="KEY=VALUE", help=argparse.SUPPRESS)  # any vpz_ctx_set tunable
    ap.add_argument("--lib", default=None, help=argparse.SUPPRESS)  # dry-run the script logic on the emulated test build
    args = ap.parse_args()
    c3 = args.impl == "ours" and args.workload == "config3"
    if args.steps is None:
        args.steps = 200 if c3 else 5
    if args.warmup is None:
        args.warmup = 1500 if c3 else 3
    if args.dump_outputs and (args.impl != "ours" or args.workload != "config4"):
        ap.error("--dump-outputs covers the default workload (--impl ours --workload config4)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    dry = args.lib is not None
    if not dry:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        if world > 1:
            # the one line rank 0 prints must be the JSON line: the "NCCL version" banner that the first
            # communicator writes to stdout goes to stderr instead
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
                dist.barrier()
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)

    def barrier():
        if dry:
            return
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    from vorbispizza_b200 import Batch, Context, SynthBatch, VorbisReader

    ctx = Context(local_rank, lib_path=args.lib)  # raises without libvpz.so / without a B200: no CPU fallback
    lib = ctx.lib
    if args.l1_bits:
        ctx.set("l1_bits", args.l1_bits)
    for kv in args.set:
        k, v = kv.split("=")
        ctx.set(k, int(v))
    # experiments (tools/gpu_r2e.sh): page scan on the host / a fixed number of host worker threads
    if os.environ.get("VPZ_BENCH_GPU_SCAN"):
        ctx.set("gpu_scan", int(os.environ["VPZ_BENCH_GPU_SCAN"]))
    if os.environ.get("VPZ_BENCH_HOST_THREADS", "0") != "0":
        ctx.set("host_threads", int(os.environ["VPZ_BENCH_HOST_THREADS"]))
        ctx.set("bulk_threads", 0)
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    if local_world > 1:
        # the ranks of one box share its host cores: split them instead of oversubscribing the bulk path's pool
        ctx.set("host_threads", max(2, min(32, (os.cpu_count() or 2) // local_world)))
    files = load_files()
    if args.workload == "config5":
        line = run_config5(args, ctx, rank, world, barrier, max_over_ranks, sum_over_ranks, local_rank)
        if rank == 0:
            print(json.dumps(line))
        ctx.close()
        if world > 1:
            dist.destroy_process_group()
        return
    if args.workload == "config3":
        line = run_config3(args, ctx, rank, world, barrier, max_over_ranks, sum_over_ranks, local_rank)
        if rank == 0:
            print(json.dumps(line))
        ctx.close()
        if world > 1:
            dist.destroy_process_group()
        return
    first_stream, n_streams = stream_assignment(args.streams, rank, world, args.scaling)

    # ---- workload: packets of every TestFile through the product's own Ogg layer -------------
    per_file = []
    for data in files:
        with VorbisReader(ctx, data) as r:
            pk = r.audio_packets()
            st = ctx.create_setup(r.header_packet(0), r.header_packet(2))
            blob = np.frombuffer(b"".join(p["data"] for p in pk), np.uint8)
            offs = np.zeros(len(pk) + 1, np.uint32)
            offs[1:] = np.cumsum([len(p["data"]) for p in pk])
            per_file.append(dict(setup=st, blob=blob, offs=offs, n=len(pk), ch=r.channels))
    batch = Batch(ctx)
    t_plan = time.perf_counter()
    n_pk = [f["n"] for f in per_file]
    n_runs = 0
    for i in range(n_streams):
        g = first_stream + i
        fi, k = stream_file_and_start(g, len(files), n_pk)
        f = per_file[fi]
        # replica r starts at audio packet (7 r) mod count; the packets before it form a second run,
        # so every packet of the file is decoded once per replica (each run re-seeds its overlap)
        n_runs = batch.add_run_raw(f["setup"], f["blob"], np.ascontiguousarray(f["offs"][k:])) + 1
        if k > 0:
            n_runs = batch.add_run_raw(f["setup"], f["blob"], np.ascontiguousarray(f["offs"][:k + 2])) + 1
    t_plan = time.perf_counter() - t_plan
    batch.upload()
    samples_rank = batch.total_floats          # one channel-sample = one fp32 PCM value
    packets_rank = batch.total_packets
    bytes_rank = batch.total_bytes

    # ---- value: device-resident, K steps back to back between two events --------------------
    clocks = ClockSampler(local_rank)
    clocks.start()   # nvidia-smi needs ~0.1 s to come up: start it before the warm-up, all samples are under load
    for _ in range(args.warmup):
        batch.decode(clip=True, sync=False)
    batch.sync()
    barrier()
    launches0 = lib.vpz_ctx_kernel_launches(ctx._h)
    t_wall = time.perf_counter()
    lib.vpz_ctx_mark(ctx._h, 0)
    for _ in range(args.steps):
        batch.decode(clip=True, sync=False)
    lib.vpz_ctx_mark(ctx._h, 1)
    ms = lib.vpz_ctx_elapsed_ms(ctx._h, 0, 1)
    batch.sync()
    barrier()
    t_wall = time.perf_counter() - t_wall
    launches = lib.vpz_ctx_kernel_launches(ctx._h) - launches0
    ms_max = max_over_ranks(ms)
    total_samples = sum_over_ranks(float(samples_rank))
    value = total_samples * args.steps / (ms_max * 1e-3)

    # ---- per-kernel durations (events around each kernel), averaged over K more steps ----------
    k1a, k1b, k3 = [], [], []
    for _ in range(args.steps):
        batch.decode(clip=True, sync=True)
        _, _, b, _ = batch.last_ms()
        a1, a2 = batch.last_ms_k1()
        k1a.append(a1)
        k1b.append(a2)
        k3.append(b)
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        # after the sampler stopped: `clocks` covers the decode steps, not the ~8 GB of copies the dump reads
        t_dump = time.perf_counter()
        dump_outputs(batch, n_runs, args.dump_outputs)
        print("dump_outputs: %d runs in %.1f s" % (n_runs, time.perf_counter() - t_dump), file=sys.stderr)
    k1a_ms, k1b_ms, k3_ms = float(np.mean(k1a)), float(np.mean(k1b)), float(np.mean(k3))
    peak, peak_src = measured_peak()
    # algorithmic bytes per launch (DESIGN.md): K1a reads the packet bytes and writes the symbol
    # record (counted as 2 B per decoded VQ entry ~ 0.34 B per channel-sample: use the packet bytes
    # in + out as the floor); K1b reads the record and writes the fp32 spectrum (4 B per
    # channel-sample); K3 reads that spectrum and writes fp32 PCM (8 B per channel-sample, SURVEY 8(d)).
    k1a_bytes = 2.0 * bytes_rank
    k1b_bytes = bytes_rank + 4.0 * samples_rank
    k3_bytes = 8.0 * samples_rank
    traffic = load_traffic()

    def roof(name, nbytes, t_ms):
        a = nbytes / (t_ms * 1e-3) / 1e9
        r = {"kernel": name, "bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak,
             "traffic": traffic.get(name), "peak_source": peak_src, "ms_per_launch": t_ms,
             "algorithmic_bytes_per_launch": nbytes}
        if traffic.get(name) and n_streams == 4096:
            # the same with the DRAM bytes ncu measured for this launch shape (profiles/traffic.json): K1b does not
            # write and K3 does not read the all-zero tail of a spectrum, so the real traffic is BELOW the
            # algorithmic figure of SURVEY 8(d) and this fraction is the lower, physical one
            r["frac_of_peak_on_dram_bytes"] = traffic[name] / (t_ms * 1e-3) / 1e9 / peak
        return r

    roof_k1a = roof("vpz_k1a_symbols", k1a_bytes, k1a_ms)
    roof_k1b = roof("vpz_k1b_spectrum", k1b_bytes, k1b_ms)
    roof_k3 = roof("vpz_k3_streams", k3_bytes, k3_ms)
    dominant = max((roof_k1a, roof_k1b, roof_k3), key=lambda r: r["ms_per_launch"])

    # ---- e2e: Ogg bytes in host memory -> PCM in pinned host memory, through vpz_decode_files ----
    e2e = None
    if not args.no_e2e:
        e_files = [files[(first_stream + i) % len(files)] for i in range(n_streams)]
        keep = [np.frombuffer(f, np.uint8) for f in e_files]
        ptrs = (C.c_void_p * n_streams)(*[k.ctypes.data for k in keep])
        lens = (C.c_size_t * n_streams)(*[k.size for k in keep])
        counts = np.zeros(n_streams, np.int64)
        # sizes: whole files emit the same samples as the two-run replicas minus the re-seeded packet
        e_total = ctx.check(lib.vpz_decode_files(ctx._h, n_streams, ptrs, lens, 1, None, 0, counts.ctypes.data))
        dst, dst_p = pinned_array(lib, e_total)   # 8.2 GB of pinned host memory per rank
        for _ in range(2):
            ctx.check(lib.vpz_decode_files(ctx._h, n_streams, ptrs, lens, 1, dst.ctypes.data, dst.size,
                                           counts.ctypes.data))
        h0, d0 = lib.vpz_transfer_bytes(0), lib.vpz_transfer_bytes(1)
        e_steps = args.steps
        barrier()
        t0 = time.perf_counter()
        for _ in range(e_steps):
            got = ctx.check(lib.vpz_decode_files(ctx._h, n_streams, ptrs, lens, 1, dst.ctypes.data, dst.size,
                                                 counts.ctypes.data))
        barrier()
        t_e2e = max_over_ranks(time.perf_counter() - t0)
        assert got == e_total
        e_samples = sum_over_ranks(float(e_total))
        e2e = {"value": e_samples * e_steps / t_e2e, "unit": UNIT,
               "h2d_bytes_per_step": (lib.vpz_transfer_bytes(0) - h0) // e_steps,
               "d2h_bytes_per_step": (lib.vpz_transfer_bytes(1) - d0) // e_steps,
               "ms_per_step": 1e3 * t_e2e / e_steps, "steps": e_steps,
               "api": "vpz_decode_files (host Ogg images -> pinned host PCM)"}
        if not dry:
            # copy-only ceiling of exactly this destination: the whole pinned PCM buffer filled once from the device in
            # the pieces the pipeline uses (512 MiB), all ranks at once -- the 1 GiB probe below re-uses one small
            # buffer, which the IOMMU / TLBs of some boxes serve faster than 8 GB of fresh pages
            import torch
            piece = 512 << 20
            src = torch.empty(piece, dtype=torch.uint8, device="cuda")
            view = torch.frombuffer((C.c_uint8 * (e_total * 4)).from_address(dst_p), dtype=torch.uint8)
            st = torch.cuda.Stream()
            with torch.cuda.stream(st):
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                for off in range(0, e_total * 4, piece):
                    n_b = min(piece, e_total * 4 - off)
                    view[off:off + n_b].copy_(src[:n_b], non_blocking=True)
                e1.record(st)
                e1.synchronize()
            t_dst = max_over_ranks(e0.elapsed_time(e1) * 1e-3)
            e2e["link_gbs_into_pcm_buffer"] = sum_over_ranks(float(e_total * 4)) / t_dst / 1e9
            del view, src
        lib.vpz_host_free(dst_p)
        # the same call with 16-bit output (SURVEY 8(f) row 4: conversion fused into the IMDCT kernel, half the
        # device-to-host bytes) -- reported beside the fp32 number, which stays the headline
        dst16 = lib.vpz_host_alloc(int(e_total) * 2)
        if dst16:
            for _ in range(2):
                ctx.check(lib.vpz_decode_files_s16(ctx._h, n_streams, ptrs, lens, 1, dst16, e_total, counts.ctypes.data))
            d1 = lib.vpz_transfer_bytes(1)
            barrier()
            t0 = time.perf_counter()
            for _ in range(e_steps):
                ctx.check(lib.vpz_decode_files_s16(ctx._h, n_streams, ptrs, lens, 1, dst16, e_total, counts.ctypes.data))
            barrier()
            t16 = max_over_ranks(time.perf_counter() - t0)
            e2e["s16"] = {"value": e_samples * e_steps / t16, "unit": UNIT, "ms_per_step": 1e3 * t16 / e_steps,
                          "d2h_bytes_per_step": (lib.vpz_transfer_bytes(1) - d1) // e_steps,
                          "api": "vpz_decode_files_s16 (16-bit PCM by the reference tests' (int)(x*32768f) rule)"}
            lib.vpz_host_free(dst16)
        if not dry:
            # what the device-to-host path of this box can carry with nothing but copies on it (all ranks at once)
            link = d2h_probe(lib, local_rank, barrier, max_over_ranks, sum_over_ranks)
            if link:
                d2h_rate = sum_over_ranks(float(e2e["d2h_bytes_per_step"])) / (e2e["ms_per_step"] * 1e-3) / 1e9
                e2e["link_gbs_measured"] = link
                e2e["d2h_gbs_in_e2e"] = d2h_rate
                e2e["frac_of_link"] = d2h_rate / link
                if e2e.get("link_gbs_into_pcm_buffer"):
                    e2e["frac_of_link_into_pcm_buffer"] = d2h_rate / e2e["link_gbs_into_pcm_buffer"]
                e2e["link_probe"] = "1 GiB device buffer -> pinned host, back to back for ~1 s, %d rank(s) at once" % world

    # ---- cpu baseline (rank 0, N=1): the oracle on all host cores, bounded sample ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_binding as ob   # the checker, timed as the reported CPU baseline only
        cores = os.cpu_count() or 1
        n0, s0 = ob.bench_decode(files, 4 * cores, cores)
        njobs = int(max(4 * cores, min(n_streams, (args.cpu_seconds / max(s0, 1e-3)) * 4 * cores)))
        njobs -= njobs % 4
        builds, wall = {}, 0.0
        for name, native in (("O2", False), ("O3_march_native", True)):
            if ob.bench_lib(native) is None:
                continue
            n1, s1 = ob.bench_decode(files, njobs, cores, native)
            builds[name] = n1 / s1
            wall += s1
        best = max(builds, key=lambda k: builds[k])
        cpu = {"value": builds[best], "unit": UNIT, "cores": cores, "kind": "port", "build": best, "builds": builds,
               "sample": "%d of the %d streams (whole files, stream g = TestFile g %% 4), streams handed to %d threads by a "
                         "shared cursor, %.1f s wall for both builds" % (njobs, n_streams, cores, wall)}

    # ---- BASELINE configs 3 and 5 as sub-objects of this line (the driver records only the default run) ------
    sub3 = sub5 = None
    if not args.no_sub and not dry:
        batch.close()
        batch = None
        args_sub = argparse.Namespace(**vars(args))
        args_sub.all_long = False
        c3 = run_config3(args_sub, ctx, rank, world, barrier, max_over_ranks, sum_over_ranks, local_rank, quick=True)
        c5 = run_config5(args_sub, ctx, rank, world, barrier, max_over_ranks, sum_over_ranks, local_rank)
        sub3 = {k: c3[k] for k in ("value", "unit", "ms_per_step", "steps", "gpu_launches", "roofline")}
        sub3["workload"] = c3["config"]["workload"]
        sub3["short_block_fraction"] = c3["config"]["short_block_fraction"]
        for k in ("cpu_baseline", "vs_cpu_baseline"):
            if k in c3:
                sub3[k] = c3[k]
        sub5 = {k: c5[k] for k in ("value", "unit", "ms_per_step", "steps", "gpu_launches", "e2e") if k in c5}
        sub5["workload"] = c5["config"]["workload"]
        sub5["excerpts_per_s"] = c5["config"]["excerpts_per_s"]
        if "cpu_baseline" in c5:
            sub5["cpu_baseline"] = c5["cpu_baseline"]
            sub5["vs_cpu_baseline"] = c5["value"] / c5["cpu_baseline"]["value"]

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic (TestFiles replicated/offset)",
            "config": {
                "workload": "config4: %d concurrent streams per GPU replicated/offset from TestFiles/{1,2,3,issue6}test.ogg, "
                            "full entropy+floor+residue+IMDCT decode, stream-sharded" % n_streams,
                "streams_per_gpu": n_streams, "packets_per_gpu": int(packets_rank),
                "compressed_bytes_per_gpu": int(bytes_rank), "channel_samples_per_gpu": int(samples_rank),
                "x_realtime": value / 44100.0, "parallelism": "stream-sharded, no collective",
                "l2": "inputs larger than L2: %.0f MB packet bytes + %.1f GB spectra per step vs 126 MB L2"
                      % (bytes_rank / 1e6, 4.0 * samples_rank / 1e9),
                "host_plan_s": t_plan,
            },
            "clocks": clk, "gpu_launches": int(launches), "wall_s_timed_region": t_wall,
            "roofline": dominant, "roofline_k1a": roof_k1a, "roofline_k1b": roof_k1b, "roofline_k3": roof_k3,
        }
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        if sub3:
            line["config3"] = sub3
        if sub5:
            line["config5"] = sub5
        print(json.dumps(line))
    if batch is not None:
        batch.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
