"""Device-output bulk calls against the host ones, in one process (one JSON line on stdout).

  files     the 4,096-stream config-4 mix of bench.py's e2e leg (whole TestFiles, stream i = file i % 4):
            vpz_decode_files (pinned fp32), vpz_decode_files_s16 (pinned int16), vpz_decode_files_device fp32
            interleaved / fp32 planar / int16 planar into a torch CUDA tensor
  excerpts  config 5's 16,384 excerpts (bench.config5_excerpts): vpz_decode_excerpts (pinned) against
            vpz_decode_excerpts_device fp32 planar
  threads   "bulk_threads_device" 4 / 8 / 0 (all) for vpz_decode_files_device fp32 planar
  k5        (--profile, run separately) K5 kernel time per call under torch.profiler, its algorithmic bytes
            (4 B read + 4 or 2 B written per channel-sample) and their rate against bench.measured_peak()

Every call returns with its output complete, so a host clock around it is the call's time.  The GPU's name and
power limit are part of the line.  --trace: one extra call of each device variant with VPZ_TRACE set (the host
time breakdown goes to stderr).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from vorbispizza_b200 import Context  # noqa: E402
from vorbispizza_b200 import _native as N  # noqa: E402


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the number is still reported, without its power limit
        limit = "unknown (%s)" % e
    return name, limit


def timed(fn, warmup, steps):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        t = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t) * 1e3)
    return {"ms_mean": float(np.mean(ts)), "ms_min": float(np.min(ts)), "ms_max": float(np.max(ts))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--profile", action="store_true", help="K5 alone under torch.profiler (no timing legs)")
    ap.add_argument("--trace", action="store_true", help="one VPZ_TRACE call of each device variant")
    ap.add_argument("--no-excerpts", action="store_true")
    ap.add_argument("--no-threads", action="store_true")
    args = ap.parse_args()
    import torch

    gpu, power_limit = gpu_identity()
    ctx = Context(0)
    lib = ctx.lib
    files = bench.load_files()
    n = args.streams
    e_files = [files[i % len(files)] for i in range(n)]
    keep = [np.frombuffer(f, np.uint8) for f in e_files]
    ptrs = (C.c_void_p * n)(*[k.ctypes.data for k in keep])
    lens = (C.c_size_t * n)(*[k.size for k in keep])
    counts = np.zeros(n, np.int64)
    total = ctx.check(lib.vpz_decode_files(ctx._h, n, ptrs, lens, 1, None, 0, counts.ctypes.data))
    dev32 = torch.empty(total, dtype=torch.float32, device="cuda:0")
    dev16 = torch.empty(total, dtype=torch.int16, device="cuda:0")
    stream = torch.cuda.current_stream().cuda_stream

    def dev_call(fmt, out):
        return lambda: ctx.check(lib.vpz_decode_files_device(ctx._h, n, ptrs, lens, 1, fmt, out.data_ptr(), total,
                                                             counts.ctypes.data, stream))

    variants = {
        "device_fp32_interleaved": (0, dev32),
        "device_fp32_planar": (N.VPZ_OUT_PLANAR, dev32),
        "device_s16_planar": (N.VPZ_OUT_PLANAR | N.VPZ_OUT_S16, dev16),
    }
    line = {"tool": "device_out_bench", "gpu": gpu, "power_limit": power_limit, "streams": n,
            "channel_samples_per_call": int(total), "warmup": args.warmup, "steps": args.steps}

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        k5 = {}
        peak, peak_src = bench.measured_peak()
        for name, (fmt, out) in variants.items():
            fn = dev_call(fmt, out)
            for _ in range(args.warmup):
                fn()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.steps):
                    fn()
                torch.cuda.synchronize()
            us = sum(e.device_time_total for e in prof.key_averages() if "vpz_k5_place" in e.key)
            launches = sum(e.count for e in prof.key_averages() if "vpz_k5_place" in e.key)
            ms = us / 1e3 / args.steps
            nbytes = float(total) * (4 + (2 if fmt & N.VPZ_OUT_S16 else 4))
            gbs = nbytes / (ms * 1e-3) / 1e9 if ms > 0 else None
            k5[name] = {"k5_ms_per_call": ms, "k5_launches_per_call": launches / args.steps,
                        "algorithmic_bytes_per_call": nbytes, "achieved_gbs": gbs,
                        "frac_of_peak": gbs / peak if gbs else None}
        line.update({"k5": k5, "peak_gbs": peak, "peak_source": peak_src})
        print(json.dumps(line))
        ctx.close()
        return

    # ---- files ---------------------------------------------------------------------------------------------------
    host32, host32_p = bench.pinned_array(lib, total)
    p16 = lib.vpz_host_alloc(int(total) * 2)
    host16 = np.ctypeslib.as_array(C.cast(p16, C.POINTER(C.c_int16)), shape=(int(total),))
    legs = {
        "host_fp32": lambda: ctx.check(lib.vpz_decode_files(ctx._h, n, ptrs, lens, 1, host32.ctypes.data, total,
                                                            counts.ctypes.data)),
        "host_s16": lambda: ctx.check(lib.vpz_decode_files_s16(ctx._h, n, ptrs, lens, 1, host16.ctypes.data, total,
                                                               counts.ctypes.data)),
    }
    for name, (fmt, out) in variants.items():
        legs[name] = dev_call(fmt, out)
    res = {}
    for name, fn in legs.items():
        r = timed(fn, args.warmup, args.steps)
        r["g_channel_samples_per_s"] = total / (r["ms_mean"] * 1e-3) / 1e9
        res[name] = r
    # the outputs agree: device interleaved fp32 == host fp32, bitwise
    legs["device_fp32_interleaved"]()
    torch.cuda.synchronize()
    line["device_equals_host_fp32"] = bool(torch.equal(dev32.view(torch.int32).cpu(),
                                                       torch.from_numpy(host32.view(np.int32))))
    line["files"] = res
    if args.trace:
        os.environ["VPZ_TRACE"] = "1"
        for name in ("host_fp32", *variants):
            print("trace %s:" % name, file=sys.stderr, flush=True)
            legs[name]()
        del os.environ["VPZ_TRACE"]
    del host32, host16
    lib.vpz_host_free(host32_p)
    lib.vpz_host_free(p16)

    # ---- bulk_threads_device ----------------------------------------------------------------------------------------
    if not args.no_threads:
        th = {}
        for k in (4, 8, 0):
            ctx.set("bulk_threads_device", k)
            th[str(k) if k else "all"] = timed(dev_call(N.VPZ_OUT_PLANAR, dev32), args.warmup, args.steps)
        line["bulk_threads_device_fp32_planar"] = th
        ctx.close()
        ctx = Context(0)
        lib = ctx.lib
    del dev32, dev16
    torch.cuda.empty_cache()

    # ---- excerpts -------------------------------------------------------------------------------------------------
    if not args.no_excerpts:
        xf = files[1:]
        file_of, start, count, _ = bench.config5_excerpts(0)
        m = int(file_of.size)
        xkeep = [np.frombuffer(f, np.uint8) for f in xf]
        xptrs = (C.c_void_p * len(xf))(*[k.ctypes.data for k in xkeep])
        xlens = (C.c_size_t * len(xf))(*[k.size for k in xkeep])
        offsets = np.zeros(m, np.int64)
        got = np.zeros(m, np.int32)
        a = (ctx._h, len(xf), xptrs, xlens, m, file_of.ctypes.data, start.ctypes.data, count.ctypes.data, 1)
        xtotal = ctx.check(lib.vpz_decode_excerpts(*a, None, 0, offsets.ctypes.data, got.ctypes.data))
        xhost, xhost_p = bench.pinned_array(lib, xtotal)
        xdev = torch.empty(xtotal, dtype=torch.float32, device="cuda:0")
        xs = {
            "host_fp32": timed(lambda: ctx.check(lib.vpz_decode_excerpts(*a, xhost.ctypes.data, xtotal, offsets.ctypes.data,
                                                                         got.ctypes.data)), args.warmup, args.steps),
            "device_fp32_planar": timed(lambda: ctx.check(lib.vpz_decode_excerpts_device(
                *a, N.VPZ_OUT_PLANAR, xdev.data_ptr(), xtotal, offsets.ctypes.data, got.ctypes.data, stream)),
                args.warmup, args.steps),
        }
        for r in xs.values():
            r["g_channel_samples_per_s"] = xtotal / (r["ms_mean"] * 1e-3) / 1e9
        if args.trace:
            os.environ["VPZ_TRACE"] = "1"
            ctx.check(lib.vpz_decode_excerpts_device(*a, N.VPZ_OUT_PLANAR, xdev.data_ptr(), xtotal, offsets.ctypes.data,
                                                     got.ctypes.data, stream))
            del os.environ["VPZ_TRACE"]
        line["excerpts"] = dict(xs, n=m, channel_samples_per_call=int(xtotal))
        del xhost
        lib.vpz_host_free(xhost_p)
    ctx.close()
    print(json.dumps(line))


if __name__ == "__main__":
    main()
