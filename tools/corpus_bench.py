"""Corpus calls (vpz_corpus_excerpts_device, K7) against the plain device excerpt call, in one process (one JSON line).

  A         config 5: 16,384 excerpts x 4,096 samples on {2test, 3test, issue6test} (bench.config5_excerpts), fp32
            planar; and r04's excerpt leg, 4,096 samples at 16 kHz mono (start scaled to 16 kHz)
  B-short   256 copies of 3test (6.5 s each), 16,384 x 4,096 fp32 planar excerpts drawn uniformly with Corpus.samples
  B-long    the same on 256 files of 5 minutes built from 3test's audio packets (10.8 MB each, 2.8 GB in all)
Every leg runs through the plain device call and the corpus call; their outputs, got and offsets must be bitwise
equal.  Reported per leg: the mean / min / max of the timed calls (2 warm-ups and 5 timed calls by default, the legs
in alternating rounds so drift on a shared machine hits all of them alike; every call returns with its output
complete, so a host clock around it is the call's time), the host-to-device bytes of one call (vpz_transfer_bytes),
and for B the corpus's open time and device bytes.  --trace FILE appends one VPZ_TRACE breakdown per leg and call to
FILE.  --profile (a separate run): K7's time per call under torch.profiler with the bytes it gathered.  The GPU's
name and power limit are part of the line.
"""
import argparse
import json
import os
import re
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402
from device_out_bench import gpu_identity  # noqa: E402
from vorbispizza_b200 import Context, Corpus, decode_excerpts_device  # noqa: E402

T = 4096


def rounds(legs, warmup, steps):
    for fn in legs.values():
        for _ in range(warmup):
            fn()
    ts = {k: [] for k in legs}
    for _ in range(steps):
        for k, fn in legs.items():
            t = time.perf_counter()
            fn()
            ts[k].append((time.perf_counter() - t) * 1e3)
    return {k: {"ms_mean": float(np.mean(v)), "ms_min": float(np.min(v)), "ms_max": float(np.max(v))} for k, v in ts.items()}


def traced(fn):
    """fn() with VPZ_TRACE set; returns the library's trace lines (written to fd 2)."""
    os.environ["VPZ_TRACE"] = "1"
    with tempfile.TemporaryFile(mode="w+") as f:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["VPZ_TRACE"]
        f.seek(0)
        return [ln.rstrip("\n") for ln in f if ln.startswith("vpz_")]


def uniform_excerpts(samples, n, seed):
    rng = np.random.default_rng(seed)
    file_of = rng.integers(0, samples.size, n).astype(np.uint32)
    start = np.array([int(rng.integers(0, max(1, int(samples[f]) - T))) for f in file_of], np.int64)
    return file_of, start, np.full(n, T, np.int32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--files", type=int, default=256, help="files of the B legs")
    ap.add_argument("--minutes", type=float, default=5.0, help="length of a B-long file (5 min of 3test: 10.8 MB)")
    ap.add_argument("--trace", default=None, help="append the VPZ_TRACE breakdowns to this file")
    ap.add_argument("--profile", action="store_true", help="K7 alone under torch.profiler (no timing legs)")
    args = ap.parse_args()
    import torch

    gpu, power_limit = gpu_identity()
    ctx = Context(0)
    lib = ctx.lib
    files = bench.load_files()
    line = {"tool": "corpus_bench", "gpu": gpu, "power_limit": power_limit, "warmup": args.warmup, "steps": args.steps}

    # ---- the legs: (files, file_of, start, count, conversion keywords) ------------------------------------------
    xf = files[1:]
    c5_file_of, c5_start, c5_count, _ = bench.config5_excerpts(0)
    legs = {
        "A_fp32_planar": (xf, c5_file_of, c5_start, c5_count, {}),
        "A_16k_mono_fp32_planar": (xf, c5_file_of, (c5_start * 16000 // 44100).astype(np.int64), c5_count,
                                   dict(sample_rate=16000, channels=1)),
    }
    from test_corpus import long_file
    t0 = time.perf_counter()
    long = long_file(ctx, args.minutes)
    line["b_long_file"] = {"bytes": len(long), "build_s": time.perf_counter() - t0}
    b_sets = {"B_short": [files[2]] * args.files, "B_long": [long] * args.files}

    corpora, opened = {}, {}
    corpora["A"] = Corpus(ctx, xf)
    for name, datas in b_sets.items():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        corpora[name] = Corpus(ctx, datas)
        opened[name] = {"open_ms": (time.perf_counter() - t0) * 1e3, "device_bytes": corpora[name].device_bytes,
                        "image_bytes": int(sum(len(d) for d in datas)),
                        "samples_per_file": int(corpora[name].samples[0])}
        file_of, start, count = uniform_excerpts(corpora[name].samples, 16384, 0x5EED0B00 + len(name))
        legs[name] = (datas, file_of, start, count, {})
    corpus_of = {k: corpora["A"] if k.startswith("A") else corpora[k] for k in legs}

    calls, outs = {}, {}
    for name, (datas, file_of, start, count, kw) in legs.items():
        c = corpus_of[name]
        C_out = kw.get("channels") or c.channels[file_of.astype(np.int64)]
        total = int((count.astype(np.int64) * C_out).sum())
        for kind in ("plain", "corpus"):
            out = torch.empty(total, dtype=torch.float32, device="cuda:0")
            res = {}
            outs[(name, kind)] = (out, res)
            if kind == "plain":
                fn = (lambda datas=datas, f=file_of, s=start, n=count, kw=kw, out=out, res=res:
                      res.update(r=decode_excerpts_device(ctx, datas, f, s, n, out=out, **kw)))
            else:
                fn = (lambda c=c, f=file_of, s=start, n=count, kw=kw, out=out, res=res:
                      res.update(r=c.excerpts(f, s, n, out=out, **kw)))
            calls["%s/%s" % (name, kind)] = fn

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        k7 = {}
        for key, fn in calls.items():
            if not key.endswith("/corpus"):
                continue
            for _ in range(args.warmup):
                fn()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.steps):
                    fn()
                torch.cuda.synchronize()
            ev = prof.key_averages()
            per = {e.key: e.device_time_total / 1e3 / args.steps for e in ev if e.key.startswith("vpz_") or "vpz_" in e.key}
            k7_ms = sum(v for k, v in per.items() if "vpz_k7_gather" in k)
            tr = traced(fn)
            m = re.search(r"K7 gathered (\d+) bytes in (\d+) pieces", tr[-1]) if tr else None
            nbytes, pieces = (int(m.group(1)), int(m.group(2))) if m else (None, None)
            k7[key.split("/")[0]] = {"k7_ms_per_call": k7_ms, "kernels_ms_per_call": per, "gathered_bytes": nbytes,
                                     "pieces": pieces,
                                     "gathered_gbs": nbytes / (k7_ms * 1e-3) / 1e9 if nbytes and k7_ms > 0 else None}
        line["k7"] = k7
        print(json.dumps(line))
        for c in corpora.values():
            c.close()
        ctx.close()
        return

    res = rounds(calls, args.warmup, args.steps)
    # one more call of each: output equality, host-to-device bytes, the trace breakdown
    equal, h2d, traces = {}, {}, []
    for key, fn in calls.items():
        torch.cuda.synchronize()
        b0 = lib.vpz_transfer_bytes(0)
        fn()
        h2d[key] = int(lib.vpz_transfer_bytes(0) - b0)
        traces += ["%s: %s" % (key, t) for t in traced(fn)]
    for name in legs:
        (po, pr), (co, cr) = outs[(name, "plain")], outs[(name, "corpus")]
        _, p_off, p_got = pr["r"]
        _, c_off, c_got = cr["r"]
        equal[name] = bool(torch.equal(po.view(torch.int32), co.view(torch.int32)) and np.array_equal(p_off, c_off)
                           and np.array_equal(p_got, c_got))
    for key in res:
        res[key]["h2d_bytes_per_call"] = h2d[key]
    line["legs"] = res
    line["outputs_equal"] = equal
    line["open"] = opened
    line["trace"] = traces
    mean = {k: v["ms_mean"] for k, v in res.items()}
    line["targets"] = {
        "A_fp32_corpus_le_plain": mean["A_fp32_planar/corpus"] <= mean["A_fp32_planar/plain"],
        "A_16k_corpus_le_plain": mean["A_16k_mono_fp32_planar/corpus"] <= mean["A_16k_mono_fp32_planar/plain"],
        "B_long_corpus_within_10pct_of_B_short": mean["B_long/corpus"] <= 1.10 * mean["B_short/corpus"],
        "B_long_speedup": mean["B_long/plain"] / mean["B_long/corpus"],
        "B_long_open_le_2x_plain": opened["B_long"]["open_ms"] <= 2 * mean["B_long/plain"],
    }
    if args.trace:
        with open(args.trace, "a") as f:
            f.write("# %s, %s\n" % (gpu, power_limit))
            f.write("\n".join(traces) + "\n")
    for c in corpora.values():
        c.close()
    ctx.close()
    print(json.dumps(line))


if __name__ == "__main__":
    main()
