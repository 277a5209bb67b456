"""Rate / channel conversion on the device (K6) against the plain device calls, in one process (one JSON line).

  files     the 4,096-stream config-4 mix (whole TestFiles, stream i = file i % 4, 44.1 kHz):
            vpz_decode_files_device fp32 planar against vpz_decode_files_device_conv to 16 kHz mono fp32 planar,
            16 kHz mono int16 planar, 48 kHz stereo fp32 planar (upsampling: the most taps per output) and the
            identity conversion (must equal the plain call bitwise); a mixed-rate variant relabels a quarter of the
            streams each as 48 / 22.05 / 8 kHz and converts all of them to 16 kHz mono
  excerpts  config 5's 16,384 excerpts as 4,096 output samples at 16 kHz mono (start scaled to 16 kHz) against the
            plain device call of the same duration at 44.1 kHz (count 11,290)
  k6        (--profile, run separately) K6 kernel time per call under torch.profiler, its algorithmic bytes (source
            fp32 read + output written), their rate against bench.measured_peak(), and FMAs per second

The legs are timed in alternating rounds, so drift on a shared machine hits all of them alike.  Every call returns
with its output complete, so a host clock around it is the call's time.  The GPU's name and power limit are part of
the line.
"""
import argparse
import ctypes as C
import json
import math
import os
import struct
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from device_out_bench import gpu_identity  # noqa: E402
from vorbispizza_b200 import Context  # noqa: E402
from vorbispizza_b200 import _native as N  # noqa: E402

PLANAR = N.VPZ_OUT_PLANAR


def relabel(data, rate):
    """The container image with its identification header's sample rate rewritten (first page's CRC redone)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oggmux
    b = bytearray(data)
    i = b.find(b"\x01vorbis")
    b[i + 12:i + 16] = struct.pack("<I", rate)
    end = 27 + b[26] + sum(b[27:27 + b[26]])
    b[22:26] = b"\0\0\0\0"
    b[22:26] = struct.pack("<I", oggmux.crc32_ogg(bytes(b[:end])))
    return bytes(b)


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


def taps(fi, fo):
    g = math.gcd(fi, fo)
    o, n = fi // g, fo // g
    return 2 * math.ceil(6 * o / (0.99 * min(o, n))) + 2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--profile", action="store_true", help="K6 alone under torch.profiler (no timing legs)")
    args = ap.parse_args()
    import torch

    gpu, power_limit = gpu_identity()
    ctx = Context(0)
    lib = ctx.lib
    files = bench.load_files()
    n = args.streams
    stream = torch.cuda.current_stream().cuda_stream

    def file_set(datas):
        keep = [np.frombuffer(f, np.uint8) for f in datas]
        return keep, (C.c_void_p * n)(*[k.ctypes.data for k in keep]), (C.c_size_t * n)(*[k.size for k in keep])

    same = file_set([files[i % len(files)] for i in range(n)])
    relabelled = {r: [relabel(f, r) for f in files] for r in (48000, 22050, 8000)}
    mixed_rates = [44100, 48000, 22050, 8000]
    mixed = file_set([files[i % len(files)] if i * 4 // n == 0 else relabelled[mixed_rates[i * 4 // n]][i % len(files)]
                      for i in range(n)])
    counts = np.zeros(n, np.int64)

    def size(fs, conv):
        if conv is None:
            return ctx.check(lib.vpz_decode_files_device(ctx._h, n, fs[1], fs[2], 1, PLANAR, None, 0, counts.ctypes.data, None))
        return ctx.check(lib.vpz_decode_files_device_conv(ctx._h, n, fs[1], fs[2], 1, C.byref(conv), None, 0,
                                                          counts.ctypes.data, None, None))

    variants = {   # name: (file set, conversion or None, source channel-samples of the set)
        "plain_fp32_planar": (same, None),
        "conv_16k_mono_fp32_planar": (same, N.OutConv(PLANAR, 16000, 1)),
        "conv_16k_mono_s16_planar": (same, N.OutConv(PLANAR | N.VPZ_OUT_S16, 16000, 1)),
        "conv_48k_stereo_fp32_planar": (same, N.OutConv(PLANAR, 48000, 2)),
        "conv_identity_fp32_planar": (same, N.OutConv(PLANAR, 0, 0)),
        "mixed_rate_to_16k_mono_fp32_planar": (mixed, N.OutConv(PLANAR, 16000, 1)),
    }
    src_total = size(same, None)
    outs, calls, meta = {}, {}, {}
    for name, (fs, conv) in variants.items():
        total = size(fs, conv)
        s16 = conv is not None and conv.format & N.VPZ_OUT_S16
        out = torch.empty(total, dtype=torch.int16 if s16 else torch.float32, device="cuda:0")
        outs[name] = out
        meta[name] = {"elements": int(total), "bytes_written": int(total) * (2 if s16 else 4)}
        if conv is None:
            calls[name] = (lambda fs=fs, out=out, total=total: ctx.check(lib.vpz_decode_files_device(
                ctx._h, n, fs[1], fs[2], 1, PLANAR, out.data_ptr(), total, counts.ctypes.data, stream)))
        else:
            calls[name] = (lambda fs=fs, out=out, total=total, conv=conv: ctx.check(lib.vpz_decode_files_device_conv(
                ctx._h, n, fs[1], fs[2], 1, C.byref(conv), out.data_ptr(), total, counts.ctypes.data, None, stream)))
    line = {"tool": "convert_bench", "gpu": gpu, "power_limit": power_limit, "streams": n,
            "source_channel_samples_per_call": int(src_total), "warmup": args.warmup, "steps": args.steps}

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        peak, peak_src = bench.measured_peak()
        k6 = {}
        for name, fn in calls.items():
            if name.startswith("plain") or name.startswith("conv_identity"):
                continue
            for _ in range(args.warmup):
                fn()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.steps):
                    fn()
                torch.cuda.synchronize()
            ev = [e for e in prof.key_averages() if "vpz_k6_convert" in e.key or "vpz_k5_place" in e.key]
            k6_ms = sum(e.device_time_total for e in ev if "vpz_k6_convert" in e.key) / 1e3 / args.steps
            k5_ms = sum(e.device_time_total for e in ev if "vpz_k5_place" in e.key) / 1e3 / args.steps
            # bytes: every source float read once (the whole mix is converted), every output element written once
            nbytes = float(src_total) * 4 + meta[name]["bytes_written"]
            conv = variants[name][1]
            fs = variants[name][0]
            rates = [44100] * n if fs is same else [mixed_rates[i * 4 // n] for i in range(n)]
            ntaps = np.array([taps(r, conv.sample_rate) if r != conv.sample_rate else 0 for r in rates], np.float64)
            size(fs, conv)
            fmas = float((counts * ntaps * conv.channels).sum())
            gbs = nbytes / (k6_ms * 1e-3) / 1e9 if k6_ms > 0 else None
            k6[name] = {"k6_ms_per_call": k6_ms, "k5_ms_per_call": k5_ms, "algorithmic_bytes_per_call": nbytes,
                        "achieved_gbs": gbs, "frac_of_peak": gbs / peak if gbs else None, "fmas_per_call": fmas,
                        "gfma_per_s": fmas / (k6_ms * 1e-3) / 1e9 if k6_ms > 0 else None}
        line.update({"k6": k6, "peak_gbs": peak, "peak_source": peak_src})
        print(json.dumps(line))
        ctx.close()
        return

    res = rounds(calls, args.warmup, args.steps)
    for name in res:
        res[name].update(meta[name])
    calls["plain_fp32_planar"]()
    calls["conv_identity_fp32_planar"]()
    torch.cuda.synchronize()
    line["identity_equals_plain"] = bool(torch.equal(outs["plain_fp32_planar"].view(torch.int32),
                                                     outs["conv_identity_fp32_planar"].view(torch.int32)))
    line["files"] = res
    del outs
    torch.cuda.empty_cache()

    # ---- excerpts: 4,096 samples at 16 kHz mono against 11,290 at 44.1 kHz ------------------------------------------
    xf = files[1:]
    file_of, start, _, _ = bench.config5_excerpts(0)
    m = int(file_of.size)
    xkeep = [np.frombuffer(f, np.uint8) for f in xf]
    xptrs = (C.c_void_p * len(xf))(*[k.ctypes.data for k in xkeep])
    xlens = (C.c_size_t * len(xf))(*[k.size for k in xkeep])
    offsets, got = np.zeros(m, np.int64), np.zeros(m, np.int32)
    p_count = np.full(m, 11290, np.int32)
    c_start = (start * 16000 // 44100).astype(np.int64)
    c_count = np.full(m, 4096, np.int32)
    conv = N.OutConv(PLANAR, 16000, 1)
    pa = (ctx._h, len(xf), xptrs, xlens, m, file_of.ctypes.data, start.ctypes.data, p_count.ctypes.data, 1)
    ca = (ctx._h, len(xf), xptrs, xlens, m, file_of.ctypes.data, c_start.ctypes.data, c_count.ctypes.data, 1)
    p_total = ctx.check(lib.vpz_decode_excerpts_device(*pa, PLANAR, None, 0, None, None, None))
    c_total = ctx.check(lib.vpz_decode_excerpts_device_conv(*ca, C.byref(conv), None, 0, None, None, None))
    p_out = torch.empty(p_total, dtype=torch.float32, device="cuda:0")
    c_out = torch.empty(c_total, dtype=torch.float32, device="cuda:0")
    xs = rounds({
        "plain_fp32_planar_11290_at_44k": lambda: ctx.check(lib.vpz_decode_excerpts_device(
            *pa, PLANAR, p_out.data_ptr(), p_total, offsets.ctypes.data, got.ctypes.data, stream)),
        "conv_16k_mono_fp32_planar_4096": lambda: ctx.check(lib.vpz_decode_excerpts_device_conv(
            *ca, C.byref(conv), c_out.data_ptr(), c_total, offsets.ctypes.data, got.ctypes.data, stream)),
    }, args.warmup, args.steps)
    line["excerpts"] = dict(xs, n=m, full_items=int((got == 4096).sum()))
    ctx.close()
    print(json.dumps(line))


if __name__ == "__main__":
    main()
