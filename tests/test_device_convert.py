"""Rate and channel conversion on the way into device memory: vpz_decode_files_device_conv /
vpz_decode_excerpts_device_conv (K6).

Unconverted items and the equal-rate channel mix are checked bitwise against the host calls.  Resampled items are
checked against a float64 restatement of torchaudio.functional.resample's default filter (sinc_interp_hann, width 6,
rolloff 0.99) applied to the host calls' fp32 output; the restatement itself is checked against properties that do
not depend on it (DC gain, passband amplitude, stopband rejection).  The TestFiles are 44.1 kHz; relabel() rewrites
the rate field of the identification header (decoding does not depend on it), so they also serve as 8 / 22.05 / 48 /
96 kHz files.  `-m gpu` runs the product library with torch CUDA tensors, the CPU suite the emulated library with
numpy destinations.
"""
import ctypes as C
import math
import struct

import numpy as np
import pytest

import cases
import oggmux
import oracle_binding as ob
import synthvorbis
from conftest import FILES, load_file
from vorbispizza_b200 import Context, decode_excerpts, decode_excerpts_device, decode_files, decode_files_device
from vorbispizza_b200 import _native as N

FORMATS = [(planar, dtype) for planar in (False, True) for dtype in ("float32", "int16")]
TOL = 2e-6   # fp32 accumulation of fp32 taps against the float64 filter, full-scale signals


# ---- helpers ------------------------------------------------------------------------------------------------------
def relabel(data, rate):
    """The container image with the identification header's sample rate set to `rate` (first page's CRC redone)."""
    b = bytearray(data)
    i = b.find(b"\x01vorbis")
    b[i + 12:i + 16] = struct.pack("<I", rate)
    nseg = b[26]
    end = 27 + nseg + sum(b[27:27 + nseg])
    b[22:26] = b"\0\0\0\0"
    b[22:26] = struct.pack("<I", oggmux.crc32_ogg(bytes(b[:end])))
    return bytes(b)


def filt(fi, fo):
    g = math.gcd(fi, fo)
    o, n = fi // g, fo // g
    base = 0.99 * min(o, n)
    return o, n, base, math.ceil(6 * o / base)


def resample_ref(x, k0, fi, fo, js):
    """Outputs js (absolute, fo) of the closed form over source samples x[:, c] at absolute k0, k0 + 1, ... (zero
    elsewhere), in float64: y[j] = (base/fi) sum_k x[k] sinc(t) cos^2(pi t / 12), t = clamp(base (k/fi - j/fo), -6, 6)."""
    x = np.asarray(x, np.float64).reshape(len(x), -1)
    o, n, base, width = filt(fi, fo)
    out = np.zeros((len(js), x.shape[1]))
    taps = np.arange(2 * width + 2)
    for a in range(0, len(js), 1 << 15):
        j = np.asarray(js[a:a + (1 << 15)], np.int64)
        k = (j * o // n)[:, None] - width + taps[None, :]
        t = base * ((taps[None, :] - width) / o - ((j * o) % n)[:, None] / (o * n))   # = base (k / o - j / n)
        t = np.clip(t, -6, 6)
        coef = base / o * np.sinc(t) * np.cos(t * np.pi / 12) ** 2
        idx = k - k0
        ok = (idx >= 0) & (idx < len(x))
        xk = np.where(ok[:, :, None], x[np.clip(idx, 0, max(len(x) - 1, 0))], 0.0)
        out[a:a + len(j)] = np.einsum("lt,ltc->lc", coef, xk)
    return out


def window_of(start, count, fi, fo):
    if fi == fo:
        return start, start + count
    o, n, _, width = filt(fi, fo)
    lo = max(0, start * o // n - width)
    return lo, max(lo, (start + count - 1) * o // n + width + 1)


def mono(x):
    """[T, C] float32 -> [T, 1]: channels added in order, then / C, in float32."""
    s = x[:, 0].astype(np.float32)
    for c in range(1, x.shape[1]):
        s = (s + x[:, c]).astype(np.float32)
    return (s / np.float32(x.shape[1])).astype(np.float32)[:, None]


def to_s16(x):
    v = np.trunc(x.astype(np.float32) * np.float32(32768.0)).astype(np.int64)
    return np.clip(v, -32768, 32767).astype(np.int16)


def as_numpy(buf):
    return buf if isinstance(buf, np.ndarray) else buf.cpu().numpy()


def emu_out(total, dtype, extra=0):
    return np.full(total + extra, np.nan if dtype == "float32" else 0x7777, dtype)


def gpu_out(total, dtype, extra=0):
    import torch
    return torch.full((total + extra,), np.nan if dtype == "float32" else 0x7777, dtype=getattr(torch, dtype), device="cuda:0")


def is_sentinel(a):
    return np.isnan(a) if a.dtype == np.float32 else a == 0x7777


def item(buf, off, n, ch, planar):
    """[n, ch] view of one item of a flat result."""
    g = buf[int(off):int(off) + int(n) * ch]
    return np.ascontiguousarray(g.reshape(ch, -1).T if planar else g.reshape(-1, ch))


def stream_info(datas):
    out = []
    for d in datas:
        i = d.find(b"\x01vorbis")
        out.append((d[i + 11], struct.unpack("<I", d[i + 12:i + 16])[0]))
    return out


def conv_files(ctx, datas, make_out, rate, channels, planar=True, dtype="float32", clip=True, extra=16):
    """The conv call into a sentinel-filled buffer: every element written, nothing behind it.  Returns the items."""
    info = stream_info(datas)
    ref, counts = decode_files(ctx, datas, clip=clip)
    cout = [channels or c for c, _ in info]
    lens = [-(-int(k) * (rate or fi) // fi) for k, (_, fi) in zip(counts, info)]
    total = int(sum(l * c for l, c in zip(lens, cout)))
    out = make_out(total, dtype, extra)
    buf, offsets, got_counts = decode_files_device(ctx, datas, clip=clip, dtype=dtype, planar=planar, out=out[:total],
                                                   sample_rate=rate, channels=channels)
    assert list(got_counts) == lens
    assert list(offsets) == list(np.concatenate([[0], np.cumsum(np.array(lens) * np.array(cout))[:-1]]).astype(np.int64))
    full = as_numpy(out)
    assert not is_sentinel(full[:total]).any(), "an element of the destination was not written"
    assert is_sentinel(full[total:]).all(), "an element behind the destination was written"
    host_off = np.concatenate([[0], np.cumsum(counts * np.array([c for c, _ in info]))[:-1]])
    items = [item(full, offsets[k], lens[k], cout[k], planar) for k in range(len(datas))]
    srcs = [ref[host_off[k]:host_off[k] + counts[k] * info[k][0]].reshape(-1, info[k][0]) for k in range(len(datas))]
    return items, srcs, info


def expected(src, fi, rate, channels, k0=0, js=None):
    """The conversion of source samples src ([T, C] fp32 at absolute k0) by the closed form, float64."""
    x = src
    if channels == 1 and x.shape[1] > 1:
        x = mono(x)
    fo = rate or fi
    if fo == fi:
        y = x.astype(np.float64)
    else:
        y = resample_ref(x, k0, fi, fo, js if js is not None else np.arange(-(-len(src) * fo // fi)))
    if channels == 2 and y.shape[1] == 1:
        y = np.repeat(y, 2, axis=1)
    return y


def check_files(ctx, datas, make_out, rate, channels, planar=True):
    items, srcs, info = conv_files(ctx, datas, make_out, rate, channels, planar)
    for k, (g, s, (_, fi)) in enumerate(zip(items, srcs, info)):
        e = expected(s, fi, rate, channels)
        assert g.shape == e.shape, (k, g.shape, e.shape)
        if (rate or fi) == fi:
            assert np.array_equal(g.view(np.uint32), e.astype(np.float32).view(np.uint32)), "file %d" % k
        else:
            err = float(np.abs(g - e).max()) if g.size else 0.0
            assert err <= TOL, "file %d (%d -> %d Hz): max abs err %.3g" % (k, fi, rate, err)
    return items


def excerpt_lists(totals, n_out_totals, n_excerpts, nread, seed):
    rng = np.random.default_rng(seed)
    file_of = list(rng.integers(0, len(totals), n_excerpts))
    start = [int(rng.integers(0, max(1, n_out_totals[f] - 1))) for f in file_of]
    for f in range(len(totals)):
        for p in (0, 1, -1, -3, -nread // 2, 10 ** 7):
            file_of.append(f)
            start.append(p if p >= 0 else max(0, n_out_totals[f] + p))
    return np.array(file_of, np.uint32), np.array(start, np.int64), np.full(len(file_of), nread, np.int32)


def check_excerpts(ctx, datas, make_out, rate, channels, n_excerpts, nread, seed, planar=True, dtype="float32", clip=True):
    info = stream_info(datas)
    totals = [ob.OracleStream(d).decode_all()[0].shape[0] for d in datas]
    out_totals = [-(-t * (rate or fi) // fi) for t, (_, fi) in zip(totals, info)]
    file_of, start, count = excerpt_lists(totals, out_totals, n_excerpts, nread, seed)
    cout = [channels or c for c, _ in info]
    total = int(sum(count[i] * cout[file_of[i]] for i in range(file_of.size)))
    out = make_out(total, dtype, 16)
    buf, offsets, got = decode_excerpts_device(ctx, datas, file_of, start, count, clip=clip, dtype=dtype, planar=planar,
                                               out=out[:total], sample_rate=rate, channels=channels)
    full = as_numpy(out)
    assert not is_sentinel(full[:total]).any(), "an element of the destination was not written"
    assert is_sentinel(full[total:]).all(), "an element behind the destination was written"
    # the source windows through the plain call
    wins = [window_of(int(start[i]), int(count[i]), info[file_of[i]][1], rate or info[file_of[i]][1]) for i in range(file_of.size)]
    w_start = np.array([w[0] for w in wins], np.int64)
    w_count = np.array([w[1] - w[0] for w in wins], np.int32)
    src, s_off, s_got = decode_excerpts(ctx, datas, file_of, w_start, w_count, clip=clip)
    for i in range(file_of.size):
        f = int(file_of[i])
        C_, fi = info[f]
        fo = rate or fi
        g = item(full, offsets[i], count[i], cout[f], planar)
        if s_got[i] < 0:
            assert got[i] == s_got[i], i
            assert not g.any()
            continue
        o, n, _, _ = filt(fi, fo)
        # resampled: the filter sees zeros from the file's end on (a reader that seeks into the last packet delivers
        # it untrimmed)
        have = int(s_got[i]) if fo == fi else max(0, min(int(s_got[i]), totals[f] - int(w_start[i])))
        e_end = int(w_start[i]) + have
        want_got = min(max(-(-e_end * n // o) - int(start[i]), 0), int(count[i]))
        assert got[i] == want_got, (i, got[i], want_got)
        assert not g[want_got:].any(), "excerpt %d: samples past got are not zero" % i
        x = src[s_off[i]:s_off[i] + have * C_].reshape(-1, C_)
        e = expected(x, fi, rate, channels, k0=int(w_start[i]), js=np.arange(int(start[i]), int(start[i]) + want_got))
        if dtype == "int16":
            continue
        if fo == fi:
            assert np.array_equal(g[:want_got].view(np.uint32), e[:want_got].astype(np.float32).view(np.uint32)), i
        elif want_got:
            err = float(np.abs(g[:want_got] - e).max())
            assert err <= TOL, "excerpt %d: max abs err %.3g" % (i, err)
    return full[:total], offsets, got, file_of, start, count


# ---- the float64 restatement against properties that do not depend on it ------------------------------------------
@pytest.mark.parametrize("fi,fo", [(44100, 16000), (48000, 44100), (22050, 16000), (8000, 16000), (44100, 48000)])
def test_reference_filter_properties(fi, fo):
    T = 3 * fi // 10
    k = np.arange(T)
    mid = np.arange(fo // 10, 2 * fo // 10)
    dc = resample_ref(np.ones(T), 0, fi, fo, mid)[:, 0]
    assert np.abs(dc - 1).max() <= 1e-3
    tone = resample_ref(np.sin(2 * np.pi * 1000 * k / fi), 0, fi, fo, mid)[:, 0]
    assert abs(np.abs(tone).max() - 1) <= 2e-3
    if 0.75 * fo < fi / 2:
        stop = resample_ref(np.sin(2 * np.pi * 0.75 * fo * k / fi), 0, fi, fo, mid)[:, 0]
        assert 20 * np.log10(np.abs(stop).max()) <= -40


def test_relabel_keeps_the_samples():
    d = load_file("1test")
    for r in (8000, 96000):
        s = ob.OracleStream(relabel(d, r))
        assert s.sample_rate == r
        assert np.array_equal(s.decode_all()[0], ob.OracleStream(d).decode_all()[0])


# ---- CPU: the emulated library ---------------------------------------------------------------------------------
def emu_datas():
    return [load_file("1test"), load_file("3test")[:40000]]


@pytest.mark.parametrize("planar,dtype", FORMATS)
def test_emu_identity_is_bitwise(emu_ctx, planar, dtype):
    datas = emu_datas()
    for rate, channels in ((0, 0), (44100, None)):
        _, counts = decode_files(emu_ctx, datas)
        total = int(sum(counts * np.array([c for c, _ in stream_info(datas)])))
        plain, p_off, p_counts = decode_files_device(emu_ctx, datas, dtype=dtype, planar=planar, out=emu_out(total, dtype))
        conv, c_off, c_counts = decode_files_device(emu_ctx, datas, dtype=dtype, planar=planar, out=emu_out(total, dtype),
                                                    sample_rate=rate, channels=channels)
        assert np.array_equal(p_off, c_off) and np.array_equal(p_counts, c_counts)
        assert np.array_equal(plain.view(np.uint8), conv.view(np.uint8))
        fo, st, co = np.array([0, 1, 1, 0], np.uint32), np.array([0, 700, 10 ** 7, 5000], np.int64), np.full(4, 900, np.int32)
        p, po, pg = decode_excerpts_device(emu_ctx, datas, fo, st, co, dtype=dtype, planar=planar,
                                           out=emu_out(900 * 7, dtype))
        c, co_, cg = decode_excerpts_device(emu_ctx, datas, fo, st, co, dtype=dtype, planar=planar,
                                            out=emu_out(900 * 7, dtype), sample_rate=rate, channels=channels)
        assert np.array_equal(po, co_) and np.array_equal(pg, cg)
        assert np.array_equal(p.view(np.uint8), c.view(np.uint8))


@pytest.mark.parametrize("planar", [False, True])
def test_emu_mix_at_equal_rate_is_bitwise(emu_ctx, planar):
    datas = emu_datas()
    check_files(emu_ctx, datas, emu_out, 0, 1, planar)        # stereo -> (L + R) / 2
    check_files(emu_ctx, datas, emu_out, 44100, 2, planar)    # mono -> duplicated
    check_excerpts(emu_ctx, datas, emu_out, 0, 1, 4, 600, 0x5EED0C01, planar)
    check_excerpts(emu_ctx, datas, emu_out, 0, 2, 4, 600, 0x5EED0C02, planar)


@pytest.mark.parametrize("rate,channels", [(16000, 1), (22050, 0), (48000, 2), (16000, 0)])
def test_emu_resampled_files(emu_ctx, rate, channels):
    datas = emu_datas() + [emu_datas()[0]]
    items = check_files(emu_ctx, datas, emu_out, rate, channels, planar=rate != 48000)
    assert np.array_equal(items[0], items[2])   # the same file twice: no bleed between runs


def test_emu_resampled_files_48k_source(emu_ctx):
    check_files(emu_ctx, [relabel(d, 48000) for d in emu_datas()], emu_out, 44100, 0, planar=False)


@pytest.mark.parametrize("rate,channels,planar", [(16000, 1, True), (48000, 0, False), (8000, 2, True)])
def test_emu_resampled_excerpts_to_file_end(emu_ctx, rate, channels, planar):
    _, _, got, _, _, count = check_excerpts(emu_ctx, emu_datas(), emu_out, rate, channels, 5, 500, 0x5EED0C03, planar)
    assert (got < 0).any() and ((got >= 0) & (got < count)).any()   # failed seeks and short reads are covered


@pytest.mark.parametrize("planar", [False, True])
def test_emu_s16_is_the_rule_on_fp32(emu_ctx, planar):
    datas = emu_datas()
    items32, _, _ = conv_files(emu_ctx, datas, emu_out, 16000, 1, planar, "float32")
    items16, _, _ = conv_files(emu_ctx, datas, emu_out, 16000, 1, planar, "int16")
    for a, b in zip(items32, items16):
        assert np.array_equal(to_s16(a), b)


def test_emu_errors_and_size_query(emu_ctx):
    conv_errors(emu_ctx, lambda n: np.zeros(n, np.float32), lambda a: a.ctypes.data)


def conv_errors(ctx, alloc, ptr_of):
    datas = [load_file("1test"), load_file("3test")]
    keep = [np.frombuffer(d, np.uint8) for d in datas]
    ptrs = (C.c_void_p * 2)(*[k.ctypes.data for k in keep])
    lens = (C.c_size_t * 2)(*[k.size for k in keep])
    lib, h = ctx.lib, ctx._h
    counts, offs = np.zeros(2, np.int64), np.zeros(2, np.int64)

    def files(conv, p, elems):
        return lib.vpz_decode_files_device_conv(h, 2, ptrs, lens, 1, C.byref(conv), p, elems, counts.ctypes.data,
                                                offs.ctypes.data, None)

    good = N.OutConv(N.VPZ_OUT_PLANAR, 16000, 1)
    total = files(good, None, 0)
    _, r_counts = decode_files(ctx, datas)
    assert list(counts) == [-(-int(c) * 16000 // 44100) for c in r_counts]
    assert total == int(counts.sum()) and list(offs) == [0, int(counts[0])]
    buf = alloc(total)
    for bad in (N.OutConv(0, 999, 0), N.OutConv(0, 384001, 0), N.OutConv(0, 16000, 3), N.OutConv(0, 16000, -1),
                N.OutConv(4, 16000, 1)):
        assert files(bad, ptr_of(buf), total) == N.VPZ_E_ARGUMENT
    assert files(good, ptr_of(buf), total - 1) == N.VPZ_E_ARGUMENT
    assert files(good, ptr_of(buf), total) == total
    six = [synthvorbis.make_stream(0x5EED0601, "ch6_coupled", n_packets=12)["ogg"]]
    k6 = np.frombuffer(six[0], np.uint8)
    p6 = (C.c_void_p * 1)(k6.ctypes.data)
    l6 = (C.c_size_t * 1)(k6.size)
    assert lib.vpz_decode_files_device_conv(h, 1, p6, l6, 1, C.byref(N.OutConv(0, 0, 2)), ptr_of(buf), total, None, None,
                                            None) == N.VPZ_E_UNSUPPORTED
    fo, st, co = np.array([0, 1], np.uint32), np.array([0, 500], np.int64), np.array([100, 300], np.int32)
    eo, got = np.zeros(2, np.int64), np.zeros(2, np.int32)
    args = (h, 2, ptrs, lens, 2, fo.ctypes.data, st.ctypes.data, co.ctypes.data, 1)
    assert lib.vpz_decode_excerpts_device_conv(*args, C.byref(good), None, 0, eo.ctypes.data, got.ctypes.data, None) == 400
    assert list(eo) == [0, 100]
    assert lib.vpz_decode_excerpts_device_conv(*args, C.byref(N.OutConv(0, 0, 2)), None, 0, eo.ctypes.data,
                                               got.ctypes.data, None) == 800
    assert lib.vpz_decode_excerpts_device_conv(*args, C.byref(good), ptr_of(buf), 399, None, None, None) == N.VPZ_E_ARGUMENT
    assert lib.vpz_decode_excerpts_device_conv(*args, C.byref(N.OutConv(0, 999, 1)), ptr_of(buf), 400, None, None,
                                               None) == N.VPZ_E_ARGUMENT
    p6b = (C.c_void_p * 1)(k6.ctypes.data)
    assert lib.vpz_decode_excerpts_device_conv(h, 1, p6b, l6, 1, fo.ctypes.data, st.ctypes.data, co.ctypes.data, 1,
                                               C.byref(N.OutConv(0, 0, 2)), ptr_of(buf), 400, None, None,
                                               None) == N.VPZ_E_UNSUPPORTED


# ---- GPU: the product library, torch CUDA tensors ----------------------------------------------------------------
RATES = [(16000, 1), (22050, 1), (48000, 0), (16000, 0), (44100, 1), (8000, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("rate,channels", RATES)
@pytest.mark.parametrize("planar", [False, True])
def test_files(gpu_ctx, rate, channels, planar):
    datas = [load_file(n) for n in FILES] + [load_file("3test")]
    items = check_files(gpu_ctx, datas, gpu_out, rate, channels, planar)
    assert np.array_equal(items[2], items[4])


@pytest.mark.gpu
def test_files_identity_is_bitwise(gpu_ctx):
    datas = [load_file(n) for n in FILES]
    _, counts = decode_files(gpu_ctx, datas)
    for planar, dtype in FORMATS:
        plain, _, _ = decode_files_device(gpu_ctx, datas, dtype=dtype, planar=planar)
        for rate, channels in ((0, 0), (44100, None)):
            conv, _, c_counts = decode_files_device(gpu_ctx, datas, dtype=dtype, planar=planar, sample_rate=rate,
                                                    channels=channels)
            assert np.array_equal(c_counts, counts)
            assert np.array_equal(as_numpy(plain).view(np.uint8), as_numpy(conv).view(np.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("planar", [False, True])
def test_files_s16_is_the_rule_on_fp32(gpu_ctx, planar):
    datas = [load_file(n) for n in FILES]
    for rate, channels in ((16000, 1), (48000, 2)):
        a, _, _ = conv_files(gpu_ctx, datas, gpu_out, rate, channels, planar, "float32")
        b, _, _ = conv_files(gpu_ctx, datas, gpu_out, rate, channels, planar, "int16")
        for x, y in zip(a, b):
            assert np.array_equal(to_s16(x), y)


@pytest.mark.gpu
def test_files_relabelled_rates(gpu_ctx):
    datas = [relabel(load_file(n), r) for n, r in (("3test", 48000), ("issue6test", 22050), ("2test", 8000),
                                                  ("1test", 96000))]
    check_files(gpu_ctx, datas, gpu_out, 44100, 0, planar=False)
    check_files(gpu_ctx, datas, gpu_out, 16000, 1, planar=True)


@pytest.mark.gpu
@pytest.mark.parametrize("force", [1, 2])
def test_files_general_paths(force):
    ctx = Context(0)
    try:
        ctx.set("force_general", force)
        check_files(ctx, [load_file(n) for n in FILES], gpu_out, 16000, 1, True)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_files_pipeline_rotation():
    """Groups of 8 streams: 64 files through all three pipeline slots several times."""
    ctx = Context(0)
    try:
        ctx.set("bulk_group", 8)
        datas = [load_file(n) for n in FILES] * 16
        items = check_files(ctx, datas, gpu_out, 16000, 1, True)
        for k in range(4, len(datas)):
            assert np.array_equal(items[k], items[k % 4])
    finally:
        ctx.close()


@pytest.mark.gpu
def test_six_channels_to_mono(gpu_ctx):
    datas = [synthvorbis.make_stream(0x5EED0601, "ch6_coupled", n_packets=60)["ogg"], load_file("3test")]
    assert [c for c, _ in stream_info(datas)] == [6, 2]
    items, srcs, info = conv_files(gpu_ctx, datas, gpu_out, 0, 1, True)
    for g, s in zip(items, srcs):
        assert np.array_equal(g.view(np.uint32), mono(s).view(np.uint32))
    items, srcs, info = conv_files(gpu_ctx, datas, gpu_out, 16000, 1, False)
    for g, s, (_, fi) in zip(items, srcs, info):
        e = expected(s, fi, 16000, 1)
        cases.assert_pcm_close_scaled(g, e.astype(np.float32), "6ch", rtol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("rate,channels", [(16000, 1), (48000, 0), (22050, 2), (44100, 1)])
def test_excerpts_to_file_end(gpu_ctx, rate, channels):
    datas = [load_file(n) for n in ["2test", "3test", "issue6test"]]
    check_excerpts(gpu_ctx, datas, gpu_out, rate, channels, 300, 4096, 0x5EED0C05, planar=True)
    _, _, got, _, _, count = check_excerpts(gpu_ctx, [load_file("1test"), load_file("3test")], gpu_out, rate, channels,
                                            64, 700, 77, planar=False)
    assert (got < 0).any() and ((got >= 0) & (got < count)).any()


@pytest.mark.gpu
def test_excerpts_s16_to_file_end(gpu_ctx):
    datas = [load_file(n) for n in ["3test", "issue6test"]]
    for planar in (False, True):
        a = check_excerpts(gpu_ctx, datas, gpu_out, 16000, 1, 40, 1000, 5, planar, "float32")[0]
        b = check_excerpts(gpu_ctx, datas, gpu_out, 16000, 1, 40, 1000, 5, planar, "int16")[0]
        assert np.array_equal(to_s16(a), b)


@pytest.mark.gpu
def test_mixed_rate_crop_batch_to_file_end(gpu_ctx):
    """Relabelled 8 / 22.05 / 44.1 / 48 / 96 kHz files to 16 kHz mono, as one [n, 1, T] batch, row by row against the
    oracle reader's SeekTo(k_lo) + Read through the float64 filter."""
    import torch
    rates = [8000, 22050, 44100, 48000, 96000]
    datas = [relabel(load_file(n), r) for n, r in zip(["3test", "issue6test", "3test", "2test", "issue6test"], rates)]
    T = 4096
    totals = [ob.OracleStream(d).decode_all()[0].shape[0] for d in datas]
    out_totals = [-(-t * 16000 // r) for t, r in zip(totals, rates)]
    file_of, start, count = excerpt_lists(totals, out_totals, 120, T, 0x5EED0C06)
    buf, offsets, got = decode_excerpts_device(gpu_ctx, datas, file_of, start, count, sample_rate=16000, channels=1)
    assert buf.is_cuda and buf.dtype == torch.float32
    batch = buf.view(file_of.size, 1, T).cpu().numpy()
    for i in range(file_of.size):
        f = int(file_of[i])
        s = ob.OracleStream(datas[f])
        C_ = s.channels
        lo, hi = window_of(int(start[i]), T, rates[f], 16000)
        try:
            s.seek(lo)
        except ob.OracleError:
            assert got[i] < 0 and not batch[i].any()
            continue
        rd = np.zeros((hi - lo) * C_, np.float32)
        n = 0
        while n < hi - lo:
            k = s.read(rd[n * C_:])
            if k <= 0:
                break
            n += k
        n = min(n, max(0, totals[f] - lo))   # the filter sees zeros from the file's end on
        o, nn, _, _ = filt(rates[f], 16000)
        want = min(max(-(-(lo + n) * nn // o) - int(start[i]), 0), T)
        assert got[i] == want, (i, got[i], want)
        e = resample_ref(mono(rd[:n * C_].reshape(-1, C_)), lo, rates[f], 16000, np.arange(int(start[i]), int(start[i]) + want))
        cases.assert_pcm_close(batch[i][0, :want][:, None], e.astype(np.float32), "crop %d" % i)
        assert not batch[i][0, want:].any()


@pytest.mark.gpu
def test_waits_for_the_callers_stream(gpu_ctx):
    import torch
    datas = [load_file(n) for n in FILES]
    ref, _, _ = decode_files_device(gpu_ctx, datas, sample_rate=16000, channels=1)
    ref = ref.cpu().numpy()
    out = torch.zeros(ref.size, dtype=torch.float32, device="cuda:0")
    a = torch.randn(4096, 4096, device="cuda:0")
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(16):
            a = a @ a
            a = a / a.norm()
        out.fill_(float("nan"))
    decode_files_device(gpu_ctx, datas, out=out, stream=side, sample_rate=16000, channels=1)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy().view(np.uint32), ref.view(np.uint32))


@pytest.mark.gpu
def test_errors_and_size_query(gpu_ctx):
    import torch
    conv_errors(gpu_ctx, lambda n: torch.empty(n, dtype=torch.float32, device="cuda:0"), lambda t: t.data_ptr())
