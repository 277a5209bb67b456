"""K6 (vpz_k6_convert) at the edges of its input space, against torchaudio.functional.resample itself.

test_device_convert.py checks the conversion at ordinary rate pairs against a float64 restatement of the filter.
This file checks the contract as documented, `torchaudio.functional.resample(x, fi, fo)` with its defaults, where
the kernel's paths change: one output per tile (thousands of taps), phase tables of tens of thousands of rows up to
the 2^22-float limit, x384 upsampling, 3..8 channels kept or mixed, excerpts much shorter than the filter, and on
the GPU a launch of many more tiles than CTAs, so that every CTA restages its shared memory for tiles of different
spans and mix modes.

Reference: x is the host call's fp32 PCM (mono-mixed with mono() for one output channel), resampled in float64.
Every output gets its own tolerance, K_TOL * 2^-24 * (sqrt(taps) + 2) * sum_i |c_i x_i| over the output's taps: the
rounding of an fp32 dot product of `taps` terms, of the fp32 coefficients and of the fp32 result (taps = 2 width + 2,
the ones K6 reads).  Each case also
proves that its check can fail: the reference of the input shifted by one source sample must differ from the true
one by at least 10x the tolerance somewhere (a one-sample indexing error would be caught).  Synth streams, whose PCM
is broadband, provide the channel counts the TestFiles do not have and the content where that margin needs it.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torchaudio.functional as AF

import synthvorbis
from conftest import load_file
from test_corpus import corpus_vs_plain
from test_device_convert import (as_numpy, conv_files, emu_out, gpu_out, is_sentinel, item, mono, relabel, stream_info,
                                 to_s16, window_of)
from vorbispizza_b200 import Context, Corpus, decode_excerpts, decode_excerpts_device, decode_files
from vorbispizza_b200 import _native as N

K_TOL = 2.0                      # errors measured up to 0.44 of the tolerance (emulated library)
DIRECT_KERNEL_BYTES = 256 << 20  # torchaudio's own call where its [n, 2 width + o] float64 kernel fits
BLOCK_ELEMS = 1 << 22            # kernel elements per block of the blocked evaluation


# ---- the reference: torchaudio.functional.resample -----------------------------------------------------------------
def pair(fi, fo):
    """(o, n, width) as torchaudio derives them: fi / fo = o / n in lowest terms."""
    g = math.gcd(fi, fo)
    o, n = fi // g, fo // g
    return o, n, math.ceil(6 * o / (min(o, n) * 0.99))


def ta_rows(o, n, width, p0, p1, c0, c1):
    """Rows p0..p1-1, columns c0..c1-1 of torchaudio's kernel (_get_sinc_resample_kernel, float64), with its
    operations in its order, so the elements are torchaudio's."""
    base = min(o, n) * 0.99
    idx = torch.arange(-width + c0, -width + c1, dtype=torch.float64)[None] / o
    t = torch.arange(-p0, -p1, -1, dtype=torch.float64)[:, None] / n + idx
    t *= base
    t = t.clamp_(-6, 6)
    window = torch.cos(t * math.pi / 6 / 2) ** 2
    t *= math.pi
    k = torch.where(t == 0, torch.tensor(1.0).to(t), t.sin() / t)
    k *= window * (base / o)
    return k.numpy()


def blocked(xs, o, n, width, n_out, block_elems=BLOCK_ELEMS):
    """torchaudio's resample of each [T, C] float64 array of xs, a block of phases at a time, and sum_i |c_i x_i| of
    xs[0].  Per block only the columns where some row's t is inside (-6, 6) are evaluated: outside them torchaudio's
    kernel is the clamped value, below 1e-32.  This is how pairs with tens of thousands of phases (a 15 GB kernel for
    44,100 -> 44,101) are evaluated; test_blocked_reference_is_torchaudio pins it to the call itself."""
    T = xs[0].shape[0]
    L = 2 * width + o
    K = -(-n_out // n)                              # conv positions (stride o) torchaudio's output uses
    X = np.concatenate(xs + [np.abs(xs[0])], axis=1)
    xp = np.zeros((K * o + L, X.shape[1]))            # torchaudio pads (width, width + o); K o >= T
    xp[width:width + T] = X
    out = np.zeros((K, n, X.shape[1]))
    nx = X.shape[1] - xs[0].shape[1]
    rows = max(1, block_elems // L)
    for p0 in range(0, min(n, n_out), rows):
        p1 = min(n, p0 + rows)
        # row p is nonzero where |column - width - o p / n| < 6 o / base <= width
        c0 = (o * p0) // n
        c1 = min(L, -(-o * (p1 - 1) // n) + 2 * width + 1)
        k = ta_rows(o, n, width, p0, p1, c0, c1)
        W = np.lib.stride_tricks.sliding_window_view(xp[c0:], (c1 - c0), axis=0)[::o][:K]   # [K, C, c1 - c0]
        out[:, p0:p1, :nx] = np.einsum("kcl,pl->kpc", W[:, :nx], k)
        out[:, p0:p1, nx:] = np.einsum("kcl,pl->kpc", W[:, nx:], np.abs(k))
    y = out.reshape(K * n, -1)[:n_out]
    return y[:, :nx], y[:, nx:]


def reference(x, fi, fo):
    """(torchaudio's resample of x [T, C], of x shifted by one source sample, the tolerance) as [n_out, C] float64."""
    x = np.asarray(x, np.float64)
    xs = np.concatenate([np.zeros((1, x.shape[1])), x[:-1]])
    o, n, width = pair(fi, fo)
    n_out = -(-len(x) * fo // fi)
    if n * (2 * width + o) * 8 <= DIRECT_KERNEL_BYTES:
        ta = [AF.resample(torch.from_numpy(np.ascontiguousarray(v.T)), fi, fo).numpy().T for v in (x, xs)]
        _, s_abs = blocked([x], o, n, width, n_out)
    else:
        both, s_abs = blocked([x, xs], o, n, width, n_out)
        ta = [both[:, :x.shape[1]], both[:, x.shape[1]:]]
    # (+ 1e-30: torchaudio's taps at the clamp |t| = 6 are ~1e-49, not 0, so silence resamples to ~1e-59, not 0)
    tol = K_TOL * 2.0 ** -24 * (math.sqrt(2 * width + 2) + 2) * s_abs + 1e-30
    return ta[0], ta[1], tol


def assert_ta(got, y, tol, what):
    """got [m, C'] within tol of y [m, C] (C' = 2 from mono: both channels)."""
    assert got.shape[0] == y.shape[0], (what, got.shape, y.shape)
    if got.shape[1] != y.shape[1]:
        y, tol = np.repeat(y, got.shape[1], 1), np.repeat(tol, got.shape[1], 1)
    err = np.abs(got.astype(np.float64) - y)
    bad = err > tol
    if got.size:
        print("%s: largest error / tolerance %.3g" % (what, float((err / np.maximum(tol, 1e-300)).max())))
    assert not bad.any(), "%s: %d outputs outside the tolerance, first at %s: got %r, want %r +- %.3g" % (
        what, int(bad.sum()), np.argwhere(bad)[0], got[tuple(np.argwhere(bad)[0])], y[tuple(np.argwhere(bad)[0])],
        tol[tuple(np.argwhere(bad)[0])])


def assert_can_fail(y, y_shift, tol, what):
    assert (np.abs(y_shift - y) >= 10 * tol).any(), "%s: a one-sample shift stays within 10x the tolerance" % what


def source(pcm, channels):
    return mono(pcm) if channels == 1 and pcm.shape[1] > 1 else pcm


# ---- the tile plan (conv_plan in reader.cpp) ------------------------------------------------------------------------
def plan(fi, fo, C_, cout):
    """(outputs per tile, staged floats of the largest tile) of a C_-channel stream converted to fo / cout."""
    per_frame = C_ + 1 if cout == 1 and C_ > 1 else C_
    budget = 32768 // 4 // per_frame
    if fi == fo:
        m = min(4096, budget)
        return m, m * per_frame
    o, n, width = pair(fi, fo)
    fixed = 2 * width + 3
    m = min(4096, (budget - fixed) * n // o + 1) if budget > fixed else 1
    span = lambda m: ((n - 1) + (m - 1) * o) // n + 2 * width + 2   # noqa: E731
    while m > 1 and span(m) > budget:
        m -= 1
    return m, span(m) * per_frame


# ---- inputs ---------------------------------------------------------------------------------------------------------
SYNTH = {3: "res012_3ch", 4: "res0_4ch", 5: dict(channels=5, res_types=(1,), coupling=4),
         6: "ch6_coupled", 7: dict(channels=7, res_types=(1,), coupling=6), 8: "ch8"}


def synth(C_, n_packets=60):
    d = synthvorbis.make_stream(0x5EED0E00 + C_, SYNTH[C_], n_packets=n_packets)["ogg"]
    assert stream_info([d])[0][0] == C_
    return d


def stereo():
    return load_file("3test")[:40000]    # the first pages of 3test: 85,952 samples


# ---- files ----------------------------------------------------------------------------------------------------------
def check_files_ta(ctx, datas, make_out, rate, channels, planar=True, dtype="float32"):
    """The conv call (sentinel checks in conv_files), every converted item against torchaudio; returns the items."""
    items, srcs, info = conv_files(ctx, datas, make_out, rate, channels, planar, dtype)
    for k, (g, s, (_, fi)) in enumerate(zip(items, srcs, info)):
        x = source(s, channels)
        what = "file %d (%d ch, %d -> %d Hz, channels=%d)" % (k, s.shape[1], fi, rate, channels)
        if fi == rate:
            e = np.repeat(x, g.shape[1] // x.shape[1], 1)
            assert np.array_equal(g.view(np.uint32), e.view(np.uint32)), what
            continue
        y, y_shift, tol = reference(x, fi, rate)
        assert_can_fail(y, y_shift, tol, what)
        assert_ta(g, y, tol, what)
    return items


# ---- excerpts -------------------------------------------------------------------------------------------------------
def edge_excerpts(n_outs, widths, counts):
    """Per file: starts 0, 1, in the last `width` outputs, at and past the end (the seek still succeeds), far past it
    (the seek fails), each with every count."""
    file_of, start, count = [], [], []
    for f, (n_out, w) in enumerate(zip(n_outs, widths)):
        for s in sorted({0, 1, n_out // 2, max(0, n_out - w), max(0, n_out - 3), max(0, n_out - 1), n_out, n_out + 2,
                         10 ** 7}):
            for c in counts:
                file_of.append(f)
                start.append(s)
                count.append(c)
    return np.array(file_of, np.uint32), np.array(start, np.int64), np.array(count, np.int32)


def check_excerpts_ta(ctx, datas, make_out, rate, channels, counts=(1, 7), planar=True):
    """One conv excerpt call over all files (a mixed-rate batch when their rates differ), every excerpt against the
    slice [start, start + got) of torchaudio's output for the whole file, after checking that the plain call's
    source window is bitwise that slice of the whole decode.  Returns got."""
    info = stream_info(datas)
    full, counts_full = decode_files(ctx, datas)
    offs = np.concatenate([[0], np.cumsum(counts_full * np.array([c for c, _ in info]))])
    pcm = [full[offs[f]:offs[f + 1]].reshape(-1, info[f][0]) for f in range(len(datas))]
    refs = [reference(source(p, channels), fi, rate) for p, (_, fi) in zip(pcm, info)]
    n_outs = [r[0].shape[0] for r in refs]
    for f, (y, y_shift, tol) in enumerate(refs):
        assert_can_fail(y, y_shift, tol, "file %d" % f)
    file_of, start, count = edge_excerpts(n_outs, [pair(fi, rate)[2] for _, fi in info], counts)
    cout = [channels or c for c, _ in info]
    total = int(sum(int(count[i]) * cout[file_of[i]] for i in range(file_of.size)))
    out = make_out(total, "float32", 16)
    _, offsets, got = decode_excerpts_device(ctx, datas, file_of, start, count, planar=planar, out=out[:total],
                                             sample_rate=rate, channels=channels)
    buf = as_numpy(out)
    assert not is_sentinel(buf[:total]).any(), "an element of the destination was not written"
    assert is_sentinel(buf[total:]).all(), "an element behind the destination was written"
    wins = [window_of(int(start[i]), int(count[i]), info[file_of[i]][1], rate) for i in range(file_of.size)]
    w_start = np.array([w[0] for w in wins], np.int64)
    src, s_off, s_got = decode_excerpts(ctx, datas, file_of, w_start, np.array([w[1] - w[0] for w in wins], np.int32))
    for i in range(file_of.size):
        f = int(file_of[i])
        C_, fi = info[f]
        what = "excerpt %d (file %d, %d -> %d Hz, start %d, count %d)" % (i, f, fi, rate, start[i], count[i])
        g = item(buf, offsets[i], count[i], cout[f], planar)
        if s_got[i] < 0:
            assert got[i] == s_got[i] and not g.any(), what
            continue
        # the plain call's window is the whole decode's samples (a reader that seeks into the last packet delivers it
        # untrimmed: the conversion sees zeros from the file's end on, so only the part inside the file counts)
        lo = int(w_start[i])
        inside = max(0, min(int(s_got[i]), pcm[f].shape[0] - lo))
        assert np.array_equal(src[s_off[i]:s_off[i] + inside * C_].view(np.uint32),
                              pcm[f][lo:lo + inside].ravel().view(np.uint32)), what + ": the source window"
        y, _, tol = refs[f]
        want = y[int(start[i]):int(start[i]) + int(count[i])]
        assert got[i] == want.shape[0], (what, got[i], want.shape[0])
        assert_ta(g[:got[i]], want, tol[int(start[i]):int(start[i]) + int(got[i])], what)
        assert not g[got[i]:].any(), what + ": samples past got are not zero"
    return got


# ---- the reference itself -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fi,fo", [(44100, 16000), (384000, 1000), (1000, 384000), (4410, 4411), (4411, 4410)])
def test_blocked_reference_is_torchaudio(fi, fo):
    """The blocked evaluation (small blocks: many of them) against torchaudio's call, where the call fits."""
    rng = np.random.default_rng(fi + fo)
    x = rng.standard_normal((3000, 2))
    o, n, width = pair(fi, fo)
    ta = AF.resample(torch.from_numpy(np.ascontiguousarray(x.T)), fi, fo).numpy().T
    y, s_abs = blocked([x], o, n, width, ta.shape[0], block_elems=40000)
    assert y.shape == ta.shape
    assert np.abs(y - ta).max() <= 1e-13 * max(1.0, s_abs.max())
    assert (s_abs >= np.abs(ta) - 1e-12).all()


def test_plan_rule():
    """The paths the cases below rely on: one output per tile, the table limit, the shared-memory refusal."""
    assert plan(384000, 1000, 2, 2) == (1, 4658 * 2)
    assert plan(384000, 1000, 8, 1) == (1, 4658 * 9)          # 164 KB
    assert plan(192000, 1000, 6, 1)[0] == 1                   # 64 KB
    assert plan(1000000, 1000, 2, 2) == (1, 12124 * 2)        # 95 KB
    assert plan(1000000, 1000, 8, 1)[1] * 4 > 227 * 1024      # refused
    o, n, width = pair(1001, 262144)
    assert n * (2 * width + 2) == 1 << 22
    o, n, width = pair(1001, 262146)
    assert n * (2 * width + 2) > 1 << 22


# ---- CPU: the emulated library --------------------------------------------------------------------------------------
EXTREME = [  # (source data, source rate, output rate, output channels)
    ("stereo", 384000, 1000, 0),
    ("synth8", 384000, 1000, 1),
    ("synth6", 192000, 1000, 1),
    ("stereo", 1000000, 1000, 0),
    ("1test", 1000, 384000, 0),
    ("1test", 1000, 384000, 2),
    ("1test", 44100, 44101, 0),
    ("1test", 44101, 44100, 0),
    ("1test", 1001, 262144, 0),
    ("stereo", 48000, 44100, 0),
    ("synth3", 11025, 16000, 0),
    ("stereo", 22050, 44100, 1),
    ("synth5", 44100, 1000, 0),
]


def data_of(name):
    return {"stereo": stereo, "1test": lambda: load_file("1test")}.get(name, lambda: synth(int(name[5:])))()


@pytest.mark.parametrize("name,fi,fo,channels", EXTREME)
def test_emu_files(emu_ctx, name, fi, fo, channels):
    check_files_ta(emu_ctx, [relabel(data_of(name), fi)], emu_out, fo, channels, planar=fi % 2 == 0)


@pytest.mark.parametrize("C_", [3, 4, 5, 7, 8])
@pytest.mark.parametrize("planar", [False, True])
def test_emu_channels_kept(emu_ctx, C_, planar):
    check_files_ta(emu_ctx, [relabel(synth(C_), 48000)], emu_out, 16000, 0, planar)


@pytest.mark.parametrize("C_", [3, 5, 7])
def test_emu_mono_mix(emu_ctx, C_):
    d = synth(C_)
    items, srcs, _ = conv_files(emu_ctx, [d], emu_out, 0, 1, planar=True)
    assert np.array_equal(items[0].view(np.uint32), mono(srcs[0]).view(np.uint32))
    check_files_ta(emu_ctx, [d], emu_out, 16000, 1, planar=False)


@pytest.mark.parametrize("planar", [False, True])
def test_emu_s16_is_the_rule_on_fp32(emu_ctx, planar):
    datas = [relabel(synth(5), 22050)]
    a, _, _ = conv_files(emu_ctx, datas, emu_out, 16000, 0, planar, "float32")
    b, _, _ = conv_files(emu_ctx, datas, emu_out, 16000, 0, planar, "int16")
    assert np.array_equal(to_s16(a[0]), b[0])


def test_emu_table_limit(emu_ctx):
    buf = np.zeros(1 << 20, np.float32)
    table_limit_checks(emu_ctx, buf.ctypes.data, buf.size)


EXCERPT_BATCHES = [  # (sources (data, rate), output rate, output channels)
    ([("stereo", 384000), ("synth8", 384000), ("synth6", 192000), ("1test", 1000000)], 1000, 1),
    ([("stereo", 1000000), ("1test", 384000), ("stereo", 44100)], 1000, 0),
    ([("1test", 1000), ("1test", 4000)], 384000, 2),
    ([("1test", 44101), ("stereo", 48000), ("synth3", 11025)], 44100, 0),
    ([("1test", 44100)], 44101, 1),
    ([("1test", 1001)], 262144, 0),
]


@pytest.mark.parametrize("batch", range(len(EXCERPT_BATCHES)))
def test_emu_excerpts(emu_ctx, batch):
    srcs, rate, channels = EXCERPT_BATCHES[batch]
    datas = [relabel(data_of(name), fi) for name, fi in srcs]
    got = check_excerpts_ta(emu_ctx, datas, emu_out, rate, channels, planar=batch % 2 == 0)
    assert (got < 0).any() and (got == 0).any() and ((got > 0) & (got < 7)).any()


def test_emu_excerpt_end_is_the_files_slice(emu_ctx):
    end_checks(emu_ctx, emu_out)


@pytest.mark.parametrize("fi,fo", [(384000, 1000), (1000, 384000)])
def test_emu_corpus(emu_ctx, fi, fo):
    corpus_checks(emu_ctx, fi, fo, emu_out)


def test_emu_refusal_and_recovery(emu_ctx, emu_lib_path):
    refusal_checks(emu_ctx, lambda: Context(0, lib_path=emu_lib_path), emu_out, lambda a: a.ctypes.data)


# ---- shared by both libraries ---------------------------------------------------------------------------------------
def table_limit_checks(ctx, buf_ptr, buf_elems):
    """1,001 -> 262,144 Hz (a table of exactly 2^22 floats) is planned; 1,001 -> 262,146 is refused, from the size
    query as from the call."""
    d = relabel(load_file("1test"), 1001)
    keep = np.frombuffer(d, np.uint8)
    ptrs, lens = (C.c_void_p * 1)(keep.ctypes.data), (C.c_size_t * 1)(keep.size)
    lib, h = ctx.lib, ctx._h
    _, samples = decode_files(ctx, [d])
    ok = N.OutConv(0, 262144, 0)
    assert lib.vpz_decode_files_device_conv(h, 1, ptrs, lens, 1, C.byref(ok), None, 0, None, None,
                                            None) == -(-int(samples[0]) * 262144 // 1001)
    bad = N.OutConv(0, 262146, 0)
    fo, st, co = np.zeros(1, np.uint32), np.zeros(1, np.int64), np.full(1, 100, np.int32)
    for p, elems in ((None, 0), (buf_ptr, buf_elems)):
        assert lib.vpz_decode_files_device_conv(h, 1, ptrs, lens, 1, C.byref(bad), p, elems, None, None,
                                                None) == N.VPZ_E_UNSUPPORTED
        assert lib.vpz_decode_excerpts_device_conv(h, 1, ptrs, lens, 1, fo.ctypes.data, st.ctypes.data, co.ctypes.data,
                                                   1, C.byref(bad), p, elems, None, None, None) == N.VPZ_E_UNSUPPORTED


def end_checks(ctx, make_out):
    """Resampled excerpts that start in a file's last packet, where the reader delivers the packet untrimmed (past
    TotalSamples): the filter sees zeros there as in the files call, so every excerpt is bitwise its slice of the
    converted file and got stops at the file's end, wherever the excerpt starts."""
    for d, rate, channels in ((load_file("1test"), 16000, 0), (stereo(), 22050, 1)):
        whole = conv_files(ctx, [d], make_out, rate, channels, planar=False)[0][0]
        n_out = whole.shape[0]
        start = np.array([n_out - 700, n_out - 200, n_out - 9, n_out - 1, n_out], np.int64)
        count = np.full(start.size, 600, np.int32)
        file_of = np.zeros(start.size, np.uint32)
        total = int(count.sum()) * whole.shape[1]
        out = make_out(total, "float32")
        _, offsets, got = decode_excerpts_device(ctx, [d], file_of, start, count, planar=False, out=out,
                                                 sample_rate=rate, channels=channels)
        buf = as_numpy(out)
        for i in range(start.size):
            want = whole[start[i]:start[i] + count[i]]
            g = item(buf, offsets[i], count[i], whole.shape[1], False)
            assert got[i] == want.shape[0], (i, got[i], want.shape[0])
            assert np.array_equal(g[:got[i]].view(np.uint32), want.view(np.uint32)), i
            assert not g[got[i]:].any(), i


def corpus_checks(ctx, fi, fo, make_out):
    """Corpus.excerpts (K7 gathering, then K6) bitwise the plain device call at an extreme pair."""
    datas = [relabel(stereo(), fi), relabel(load_file("1test"), fi)]
    with Corpus(ctx, datas) as c:
        n_outs = [-(-int(t) * fo // fi) for t in c.samples]
        for channels in (0, 1):
            file_of, start, count = edge_excerpts(n_outs, [pair(fi, fo)[2]] * 2, (1, 7, 300))
            got = corpus_vs_plain(ctx, c, datas, file_of, start, count, make_out, "%d -> %d" % (fi, fo),
                                  sample_rate=fo, channels=channels)
            assert (got > 0).any()


def refusal_checks(ctx, fresh_ctx, make_out, ptr_of):
    """8 channels labelled 1,000,000 Hz to 1 kHz mono: one output's tile needs 12,124 taps x 9 staged floats (436 KB)
    of shared memory.  The size query and the call fail with VPZ_E_UNSUPPORTED, the destination keeps its sentinel,
    and the same context then converts like a fresh one."""
    d = relabel(synth(8), 1000000)
    keep = np.frombuffer(d, np.uint8)
    ptrs, lens = (C.c_void_p * 1)(keep.ctypes.data), (C.c_size_t * 1)(keep.size)
    lib, h = ctx.lib, ctx._h
    conv = N.OutConv(0, 1000, 1)
    out = make_out(4096, "float32")
    fo, st, co = np.zeros(3, np.uint32), np.array([0, 5, 10], np.int64), np.full(3, 1000, np.int32)
    for p, elems in ((None, 0), (ptr_of(out), 4096)):
        assert lib.vpz_decode_files_device_conv(h, 1, ptrs, lens, 1, C.byref(conv), p, elems, None, None,
                                                None) == N.VPZ_E_UNSUPPORTED
        assert b"shared memory" in lib.vpz_last_error(h)
        assert lib.vpz_decode_excerpts_device_conv(h, 1, ptrs, lens, 3, fo.ctypes.data, st.ctypes.data, co.ctypes.data,
                                                   1, C.byref(conv), p, elems, None, None, None) == N.VPZ_E_UNSUPPORTED
    assert is_sentinel(as_numpy(out)).all(), "a refused call wrote into the destination"
    datas = [relabel(synth(8), 384000), relabel(stereo(), 1000000)]
    a = conv_files(ctx, datas, make_out, 1000, 1, planar=False)[0]
    f = fresh_ctx()
    try:
        b = conv_files(f, datas, make_out, 1000, 1, planar=False)[0]
    finally:
        f.close()
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))


# ---- GPU: the product library, torch CUDA tensors -------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,fi,fo,channels", EXTREME)
def test_files(gpu_ctx, name, fi, fo, channels):
    check_files_ta(gpu_ctx, [relabel(data_of(name), fi)], gpu_out, fo, channels, planar=fi % 2 == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("planar", [False, True])
def test_channels(gpu_ctx, planar):
    for C_ in (3, 4, 5, 7, 8):
        check_files_ta(gpu_ctx, [relabel(synth(C_), 48000)], gpu_out, 16000, 0, planar)
    for C_ in (3, 5, 7):
        items, srcs, _ = conv_files(gpu_ctx, [synth(C_)], gpu_out, 0, 1, planar)
        assert np.array_equal(items[0].view(np.uint32), mono(srcs[0]).view(np.uint32))
        check_files_ta(gpu_ctx, [synth(C_)], gpu_out, 16000, 1, planar)
    datas = [relabel(synth(5), 22050)]
    a, _, _ = conv_files(gpu_ctx, datas, gpu_out, 16000, 0, planar, "float32")
    b, _, _ = conv_files(gpu_ctx, datas, gpu_out, 16000, 0, planar, "int16")
    assert np.array_equal(to_s16(a[0]), b[0])


@pytest.mark.gpu
@pytest.mark.parametrize("batch", range(len(EXCERPT_BATCHES)))
def test_excerpts(gpu_ctx, batch):
    srcs, rate, channels = EXCERPT_BATCHES[batch]
    datas = [relabel(data_of(name), fi) for name, fi in srcs]
    got = check_excerpts_ta(gpu_ctx, datas, gpu_out, rate, channels, planar=batch % 2 == 0)
    assert (got < 0).any() and (got == 0).any() and ((got > 0) & (got < 7)).any()


@pytest.mark.gpu
def test_tile_grid(gpu_ctx):
    """One launch of far more tiles than K6 has CTAs (8 per SM): whole files at 384 kHz (one output per tile, 4,658
    taps) and at 44.1 kHz (50 outputs per tile), mono kept and stereo mixed, all to 1 kHz mono.  Every CTA converts
    several tiles of different spans and mix modes in turn; each item must be bitwise what a one-item call writes."""
    names = ["3test", "issue6test", "2test", "3test", "issue6test"]
    rates = [384000, 384000, 384000, 44100, 44100]
    datas = [relabel(load_file(nm), r) for nm, r in zip(names, rates)]
    info = stream_info(datas)
    _, counts = decode_files(gpu_ctx, datas)
    tiles = sum(-(-(-(-int(t) * 1000 // fi)) // plan(fi, 1000, c, 1)[0]) for t, (c, fi) in zip(counts, info))
    assert tiles > 8 * torch.cuda.get_device_properties(0).multi_processor_count, tiles
    print("K6 tiles in one launch: %d (SMs: %d)" % (tiles, torch.cuda.get_device_properties(0).multi_processor_count))
    for planar in (False, True):
        items = check_files_ta(gpu_ctx, datas, gpu_out, 1000, 1, planar)
        for k, d in enumerate(datas):
            alone = conv_files(gpu_ctx, [d], gpu_out, 1000, 1, planar)[0][0]
            assert np.array_equal(items[k].view(np.uint32), alone.view(np.uint32)), k


@pytest.mark.gpu
def test_excerpt_end_is_the_files_slice(gpu_ctx):
    end_checks(gpu_ctx, gpu_out)


@pytest.mark.gpu
@pytest.mark.parametrize("fi,fo", [(384000, 1000), (1000, 384000)])
def test_corpus(gpu_ctx, fi, fo):
    corpus_checks(gpu_ctx, fi, fo, gpu_out)


@pytest.mark.gpu
def test_table_limit(gpu_ctx):
    buf = torch.zeros(1 << 20, dtype=torch.float32, device="cuda:0")
    table_limit_checks(gpu_ctx, buf.data_ptr(), buf.numel())


@pytest.mark.gpu
def test_refusal_and_recovery(gpu_ctx):
    refusal_checks(gpu_ctx, lambda: Context(0), gpu_out, lambda t: t.data_ptr())

