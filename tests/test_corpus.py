"""Corpus: container images opened once, excerpt batches cut from them many times (vpz_corpus_*).

A corpus call decodes exactly what vpz_decode_excerpts_device(_conv) decodes on the same images; only the per-file
work (page scan, headers, setup tables, seek index, total samples) is done once at open.  So every case compares the
corpus call bitwise against the plain device call on the same bytes, including got, the offsets and the errors.
`-m gpu` runs the product library with torch CUDA tensors; the CPU suite runs the emulated library, whose device
memory is host memory, with numpy arrays as the destination.
"""
import ctypes as C

import numpy as np
import pytest

import cases
import oggmux
import oracle_binding as ob
from conftest import FILES, load_file
from test_container import _chained, damaged_streams
from test_device_output import EDGE_STARTS, FORMATS, as_numpy, emu_out, excerpt_lists, gpu_out
from vorbispizza_b200 import Corpus, decode_excerpts_device, scan_pages
from vorbispizza_b200 import _native as N

CONVS = [(16000, 1), (48000, 2), (None, None), (0, 0)]


def same(a, b):
    a, b = np.ascontiguousarray(as_numpy(a)), np.ascontiguousarray(as_numpy(b))
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def corpus_vs_plain(ctx, corpus, datas, file_of, start, count, make_out, what="", **kw):
    """The corpus call and the plain device call on the same excerpts into sentinel-filled buffers: bitwise equal
    buffers (nothing behind the result written), offsets and got."""
    dtype = kw.get("dtype", "float32")
    conv = {k: kw.pop(k) for k in ("sample_rate", "channels") if k in kw}
    plain_conv = conv if any(v is not None for v in conv.values()) else {}
    chans = conv.get("channels") or corpus.channels[np.asarray(file_of, np.int64)]
    total = int((np.asarray(count, np.int64) * chans).sum())
    ref, r_off, r_got = decode_excerpts_device(ctx, datas, file_of, start, count, out=make_out(total, dtype), **kw,
                                               **plain_conv)
    assert ref.shape[0] == total
    out = make_out(ref.shape[0], dtype, 16)
    buf, off, got = corpus.excerpts(file_of, start, count, out=out[:ref.shape[0]], **kw, **conv)
    assert np.array_equal(off, r_off) and np.array_equal(got, r_got), what
    full = as_numpy(out)
    assert same(full[:ref.shape[0]], ref), what
    tail = full[ref.shape[0]:]
    assert (np.isnan(tail).all() if dtype == "float32" else (tail == 0x7777).all()), what
    return r_got


def info_vs_oracle(corpus, datas):
    for i, d in enumerate(datas):
        s = ob.OracleStream(d)
        assert corpus.channels[i] == s.channels and corpus.sample_rates[i] == s.sample_rate, i
        assert corpus.samples[i] == s.total_samples, (i, corpus.samples[i], s.total_samples)


def long_file(ctx, minutes):
    """3test's audio packets with a span repeated until the stream lasts about `minutes`, granules recomputed from
    the packet geometry.  The span [a, b) is chosen so that the block sizes on both sides of the seam are those the
    packets' window flags were encoded against, so the oracle decodes it without a fault."""
    s = ob.OracleStream(load_file("3test"))
    hdr = [s.header_packet(i) for i in range(3)]
    pk = [p for p in s.audio_packets() if p["data"]]
    st = ctx.create_setup(hdr[0], hdr[2])
    size = [ctx.packet_info(st, p["data"])[1][0] for p in pk]
    ctx.release_setup(st)
    a, b = None, None
    for i in range(4, len(pk) // 3):
        for j in range(len(pk) - 4, 2 * len(pk) // 3, -1):
            if size[j - 1] == size[i - 1] and size[j] == size[i]:
                a, b = i, j
                break
        if a is not None:
            break
    assert a is not None
    span_samples = sum(size[k - 1] // 4 + size[k] // 4 for k in range(a, b))
    reps = max(1, int(minutes * 60 * s.sample_rate / span_samples))
    order = list(range(a)) + list(range(a, b)) * reps + list(range(b, len(pk)))
    out, g, prev_page, page = [], 0, None, -1
    for k, q in enumerate(order):
        if k > 0:
            g += size[order[k - 1]] // 4 + size[q] // 4
        if k == 0 or pk[q]["page_index"] != prev_page or q == a:   # every repetition gets pages of its own
            page += 1
            prev_page = pk[q]["page_index"]
        out.append(dict(data=pk[q]["data"], granule=g, page_index=page))
    return oggmux.remux(hdr, out)


def long_file_checks(ctx, data, make_out, n_oracle):
    T = 4096
    s = ob.OracleStream(data)
    total = s.total_samples
    assert total > 0
    starts = [0, 1, 1000, total // 2, total // 2 + 777, total - T, total - 100, total - 1]
    rng = np.random.default_rng(0x5EED0106)
    starts += [int(x) for x in rng.integers(0, total, 16)]
    file_of = np.zeros(len(starts), np.uint32)
    start = np.array(starts, np.int64)
    count = np.full(len(starts), T, np.int32)
    with Corpus(ctx, [data]) as c:
        assert c.samples[0] == total
        got = corpus_vs_plain(ctx, c, [data], file_of, start, count, make_out, "long", planar=False)
        buf, off, got2 = c.excerpts(file_of, start, count, planar=False, out=make_out(int(count.sum()) * s.channels, "float32"))
        assert np.array_equal(got, got2)
        buf = as_numpy(buf)
    ch = s.channels
    rd = np.zeros(T * ch, np.float32)
    for i in list(range(min(n_oracle, len(starts)))):
        o = ob.OracleStream(data)
        o.seek(int(start[i]))
        n = 0
        while n < T:
            k = o.read(rd[n * ch:])
            assert k >= 0, "oracle fault at excerpt %d" % i
            if k == 0:
                break
            n += k
        assert got[i] == n, (i, got[i], n)
        cases.assert_pcm_close(buf[off[i]:off[i] + n * ch], rd[:n * ch], "long excerpt %d" % i)


def invalid_file():
    d = bytearray(load_file("1test"))
    i = d.find(b"\x01vorbis")
    d[i:i + 7] = b"\x01xxxxxx"    # the identification header no longer is one
    return bytes(d)


def error_checks(ctx, make_out):
    lib, h = ctx.lib, ctx._h
    datas = [load_file("1test"), load_file("3test")]
    bad = [datas[0], invalid_file()]
    # open of an invalid file: the plain call's code and text
    fo, st, co = np.array([0, 1], np.uint32), np.array([0, 10], np.int64), np.array([100, 100], np.int32)
    with pytest.raises(N.VpzError) as plain:
        decode_excerpts_device(ctx, bad, fo, st, co)
    with pytest.raises(N.VpzError) as corp:
        Corpus(ctx, bad)
    assert corp.value.code == plain.value.code and str(corp.value) == str(plain.value)
    out_h = C.c_void_p()
    keep = [np.frombuffer(d, np.uint8) for d in bad]
    ptrs = (C.c_void_p * 2)(*[k.ctypes.data for k in keep])
    lens = (C.c_size_t * 2)(*[k.size for k in keep])
    assert lib.vpz_corpus_open(h, 2, ptrs, lens, 0, C.byref(out_h)) == plain.value.code and not out_h.value
    assert lib.vpz_corpus_open(None, 2, ptrs, lens, 0, C.byref(out_h)) == N.VPZ_E_ARGUMENT
    # NULL corpus
    conv = N.OutConv(0, 0, 0)
    assert lib.vpz_corpus_excerpts_device(None, 0, None, None, None, 1, C.byref(conv), None, 0, None, None, None) == N.VPZ_E_ARGUMENT
    assert lib.vpz_corpus_info(None, None, None, None) == N.VPZ_E_ARGUMENT
    lib.vpz_corpus_close(None)
    with Corpus(ctx, datas) as c:
        assert len(c) == 2 and lib.vpz_corpus_info(c._h, None, None, None) == 2
        fo, st, co = np.array([0, 1, 1], np.uint32), np.array([0, 500, 10 ** 7], np.int64), np.array([100, 300, 50], np.int32)
        offs, got = np.zeros(3, np.int64), np.zeros(3, np.int32)
        r_off = np.zeros(3, np.int64)
        # size query: the plain call's total and offsets
        r_total = lib.vpz_decode_excerpts_device(h, 2, (C.c_void_p * 2)(*[np.frombuffer(d, np.uint8).ctypes.data for d in datas]),
                                                 (C.c_size_t * 2)(*[len(d) for d in datas]), 3, fo.ctypes.data,
                                                 st.ctypes.data, co.ctypes.data, 1, 0, None, 0, r_off.ctypes.data, None, None)

        def call(fo, st, co, ptr, elems, conv=conv):
            return lib.vpz_corpus_excerpts_device(c._h, fo.size, fo.ctypes.data, st.ctypes.data, co.ctypes.data, 1,
                                                  C.byref(conv), ptr, elems, offs.ctypes.data, got.ctypes.data, None)

        assert call(fo, st, co, None, 0) == r_total == 800 and np.array_equal(offs, r_off)
        out = make_out(r_total, "float32", 0)
        ptr = out.ctypes.data if isinstance(out, np.ndarray) else out.data_ptr()
        assert call(fo, st, co, ptr, r_total - 1) == N.VPZ_E_ARGUMENT
        assert call(np.array([0, 2, 1], np.uint32), st, co, ptr, r_total) == N.VPZ_E_ARGUMENT
        assert call(fo, np.array([0, -1, 0], np.int64), co, ptr, r_total) == N.VPZ_E_ARGUMENT
        assert call(fo, st, np.array([100, -3, 50], np.int32), ptr, r_total) == N.VPZ_E_ARGUMENT
        assert call(fo, st, co, ptr, r_total, N.OutConv(4, 0, 0)) == N.VPZ_E_ARGUMENT
        assert call(fo, st, co, ptr, r_total, N.OutConv(0, 500, 0)) == N.VPZ_E_ARGUMENT
        assert call(fo, st, co, ptr, r_total) == r_total
        with pytest.raises(N.VpzError):
            c.excerpts([5], [0], [10])
    return datas


def no_state_checks(ctx, datas, make_out, n, T):
    other = [load_file("issue6test"), load_file("1test")]
    with Corpus(ctx, datas) as c, Corpus(ctx, other) as c2:
        for k, seed in enumerate((11, 12, 13)):
            file_of, start, count = excerpt_lists(datas, n, T, seed, extra_positions=(0, -1))
            corpus_vs_plain(ctx, c, datas, file_of, start, count, make_out, "call %d" % k, planar=bool(k & 1))
            f2, s2, c2n = excerpt_lists(other, n // 2, T // 2, seed + 100, extra_positions=(1,))
            corpus_vs_plain(ctx, c2, other, f2, s2, c2n, make_out, "second corpus %d" % k, sample_rate=16000, channels=1)


def copy_checks(ctx, make_out, n, T):
    orig = [load_file("3test"), load_file("1test")]
    bufs = [bytearray(d) for d in orig]
    arrs = [np.frombuffer(b, np.uint8) for b in bufs]
    file_of, start, count = excerpt_lists(orig, n, T, 0x5EED0C09, extra_positions=(0, -1))
    with Corpus(ctx, arrs, copy=True) as c:
        for a in arrs:
            a[:] = 0x55   # the caller's bytes are gone; the corpus decodes its own copy
        corpus_vs_plain(ctx, c, orig, file_of, start, count, make_out, "copy=1")


def openable(ctx, datas):
    """The files a corpus opens; a file it refuses must be refused by the plain call with the same code and text."""
    keep = []
    for d in datas:
        try:
            Corpus(ctx, [d]).close()
            keep.append(d)
        except N.VpzError as e:
            with pytest.raises(N.VpzError) as plain:   # no excerpts: the call still opens the file
                decode_excerpts_device(ctx, [d], [], [], [], out=np.zeros(0, np.float32))
            assert plain.value.code == e.code and str(plain.value) == str(e)
    return keep


def continued_pages(ctx, data):
    pages, _, _ = scan_pages(ctx, [data])[0]
    return int(pages["is_continued"].sum())


K7_TRACE = r"K7 gathered (\d+) bytes in (\d+) pieces \((\d+) packets over pages\) in (\d+) of (\d+) groups"


def gathered(ctx, corpus, datas, file_of, start, count, make_out, capfd, monkeypatch):
    """One corpus call under VPZ_TRACE (equal to the plain call): (bytes, pieces, packets over pages, groups
    gathered, groups) from its trace line."""
    import re
    corpus_vs_plain(ctx, corpus, datas, file_of, start, count, make_out, "warm")
    capfd.readouterr()
    monkeypatch.setenv("VPZ_TRACE", "1")
    corpus_vs_plain(ctx, corpus, datas, file_of, start, count, make_out, "traced")
    monkeypatch.delenv("VPZ_TRACE")
    m = [re.search(K7_TRACE, ln) for ln in capfd.readouterr().err.splitlines() if "_corpus" in ln]
    assert len(m) == 1 and m[0], "no corpus trace line"
    return tuple(int(x) for x in m[0].groups())


def dense_3test(step):
    """Excerpts of 3test every `step` samples: every packet, the 18 continued over pages included, is in one."""
    total = ob.OracleStream(load_file("3test")).total_samples
    start = np.arange(0, total, step, dtype=np.int64)
    return np.zeros(start.size, np.uint32), start, np.full(start.size, step + 64, np.int32)


def sliced_open_checks(ctx, make_out, n, T):
    """Opened in slices of 64 KiB (several device scans one after another) the corpus equals the plain call."""
    datas = [load_file(n_) for n_ in FILES] * 3
    file_of, start, count = excerpt_lists(datas, n, T, 0x5EED0C17, extra_positions=(0, -1))
    ctx.set("bulk_group_bytes", 1 << 16)
    try:
        with Corpus(ctx, datas) as c:
            assert c.device_bytes == sum((len(d) + 31) & ~15 for d in datas)
            corpus_vs_plain(ctx, c, datas, file_of, start, count, make_out, "sliced open")
    finally:
        ctx.set("bulk_group_bytes", 0)


# ---- CPU: the emulated library, numpy destinations ----------------------------------------------------------------
@pytest.fixture(scope="module")
def emu_corpus(emu_ctx):
    datas = [load_file(n) for n in FILES]
    c = Corpus(emu_ctx, datas)
    yield datas, c
    c.close()


def test_emu_info(emu_corpus):
    datas, c = emu_corpus
    info_vs_oracle(c, datas)


@pytest.mark.parametrize("planar,dtype", FORMATS)
@pytest.mark.parametrize("clip", [True, False])
def test_emu_equal_to_plain(emu_ctx, emu_corpus, planar, dtype, clip):
    datas, c = emu_corpus
    assert continued_pages(emu_ctx, datas[2]) > 0   # 3test: packets over two pages
    file_of, start, count = excerpt_lists(datas, 8, 600, 0x5EED0C01, extra_positions=EDGE_STARTS)
    got = corpus_vs_plain(emu_ctx, c, datas, file_of, start, count, emu_out, planar=planar, dtype=dtype, clip=clip)
    assert (got < 0).any() and (got < count).sum() > (got < 0).sum()   # failed seeks and short reads are covered


@pytest.mark.parametrize("rate,chans", CONVS)
def test_emu_equal_to_plain_conv(emu_ctx, emu_corpus, rate, chans):
    datas, c = emu_corpus
    file_of, start, count = excerpt_lists(datas, 6, 500, 0x5EED0C02, extra_positions=(0, 1, 1024, -1, -600, 10 ** 7))
    corpus_vs_plain(emu_ctx, c, datas, file_of, start, count, emu_out, sample_rate=rate, channels=chans)


def test_emu_damaged_and_chained(emu_ctx):
    datas = list(damaged_streams("1test").values()) + list(damaged_streams("3test", 110).values())
    datas = openable(emu_ctx, datas + [_chained(["1test", "2test"], 30)])
    assert len(datas) >= 10
    with Corpus(emu_ctx, datas) as c:
        info_vs_oracle(c, datas)
        file_of, start, count = excerpt_lists(datas, 12, 400, 0x5EED0C03, extra_positions=(0, 1, -1, -300))
        corpus_vs_plain(emu_ctx, c, datas, file_of, start, count, emu_out, clip=False)


def test_emu_no_state_between_calls(emu_ctx):
    no_state_checks(emu_ctx, [load_file("3test"), load_file("2test")], emu_out, 6, 500)


def test_emu_copy(emu_ctx):
    copy_checks(emu_ctx, emu_out, 6, 500)


def test_emu_long_file(emu_ctx):
    long_file_checks(emu_ctx, long_file(emu_ctx, 1.0), emu_out, 6)


def test_emu_errors(emu_ctx):
    error_checks(emu_ctx, emu_out)


def test_emu_k7_gathers_every_group(emu_ctx, capfd, monkeypatch):
    """K7 writes the packet bytes of every group, those of the packets continued over pages included."""
    data = [load_file("3test")]
    with Corpus(emu_ctx, data) as c:
        nbytes, pieces, multi, groups_k7, groups = gathered(emu_ctx, c, data, *dense_3test(1024), emu_out, capfd,
                                                            monkeypatch)
    assert nbytes > 0 and pieces > multi > 0 and groups_k7 == groups


def test_emu_lifetime(emu_lib_path):
    """A dropped corpus is closed; closing the context closes the corpora still open."""
    import gc
    from vorbispizza_b200 import Context
    ctx = Context(0, lib_path=emu_lib_path)
    c = Corpus(ctx, [load_file("1test")])
    assert c.device_bytes > 0 and len(ctx._corpora) == 1
    del c
    gc.collect()
    assert len(ctx._corpora) == 0
    c = Corpus(ctx, [load_file("1test")], copy=True)
    ctx.close()
    assert c._h is None and c.device_bytes == 0


def test_emu_sliced_open(emu_ctx):
    sliced_open_checks(emu_ctx, emu_out, 6, 400)


def test_emu_host_scan_and_slices(emu_lib_path):
    """gpu_scan 0 (host page scan) and open slices of 64 KiB: the same opened files, the same results."""
    from vorbispizza_b200 import Context
    datas = [load_file(n) for n in FILES] + [load_file("1test")]
    file_of, start, count = excerpt_lists(datas, 8, 500, 0x5EED0C04, extra_positions=(0, -1))
    for key, value in (("gpu_scan", 0), ("bulk_group_bytes", 1 << 16)):
        with Context(0, lib_path=emu_lib_path) as ctx:
            ctx.set(key, value)
            with Corpus(ctx, datas) as c:
                corpus_vs_plain(ctx, c, datas, file_of, start, count, emu_out, key)


# ---- GPU: the product library, torch CUDA tensors ----------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu_corpus(gpu_ctx):
    datas = [load_file(n) for n in FILES]
    c = Corpus(gpu_ctx, datas)
    yield datas, c
    c.close()


@pytest.mark.gpu
def test_info(gpu_corpus):
    datas, c = gpu_corpus
    info_vs_oracle(c, datas)


@pytest.mark.gpu
@pytest.mark.parametrize("planar,dtype", FORMATS)
@pytest.mark.parametrize("clip", [True, False])
def test_equal_to_plain(gpu_ctx, gpu_corpus, planar, dtype, clip):
    datas, c = gpu_corpus
    assert continued_pages(gpu_ctx, datas[2]) == 18
    file_of, start, count = excerpt_lists(datas, 400, 4096, 0x5EED0C11, extra_positions=EDGE_STARTS)
    got = corpus_vs_plain(gpu_ctx, c, datas, file_of, start, count, gpu_out, planar=planar, dtype=dtype, clip=clip)
    assert (got < 0).any() and (got < count).sum() > (got < 0).sum()   # failed seeks and short reads are covered


@pytest.mark.gpu
@pytest.mark.parametrize("rate,chans", CONVS)
def test_equal_to_plain_conv(gpu_ctx, gpu_corpus, rate, chans):
    datas, c = gpu_corpus
    file_of, start, count = excerpt_lists(datas, 300, 4096, 0x5EED0C12)
    for planar, dtype in FORMATS:
        corpus_vs_plain(gpu_ctx, c, datas, file_of, start, count, gpu_out, sample_rate=rate, channels=chans,
                        planar=planar, dtype=dtype)


@pytest.mark.gpu
def test_damaged_and_chained(gpu_ctx):
    datas = []
    for name in FILES:
        datas += list(damaged_streams(name).values())
    datas = openable(gpu_ctx, datas + [_chained(["1test", "3test", "2test"])])
    assert len(datas) >= 20
    with Corpus(gpu_ctx, datas) as c:
        info_vs_oracle(c, datas)
        file_of, start, count = excerpt_lists(datas, 600, 2048, 0x5EED0C13, extra_positions=(0, 1, -1, -300, 10 ** 7))
        for clip in (True, False):
            corpus_vs_plain(gpu_ctx, c, datas, file_of, start, count, gpu_out, clip=clip)


@pytest.mark.gpu
def test_no_state_between_calls(gpu_ctx):
    no_state_checks(gpu_ctx, [load_file(n) for n in ("3test", "2test", "1test")], gpu_out, 200, 4096)


@pytest.mark.gpu
def test_copy(gpu_ctx):
    copy_checks(gpu_ctx, gpu_out, 200, 4096)


@pytest.mark.gpu
def test_long_file(gpu_ctx):
    long_file_checks(gpu_ctx, long_file(gpu_ctx, 10.0), gpu_out, 8)


@pytest.mark.gpu
def test_errors(gpu_ctx):
    import torch
    datas = error_checks(gpu_ctx, gpu_out)
    lib = gpu_ctx.lib
    with Corpus(gpu_ctx, datas) as c:
        fo, st, co = np.array([0, 1], np.uint32), np.array([0, 500], np.int64), np.array([100, 300], np.int32)
        conv = N.OutConv(0, 0, 0)

        def call(ptr, elems):
            return lib.vpz_corpus_excerpts_device(c._h, 2, fo.ctypes.data, st.ctypes.data, co.ctypes.data, 1,
                                                  C.byref(conv), ptr, elems, None, None, None)

        total = call(None, 0)
        pageable = np.zeros(total, np.float32)
        assert call(pageable.ctypes.data, total) == N.VPZ_E_ARGUMENT
        pinned = lib.vpz_host_alloc(total * 4)
        try:
            assert call(pinned, total) == N.VPZ_E_ARGUMENT
        finally:
            lib.vpz_host_free(pinned)
        dev = torch.empty(total, dtype=torch.float32, device="cuda:0")
        assert call(dev.data_ptr(), total) == total


@pytest.mark.gpu
def test_no_packet_bytes_over_pcie(gpu_ctx):
    """Packets of about 4 KB: a corpus call uploads less than the packets holding the excerpts' starts, which the
    plain call has to upload, and the same amount when 8 large files no excerpt references join the corpus."""
    import synthvorbis
    st = synthvorbis.make_stream(0x5EED0C15, "stereo_res2", n_packets=240, mean_len=4000)
    data = st["ogg"]
    lens = np.array([len(p) for p in st["packets"]], np.int64)
    cum = np.cumsum(synthvorbis.packet_counts(st["info"], st["kinds"]))
    rng = np.random.default_rng(0x5EED0C16)
    start = np.sort(rng.integers(0, int(cum[-1]) - 4096, 48)).astype(np.int64)
    file_of = np.zeros(start.size, np.uint32)
    count = np.full(start.size, 1024, np.int32)
    i = np.searchsorted(cum, start, side="right")
    held = int(sum(lens[max(k - 1, 0):k + 2].min() for k in i))   # at least the packet holding the start
    big = [load_file("3test")] * 8
    lib = gpu_ctx.lib
    deltas = []
    for files in ([data], [data] + big, big + [data]):
        fo = file_of + (8 if files[0] is not data else 0)
        with Corpus(gpu_ctx, files) as c:
            c.excerpts(fo, start, count)   # warm: the pipeline's buffers exist
            t0 = lib.vpz_transfer_bytes(0)
            buf, _, got = c.excerpts(fo, start, count)
            deltas.append(lib.vpz_transfer_bytes(0) - t0)
            ref, _, r_got = decode_excerpts_device(gpu_ctx, files, fo, start, count)
            assert np.array_equal(got, r_got) and same(buf, ref)
    assert deltas[0] < held, (deltas, held)
    assert deltas[0] == deltas[1] == deltas[2], deltas


@pytest.mark.gpu
def test_sliced_open(gpu_ctx):
    """Slices of 64 KiB: each slice's images are copied out of the scan's buffer before the next scan reuses it."""
    sliced_open_checks(gpu_ctx, gpu_out, 400, 4096)


@pytest.mark.gpu
def test_k7_gathers_every_group(gpu_ctx, capfd, monkeypatch):
    data = [load_file("3test")]
    with Corpus(gpu_ctx, data) as c:
        nbytes, pieces, multi, groups_k7, groups = gathered(gpu_ctx, c, data, *dense_3test(256), gpu_out, capfd,
                                                            monkeypatch)
    assert nbytes > 0 and pieces > multi > 0 and groups_k7 == groups


@pytest.mark.gpu
def test_crop_batch_view(gpu_ctx):
    """Uniform crops drawn with Corpus.samples: buf.view(n, C, T) is the plain call's batch."""
    import torch
    datas = [load_file("3test"), load_file("issue6test")]
    T = 4096
    with Corpus(gpu_ctx, datas) as c:
        rng = np.random.default_rng(0x5EED0C14)
        file_of = rng.integers(0, 2, 512).astype(np.uint32)
        start = np.array([int(rng.integers(0, max(1, c.samples[f] - T))) for f in file_of], np.int64)
        count = np.full(file_of.size, T, np.int32)
        buf, _, got = c.excerpts(file_of, start, count, sample_rate=16000, channels=1)
        assert buf.is_cuda and buf.view(file_of.size, 1, T).shape == (file_of.size, 1, T)
        ref, _, r_got = decode_excerpts_device(gpu_ctx, datas, file_of, start, count, sample_rate=16000, channels=1)
        assert torch.equal(buf.view(torch.int32), ref.view(torch.int32)) and np.array_equal(got, r_got)
