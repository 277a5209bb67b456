"""Bulk decode into caller-owned device memory: vpz_decode_files_device / vpz_decode_excerpts_device (K5).

The device calls decode exactly what the host calls decode; only where the samples land differs (interleaved or
channel-major, fp32 or int16 by the reference tests' rule).  So every case here compares against the host calls on
the same inputs, bitwise, and the crop batch also against the oracle's reader.  `-m gpu` runs the product library
with torch CUDA tensors; the CPU suite runs the emulated library, whose device memory is host memory, with numpy
arrays as the destination.
"""
import ctypes as C

import numpy as np
import pytest

import cases
import oracle_binding as ob
import synthvorbis
from conftest import FILES, load_file
from vorbispizza_b200 import (Context, decode_excerpts, decode_excerpts_device, decode_files,
                              decode_files_device)
from vorbispizza_b200 import _native as N

FORMATS = [(planar, dtype) for planar in (False, True) for dtype in ("float32", "int16")]
EDGE_STARTS = (0, 1, 127, 128, 1023, 1024, -1, -2, -4096, -5000, 10 ** 7)


def to_s16(x):
    v = np.trunc(x.astype(np.float32) * np.float32(32768.0)).astype(np.int64)
    return np.clip(v, -32768, 32767).astype(np.int16)


def channels_of(datas):
    return [ob.OracleStream(d).channels for d in datas]


def as_numpy(buf):
    return buf if isinstance(buf, np.ndarray) else buf.cpu().numpy()


def sentinel(dtype):
    return np.nan if dtype == "float32" else 0x7777


def is_sentinel(a, dtype):
    return np.isnan(a) if dtype == "float32" else a == 0x7777


def emu_out(total, dtype, extra=0):
    """A numpy 'device' buffer for the emulated library, prefilled with the sentinel, `extra` elements behind it."""
    return np.full(total + extra, sentinel(dtype), dtype)


def gpu_out(total, dtype, extra=0):
    import torch
    return torch.full((total + extra,), sentinel(dtype), dtype=getattr(torch, dtype), device="cuda:0")


def assert_items(dev, ref, offsets, lengths, chans, planar, dtype, what=""):
    """dev: device-call result; ref: the host call's interleaved fp32 result with the same offsets."""
    for k, (o, n, ch) in enumerate(zip(offsets, lengths, chans)):
        o, n = int(o), int(n)
        r = ref[o:o + n * ch].reshape(-1, ch)
        if dtype == "int16":
            r = to_s16(r)
        g = dev[o:o + n * ch]
        g = g.reshape(ch, -1).T if planar else g.reshape(-1, ch)
        assert np.array_equal(np.ascontiguousarray(g).view(np.uint8), np.ascontiguousarray(r).view(np.uint8)), \
            "%s item %d (%d samples x %d ch, planar %s, %s)" % (what, k, n, ch, planar, dtype)


def files_case(ctx, datas, clip, planar, dtype, make_out, extra=16):
    """Device result of datas vs the host call; the elements behind the destination are untouched."""
    ref, counts = decode_files(ctx, datas, clip=clip)
    out = make_out(ref.size, dtype, extra)
    buf, offsets, got_counts = decode_files_device(ctx, datas, clip=clip, dtype=dtype, planar=planar, out=out[:ref.size])
    assert np.array_equal(got_counts, counts)
    chans = channels_of(datas)
    host_off = np.concatenate([[0], np.cumsum(counts * np.array(chans))[:-1]]).astype(np.int64)
    assert np.array_equal(offsets, host_off)
    full = as_numpy(out)
    assert not is_sentinel(full[:ref.size], dtype).any(), "an element of the destination was not written"
    assert is_sentinel(full[ref.size:], dtype).all(), "an element behind the destination was written"
    assert_items(full[:ref.size], ref, offsets, counts, chans, planar, dtype, "files")
    return full[:ref.size], counts


def excerpt_lists(datas, n_excerpts, nread, seed, extra_positions=EDGE_STARTS):
    totals = [max(ob.OracleStream(d).decode_all()[0].shape[0], 2) for d in datas]
    rng = np.random.default_rng(seed)
    file_of = list(rng.integers(0, len(datas), n_excerpts))
    start = [int(rng.integers(0, max(1, totals[f] - 1))) for f in file_of]
    for f in range(len(datas)):
        for p in extra_positions:
            file_of.append(f)
            start.append(int(p) if p >= 0 else totals[f] + int(p))
    return np.array(file_of, np.uint32), np.array(start, np.int64), np.full(len(file_of), nread, np.int32)


def excerpts_case(ctx, datas, file_of, start, count, clip, planar, dtype, make_out, extra=16):
    ref, offsets, got = decode_excerpts(ctx, datas, file_of, start, count, clip=clip)
    out = make_out(ref.size, dtype, extra)
    buf, d_offsets, d_got = decode_excerpts_device(ctx, datas, file_of, start, count, clip=clip, dtype=dtype,
                                                   planar=planar, out=out[:ref.size])
    assert np.array_equal(d_offsets, offsets) and np.array_equal(d_got, got)
    full = as_numpy(out)
    assert not is_sentinel(full[:ref.size], dtype).any(), "an element of the destination was not written"
    assert is_sentinel(full[ref.size:], dtype).all(), "an element behind the destination was written"
    chans = channels_of(datas)
    ch = [chans[f] for f in file_of]
    assert_items(full[:ref.size], ref, offsets, count, ch, planar, dtype, "excerpts")
    for i in range(file_of.size):   # undelivered samples are zero
        have = max(int(got[i]), 0)
        o, n = int(offsets[i]), int(count[i])
        row = full[o:o + n * ch[i]].reshape(ch[i], n) if planar else full[o:o + n * ch[i]].reshape(n, ch[i]).T
        assert not row[:, have:].any(), "excerpt %d: samples past %d are not zero" % (i, have)
    return full[:ref.size], offsets, got


# ---- CPU: the emulated library, numpy destinations ----------------------------------------------------------------
def emu_datas():
    # mono and (a truncated) stereo: both placement paths of K5 at emulator sizes
    return [load_file("1test"), load_file("3test")[:40000], load_file("1test")]


@pytest.mark.parametrize("planar,dtype", FORMATS)
@pytest.mark.parametrize("clip", [True, False])
def test_emu_files(emu_ctx, planar, dtype, clip):
    files_case(emu_ctx, emu_datas(), clip, planar, dtype, emu_out)


@pytest.fixture(scope="module", params=[1, 2])
def emu_general_ctx(emu_lib_path, request):
    ctx = Context(0, lib_path=emu_lib_path)
    ctx.set("force_general", request.param)
    yield ctx
    ctx.close()


def test_emu_files_general_path(emu_general_ctx):
    files_case(emu_general_ctx, [load_file("1test")], True, True, "float32", emu_out)


def test_emu_files_s16_matches_host_s16(emu_ctx):
    datas = emu_datas()
    dev, _ = files_case(emu_ctx, datas, True, False, "int16", emu_out)
    host16, _ = decode_files(emu_ctx, datas, clip=True, s16=True)
    assert np.array_equal(dev, host16)


@pytest.mark.parametrize("planar,dtype", FORMATS)
def test_emu_excerpts(emu_ctx, planar, dtype):
    datas = [load_file("1test"), load_file("3test")[:40000]]
    file_of, start, count = excerpt_lists(datas, 4, 700, 0x5EED0009, extra_positions=(0, 1, 1024, -1, -300, 10 ** 7))
    _, _, got = excerpts_case(emu_ctx, datas, file_of, start, count, False, planar, dtype, emu_out)
    assert (got < 0).any() and (got < count).sum() > (got < 0).sum()   # failed seeks and short reads are covered


def test_emu_errors_and_size_query(emu_ctx):
    datas = [load_file("1test")]
    keep = [np.frombuffer(d, np.uint8) for d in datas]
    ptrs = (C.c_void_p * 1)(keep[0].ctypes.data)
    lens = (C.c_size_t * 1)(keep[0].size)
    counts = np.zeros(1, np.int64)
    lib = emu_ctx.lib
    ref, ref_counts = decode_files(emu_ctx, datas)
    total = lib.vpz_decode_files_device(emu_ctx._h, 1, ptrs, lens, 1, N.VPZ_OUT_PLANAR, None, 0, counts.ctypes.data, None)
    assert total == ref.size and np.array_equal(counts, ref_counts)
    out = np.zeros(ref.size, np.float32)
    assert lib.vpz_decode_files_device(emu_ctx._h, 1, ptrs, lens, 1, 4, out.ctypes.data, out.size, None, None) == N.VPZ_E_ARGUMENT
    assert lib.vpz_decode_files_device(emu_ctx._h, 1, ptrs, lens, 1, 0, out.ctypes.data, out.size - 1, None, None) == N.VPZ_E_ARGUMENT
    fo, st, co = np.zeros(2, np.uint32), np.array([0, 500], np.int64), np.array([100, 300], np.int32)
    offs, got = np.zeros(2, np.int64), np.zeros(2, np.int32)
    args = (emu_ctx._h, 1, ptrs, lens, 2, fo.ctypes.data, st.ctypes.data, co.ctypes.data, 1)
    assert lib.vpz_decode_excerpts_device(*args, 0, None, 0, offs.ctypes.data, got.ctypes.data, None) == 400
    assert lib.vpz_decode_excerpts_device(*args, 8, out.ctypes.data, 400, offs.ctypes.data, got.ctypes.data, None) == N.VPZ_E_ARGUMENT
    assert lib.vpz_decode_excerpts_device(*args, 0, out.ctypes.data, 399, offs.ctypes.data, got.ctypes.data, None) == N.VPZ_E_ARGUMENT


# ---- GPU: the product library, torch CUDA tensors ----------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("planar,dtype", FORMATS)
@pytest.mark.parametrize("clip", [True, False])
def test_files(gpu_ctx, planar, dtype, clip):
    """fp32 interleaved is bitwise the host call; planar is the host item transposed; int16 is the rule on it."""
    files_case(gpu_ctx, [load_file(n) for n in FILES + ["3test", "1test"]], clip, planar, dtype, gpu_out)


@pytest.mark.gpu
@pytest.mark.parametrize("force", [1, 2])
def test_files_general_paths(force):
    """The general K1b, the generic K3 (1) and also the full K1a (2) feed K5."""
    ctx = Context(0)
    try:
        ctx.set("force_general", force)
        for planar, dtype in FORMATS:
            files_case(ctx, [load_file(n) for n in FILES], True, planar, dtype, gpu_out)
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("clip", [True, False])
def test_files_s16_matches_host_s16(gpu_ctx, clip):
    datas = [load_file(n) for n in FILES]
    dev, _ = files_case(gpu_ctx, datas, clip, False, "int16", gpu_out)
    host16, _ = decode_files(gpu_ctx, datas, clip=clip, s16=True)
    assert np.array_equal(dev, host16)


@pytest.mark.gpu
def test_files_s16_six_channels(gpu_ctx):
    """A generated 6-channel stream beside a stereo one: the generic K3 feeds K5, which converts after it."""
    datas = [synthvorbis.make_stream(0x5EED0601, "ch6_coupled", n_packets=60)["ogg"], load_file("3test")]
    assert channels_of(datas) == [6, 2]
    for planar in (False, True):
        files_case(gpu_ctx, datas, True, planar, "float32", gpu_out)
        dev16, _ = files_case(gpu_ctx, datas, True, planar, "int16", gpu_out)
        if not planar:
            host16, _ = decode_files(gpu_ctx, datas, clip=True, s16=True)
            assert np.array_equal(dev16, host16)


@pytest.mark.gpu
def test_files_pipeline_rotation():
    """Groups of 8 streams: 64 files go through all three pipeline slots several times."""
    ctx = Context(0)
    try:
        ctx.set("bulk_group", 8)
        datas = [load_file(n) for n in FILES] * 16
        for planar, dtype in FORMATS:
            files_case(ctx, datas, True, planar, dtype, gpu_out)
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("planar,dtype", FORMATS)
def test_excerpts(gpu_ctx, planar, dtype):
    datas = [load_file(n) for n in ["2test", "3test", "issue6test"]]
    file_of, start, count = excerpt_lists(datas, 300, 4096, 0x5EED0005)
    excerpts_case(gpu_ctx, datas, file_of, start, count, True, planar, dtype, gpu_out)
    datas = [load_file(n) for n in ["1test", "3test"]]
    file_of, start, count = excerpt_lists(datas, 64, 700, 77)
    _, _, got = excerpts_case(gpu_ctx, datas, file_of, start, count, False, planar, dtype, gpu_out)
    assert (got < 0).any() and (got < count).sum() > (got < 0).sum()


@pytest.mark.gpu
def test_dense_crop_batch(gpu_ctx):
    """Stereo files, one count: out.view(n, C, T) row by row against the oracle reader's SeekTo + Read."""
    import torch
    datas = [load_file("3test"), load_file("issue6test")]
    T = 2048
    file_of, start, count = excerpt_lists(datas, 96, T, 0x5EED00C5, extra_positions=(0, 1, 1024))
    buf, offsets, got = decode_excerpts_device(gpu_ctx, datas, file_of, start, count, clip=True)
    assert buf.is_cuda and buf.dtype == torch.float32
    batch = buf.view(file_of.size, 2, T).cpu().numpy()
    rd = np.zeros(T * 2, np.float32)
    for i in range(file_of.size):
        s = ob.OracleStream(datas[int(file_of[i])])
        s.seek(int(start[i]))
        n = 0
        while n < T:
            k = s.read(rd[n * 2:])
            if k <= 0:
                break
            n += k
        assert got[i] == n
        cases.assert_pcm_close(batch[i][:, :n].T, rd[:n * 2].reshape(-1, 2), "crop %d" % i)
        assert not batch[i][:, n:].any()


@pytest.mark.gpu
def test_waits_for_the_callers_stream(gpu_ctx):
    """The destination is overwritten with NaN on a busy side stream just before the call; the call is given that
    stream, so its samples land after the fill."""
    import torch
    datas = [load_file(n) for n in FILES]
    ref, counts = decode_files(gpu_ctx, datas)
    out = torch.zeros(ref.size, dtype=torch.float32, device="cuda:0")
    a = torch.randn(4096, 4096, device="cuda:0")
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(16):
            a = a @ a
            a = a / a.norm()
        out.fill_(float("nan"))
    buf, _, _ = decode_files_device(gpu_ctx, datas, planar=False, out=out, stream=side)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy().view(np.uint32), ref.view(np.uint32))


@pytest.mark.gpu
def test_errors_and_size_query(gpu_ctx):
    import torch
    datas = [load_file(n) for n in ["1test", "3test"]]
    keep = [np.frombuffer(d, np.uint8) for d in datas]
    ptrs = (C.c_void_p * 2)(*[k.ctypes.data for k in keep])
    lens = (C.c_size_t * 2)(*[k.size for k in keep])
    counts = np.zeros(2, np.int64)
    lib, h = gpu_ctx.lib, gpu_ctx._h
    ref, ref_counts = decode_files(gpu_ctx, datas)
    total = lib.vpz_decode_files_device(h, 2, ptrs, lens, 1, N.VPZ_OUT_S16, None, 0, counts.ctypes.data, None)
    assert total == ref.size and np.array_equal(counts, ref_counts)

    def files(ptr, elems, fmt=0):
        return lib.vpz_decode_files_device(h, 2, ptrs, lens, 1, fmt, ptr, elems, None, None)

    pageable = np.zeros(ref.size, np.float32)
    assert files(pageable.ctypes.data, ref.size) == N.VPZ_E_ARGUMENT
    assert lib.vpz_last_error(h)
    pinned = lib.vpz_host_alloc(ref.size * 4)
    try:
        assert files(pinned, ref.size) == N.VPZ_E_ARGUMENT
    finally:
        lib.vpz_host_free(pinned)
    dev = torch.empty(ref.size, dtype=torch.float32, device="cuda:0")
    assert files(dev.data_ptr(), ref.size - 1) == N.VPZ_E_ARGUMENT
    assert files(dev.data_ptr(), ref.size, 4) == N.VPZ_E_ARGUMENT
    assert files(dev.data_ptr(), ref.size) == ref.size
    torch.cuda.synchronize()
    assert np.array_equal(dev.cpu().numpy().view(np.uint32), ref.view(np.uint32))
    # excerpts: the size query and its offsets are the host call's
    fo, st, co = np.array([0, 1, 1], np.uint32), np.array([0, 500, 10 ** 7], np.int64), np.array([100, 300, 50], np.int32)
    r_pcm, r_off, r_got = decode_excerpts(gpu_ctx, datas, fo, st, co)
    offs, got = np.zeros(3, np.int64), np.zeros(3, np.int32)
    args = (h, 2, ptrs, lens, 3, fo.ctypes.data, st.ctypes.data, co.ctypes.data, 1)
    assert lib.vpz_decode_excerpts_device(*args, 0, None, 0, offs.ctypes.data, got.ctypes.data, None) == r_pcm.size
    assert np.array_equal(offs, r_off)
    assert lib.vpz_decode_excerpts_device(*args, 0, pageable.ctypes.data, r_pcm.size, None, None, None) == N.VPZ_E_ARGUMENT
    assert lib.vpz_decode_excerpts_device(*args, 0, dev.data_ptr(), r_pcm.size - 1, None, None, None) == N.VPZ_E_ARGUMENT
    assert lib.vpz_decode_excerpts_device(*args, 16, dev.data_ptr(), r_pcm.size, None, None, None) == N.VPZ_E_ARGUMENT
