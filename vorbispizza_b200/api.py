"""Python host mirror of the reference's reader interface over the C ABI (include/vpz.h).

Names and behaviour follow NVorbis/VorbisReader.cs and NVorbis/Contracts/IStreamDecoder.cs
(ReadSamples, SeekTo, Streams, SwitchStreams, FindNextStream, Tags, ClipSamples, HasClipped,
IsEndOfStream, TotalSamples, SamplePosition ...), spelled the Python way.  Errors map onto the
reference's exception types the way INTEGRATION.md lists them.
"""
import ctypes as C
import weakref

import numpy as np

from . import _native as N


class InvalidDataError(N.VpzError):        # System.IO.InvalidDataException
    pass


class SeekOutOfRangeError(N.VpzError):     # NVorbis.SeekOutOfRangeException
    pass


class PreRollPacketError(N.VpzError):      # NVorbis.PreRollPacketException
    pass


_EXC = {
    N.VPZ_E_INVALID_DATA: InvalidDataError,
    N.VPZ_E_SEEK_RANGE: SeekOutOfRangeError,
    N.VPZ_E_PREROLL: PreRollPacketError,
}


def _u8(data):
    """bytes / bytearray / uint8 ndarray -> (keepalive ndarray, pointer, length)"""
    if isinstance(data, np.ndarray):
        a = np.ascontiguousarray(data, dtype=np.uint8)
    else:
        a = np.frombuffer(data, dtype=np.uint8)
    return a, (a.ctypes.data if a.size else None), a.size


class Context:
    """One per GPU (vpz_ctx): stream, setup-table cache, tunables."""

    def __init__(self, device=-1, lib_path=None):
        self.lib = N.load(lib_path)
        self.device = device
        h = C.c_void_p()
        rc = self.lib.vpz_ctx_create(device, C.byref(h))
        if rc:
            raise N.VpzError(rc, self.lib.vpz_strerror(rc).decode())
        self._h = h
        self._corpora = weakref.WeakSet()   # open Corpus objects: closed before the context

    def check(self, rc):
        if rc is not None and rc < 0:
            text = self.lib.vpz_last_error(self._h).decode(errors="replace") or self.lib.vpz_strerror(rc).decode()
            raise _EXC.get(rc, N.VpzError)(rc, text)
        return rc

    def set(self, key, value):
        self.check(self.lib.vpz_ctx_set(self._h, key.encode(), int(value)))

    def close(self):
        if self._h:
            for c in list(self._corpora):   # a corpus must be closed before its context
                c.close()
            self.lib.vpz_ctx_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def create_setup(self, id_packet, setup_packet):
        a, pa, na = _u8(id_packet)
        b, pb, nb = _u8(setup_packet)
        s = C.c_void_p()
        self.check(self.lib.vpz_setup_create(self._h, pa, na, pb, nb, C.byref(s)))
        return s

    def release_setup(self, s):
        self.lib.vpz_setup_release(s)

    def setup_info(self, s):
        info = N.SetupInfo()
        self.check(self.lib.vpz_setup_get_info(s, C.byref(info)))
        return info

    def packet_info(self, s, packet):
        a, p, n = _u8(packet)
        out = (C.c_int32 * 6)()
        rc = self.check(self.lib.vpz_packet_info(s, p, n, out))
        return rc, list(out)

    def debug_decode_packet(self, s, packet, channels, block_size1, cap=8192):
        """Every stage of one audio packet (bit-exact parity tests)."""
        a, p, n = _u8(packet)
        dump = N.PacketDump()
        scal = np.zeros(cap, np.int32)
        cls = np.zeros(cap, np.int32)
        res = np.zeros(channels * block_size1 // 2, np.float32)
        spec = np.zeros(channels * block_size1 // 2, np.float32)
        imd = np.zeros(channels * block_size1, np.float32)
        self.check(self.lib.vpz_debug_decode_packet(self._h, s, p, n, C.byref(dump), scal.ctypes.data, cap,
                                                    cls.ctypes.data, cap, res.ctypes.data, spec.ctypes.data,
                                                    imd.ctypes.data))
        out = dict(status=dump.status, mode=dump.mode, block_size=dump.block_size, info=list(dump.info),
                   bits_read=dump.bits_read, exec_mask=dump.exec_mask, no_execute_mask=dump.no_execute_mask,
                   scalars_n=dump.scalars_n, classes_n=dump.classes_n, scalars=scal[:min(dump.scalars_n, cap)].copy(),
                   classes=cls[:min(dump.classes_n, cap)].copy(),
                   post_count=[dump.post_count[c] for c in range(channels)],
                   raw_posts=np.array([list(dump.raw_posts[c]) for c in range(channels)], np.int32),
                   final_y=np.array([list(dump.final_y[c]) for c in range(channels)], np.int32),
                   step_flags=np.array([list(dump.step_flags[c]) for c in range(channels)], np.int32))
        if dump.status == 0:
            nb = dump.block_size
            out["residue"] = res[:channels * nb // 2].reshape(channels, nb // 2).copy()
            out["spectrum"] = spec[:channels * nb // 2].reshape(channels, nb // 2).copy()
            out["imdct"] = imd[:channels * nb].reshape(channels, nb).copy()
        return out


class Batch:
    """Many packets of many streams in one GPU pass (vpz_batch_*): the IPacketProvider-side seam."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.lib = ctx.lib
        h = C.c_void_p()
        ctx.check(self.lib.vpz_batch_create(ctx._h, C.byref(h)))
        self._h = h
        self._keep = []

    def close(self):
        if self._h:
            self.lib.vpz_batch_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def reset(self):
        self.ctx.check(self.lib.vpz_batch_reset(self._h))

    def add_run(self, setup, packets, trim=None):
        """packets: list of bytes objects (one fresh-decoder run).  Returns the run index."""
        lens = np.fromiter((len(p) for p in packets), dtype=np.int64, count=len(packets))
        offs = np.zeros(len(packets) + 1, np.uint32)
        offs[1:] = np.cumsum(lens)
        blob = np.frombuffer(b"".join(packets), np.uint8)
        return self.add_run_raw(setup, blob, offs, trim)

    def add_run_raw(self, setup, blob, offs, trim=None):
        t = None
        if trim is not None:
            t = np.ascontiguousarray(trim, dtype=np.int32)
        rc = self.lib.vpz_batch_add_run(self._h, setup, blob.ctypes.data if blob.size else None, offs.ctypes.data,
                                        len(offs) - 1, t.ctypes.data if t is not None else None)
        return self.ctx.check(rc)

    def run_samples(self, run):
        return self.ctx.check(self.lib.vpz_batch_run_samples(self._h, run))

    def run_channels(self, run):
        return self.ctx.check(self.lib.vpz_batch_run_channels(self._h, run))

    def run_status(self, run):
        stop = C.c_int32(-1)
        rc = self.lib.vpz_batch_run_status(self._h, run, C.byref(stop))
        return rc, stop.value

    def run_packet_samples(self, run, n_pkts):
        a = np.zeros(n_pkts, np.int32)
        self.ctx.check(self.lib.vpz_batch_run_packet_samples(self._h, run, a.ctypes.data))
        return a

    @property
    def total_floats(self):
        return self.lib.vpz_batch_total_floats(self._h)

    @property
    def total_packets(self):
        return self.lib.vpz_batch_total_packets(self._h)

    @property
    def total_bytes(self):
        return self.lib.vpz_batch_total_bytes(self._h)

    def upload(self):
        self.ctx.check(self.lib.vpz_batch_upload(self._h))

    def decode(self, clip=True, sync=True):
        self.ctx.check(self.lib.vpz_batch_decode(self._h, int(bool(clip))))
        if sync:
            self.sync()

    def sync(self):
        self.ctx.check(self.lib.vpz_batch_sync(self._h))

    @property
    def has_clipped(self):
        return bool(self.ctx.check(self.lib.vpz_batch_has_clipped(self._h)))

    def read_run(self, run):
        n, ch = self.run_samples(run), self.run_channels(run)
        out = np.zeros((n, ch), np.float32)
        if n:
            self.ctx.check(self.lib.vpz_batch_read_run(self._h, run, out.ctypes.data))
        return out

    def read_all(self, dst=None):
        n = self.total_floats
        if dst is None:
            dst = np.zeros(n, np.float32)
        self.ctx.check(self.lib.vpz_batch_read_all(self._h, dst.ctypes.data))
        return dst

    def last_ms(self):
        """(total, entropy stage, imdct/ola) device milliseconds and kernel launches of the last decode."""
        ln = C.c_int(0)
        tot = self.lib.vpz_batch_last_ms(self._h, 0, C.byref(ln))
        return tot, self.lib.vpz_batch_last_ms(self._h, 1, None), self.lib.vpz_batch_last_ms(self._h, 3, None), ln.value

    def last_ms_k1(self):
        """(symbol decode K1a, spectrum build K1b) device milliseconds of the last decode."""
        return self.lib.vpz_batch_last_ms(self._h, 11, None), self.lib.vpz_batch_last_ms(self._h, 12, None)

    def device_pcm(self):
        return self.lib.vpz_batch_device_pcm(self._h)

    def run_offset(self, run):
        return self.ctx.check(self.lib.vpz_batch_run_offset(self._h, run))


class SynthBatch(Batch):
    """Kernel-only IMDCT + window + overlap-add on caller spectra (BASELINE config 3)."""

    def __init__(self, ctx, channels, log2_size0, log2_size1, flags, spectra):
        self.ctx = ctx
        self.lib = ctx.lib
        flags = np.ascontiguousarray(flags, dtype=np.uint8)
        spectra = np.ascontiguousarray(spectra, dtype=np.float32)
        n_streams, n_blocks = flags.shape
        h = C.c_void_p()
        ctx.check(self.lib.vpz_synth_create(ctx._h, channels, log2_size0, log2_size1, n_streams, n_blocks,
                                            flags.ctypes.data, spectra.ctypes.data, C.byref(h)))
        self._h = h
        self._keep = []


class VorbisReader:
    """VorbisReader (NVorbis/VorbisReader.cs) over container bytes in memory."""

    def __init__(self, ctx, data, lookahead=None):
        self.ctx = ctx
        self.lib = ctx.lib
        self._buf, p, n = _u8(data)
        h = C.c_void_p()
        ctx.check(self.lib.vpz_reader_open_memory(ctx._h, p, n, 0, C.byref(h)))
        self._h = h
        if lookahead is not None:
            self.set_lookahead(lookahead)

    def close(self):  # Dispose
        if self._h:
            self.lib.vpz_reader_close(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- streams
    @property
    def stream_count(self):
        return self.lib.vpz_reader_stream_count(self._h)

    @property
    def stream_index(self):
        return self.lib.vpz_reader_stream_index(self._h)

    def switch_streams(self, index):
        return bool(self.ctx.check(self.lib.vpz_reader_switch_stream(self._h, index)))

    def find_next_stream(self):
        return bool(self.ctx.check(self.lib.vpz_reader_find_next_stream(self._h)))

    @property
    def can_seek(self):
        return bool(self.lib.vpz_reader_can_seek(self._h))

    # ---- properties of the current stream
    @property
    def channels(self):
        return self.lib.vpz_reader_channels(self._h)

    @property
    def sample_rate(self):
        return self.lib.vpz_reader_sample_rate(self._h)

    @property
    def upper_bitrate(self):
        return self.lib.vpz_reader_bitrate(self._h, 0)

    @property
    def nominal_bitrate(self):
        return self.lib.vpz_reader_bitrate(self._h, 1)

    @property
    def lower_bitrate(self):
        return self.lib.vpz_reader_bitrate(self._h, 2)

    @property
    def stream_serial(self):
        return self.lib.vpz_reader_stream_serial(self._h)

    @property
    def total_samples(self):
        return self.ctx.check(self.lib.vpz_reader_total_samples(self._h))

    @property
    def sample_position(self):
        return self.lib.vpz_reader_sample_position(self._h)

    @property
    def is_end_of_stream(self):
        return bool(self.lib.vpz_reader_is_end_of_stream(self._h))

    @property
    def has_clipped(self):
        return bool(self.lib.vpz_reader_has_clipped(self._h))

    @property
    def clip_samples(self):
        return bool(self.lib.vpz_reader_get_clip(self._h))

    @clip_samples.setter
    def clip_samples(self, v):
        self.lib.vpz_reader_set_clip(self._h, int(bool(v)))

    @property
    def container_overhead_bits(self):
        return self.lib.vpz_reader_container_overhead_bits(self._h)

    @property
    def container_waste_bits(self):
        return self.lib.vpz_reader_container_waste_bits(self._h)

    @property
    def vendor(self):
        n = C.c_int(0)
        p = self.lib.vpz_reader_vendor(self._h, C.byref(n))
        return C.string_at(p, n.value) if p else b""

    @property
    def comments(self):
        out = []
        for i in range(self.lib.vpz_reader_comment_count(self._h)):
            n = C.c_int(0)
            p = self.lib.vpz_reader_comment(self._h, i, C.byref(n))
            out.append(C.string_at(p, n.value) if p else b"")
        return out

    @property
    def tags(self):
        """TagData-style dictionary: upper-cased key -> list of values (TagData.cs:12-46)."""
        d = {}
        for c in self.comments:
            k, sep, v = c.partition(b"=")
            if sep:
                d.setdefault(k.decode("utf-8", "replace").upper(), []).append(v.decode("utf-8", "replace"))
        return d

    # ---- decode
    def read_samples(self, buf):
        """ReadSamples(Span<float>) (VorbisReader.cs:232-241): interleaved; returns samples per channel."""
        assert buf.dtype == np.float32 and buf.flags.c_contiguous
        count = buf.size - buf.size % self.channels
        if count == 0:
            return 0
        return self.ctx.check(self.lib.vpz_reader_read(self._h, buf.ctypes.data, count))

    def read_samples_planar(self, buf, samples_to_read, channel_stride):
        """ReadSamples(Span<float>, samplesToRead, channelStride) (VorbisReader.cs:244-253)."""
        assert buf.dtype == np.float32 and buf.flags.c_contiguous
        count = buf.size - buf.size % self.channels
        if count == 0:
            return 0
        return self.ctx.check(self.lib.vpz_reader_read_planar(self._h, buf.ctypes.data, count, samples_to_read,
                                                              channel_stride))

    def seek_to(self, sample_position, origin=0):
        self.ctx.check(self.lib.vpz_reader_seek(self._h, int(sample_position), origin))

    def set_lookahead(self, packets):
        self.ctx.check(self.lib.vpz_reader_set_lookahead(self._h, packets))

    def decode_all(self, chunk_floats=48000):
        """TestApp-style drain (TestApp/Program.cs:42,155).  Returns (pcm[samples, ch], per-call counts, fault)."""
        ch = self.channels
        chunk_floats -= chunk_floats % ch
        buf = np.empty(chunk_floats, np.float32)
        out, counts, fault = [], [], 0
        while True:
            n = self.lib.vpz_reader_read(self._h, buf.ctypes.data, buf.size)
            if n < 0:
                fault = n
                break
            if n == 0:
                break
            counts.append(n)
            out.append(buf[:n * ch].copy())
        pcm = np.concatenate(out).reshape(-1, ch) if out else np.zeros((0, ch), np.float32)
        return pcm, counts, fault

    # ---- packet access
    def audio_packets(self):
        n = self.ctx.check(self.lib.vpz_reader_audio_packet_count(self._h))
        out = []
        for i in range(n):
            p, ln, g, fl = C.c_void_p(), C.c_uint32(0), C.c_int64(0), C.c_int32(0)
            self.ctx.check(self.lib.vpz_reader_audio_packet(self._h, i, C.byref(p), C.byref(ln), C.byref(g), C.byref(fl)))
            out.append(dict(data=C.string_at(p, ln.value) if ln.value else b"", granule=g.value,
                            is_resync=bool(fl.value & 1), is_eos=bool(fl.value & 2)))
        return out

    def header_packet(self, which):
        n = C.c_uint32(0)
        p = self.lib.vpz_reader_header_packet(self._h, which, C.byref(n))
        return C.string_at(p, n.value) if p else b""

    @property
    def setup(self):
        return C.c_void_p(self.lib.vpz_reader_setup(self._h))


def decode_files(ctx, files, clip=True, dst=None, s16=False):
    """Bulk decode of whole container images in ONE GPU batch (vpz_decode_files / vpz_decode_files_s16).

    files: list of bytes / uint8 arrays.  Returns (pcm 1-D: file after file, interleaved; float32, or
    int16 with s16=True: the reference tests' (int)(x * 32768f) rule applied on the GPU), per-file
    samples-per-channel counts.  dst may be a preallocated (pinned) array of the output type.
    """
    keep = [_u8(f) for f in files]
    n = len(keep)
    ptrs = (C.c_void_p * n)(*[k[1] for k in keep])
    lens = (C.c_size_t * n)(*[k[2] for k in keep])
    counts = np.zeros(n, np.int64)
    fn = ctx.lib.vpz_decode_files_s16 if s16 else ctx.lib.vpz_decode_files
    if dst is None:
        # sizes are only known after the headers are parsed: first pass without output
        total = ctx.check(fn(ctx._h, n, ptrs, lens, int(bool(clip)), None, 0, counts.ctypes.data))
        dst = np.zeros(total, np.int16 if s16 else np.float32)
    total = ctx.check(fn(ctx._h, n, ptrs, lens, int(bool(clip)), dst.ctypes.data, dst.size, counts.ctypes.data))
    return dst[:total], counts


def decode_excerpts(ctx, files, file_of, start, count, clip=True, dst=None):
    """Bulk random access (vpz_decode_excerpts): excerpt i = SeekTo(start[i]) + read count[i] samples per
    channel on files[file_of[i]], every excerpt like a fresh reader; the windows of many excerpts share one
    GPU batch.  Returns (pcm float32 1-D, offsets int64 (float offset of each excerpt in pcm), got int32
    (samples per channel delivered, or the negative status SeekTo raised))."""
    keep = [_u8(f) for f in files]
    nf = len(keep)
    ptrs = (C.c_void_p * nf)(*[k[1] for k in keep])
    lens = (C.c_size_t * nf)(*[k[2] for k in keep])
    file_of = np.ascontiguousarray(file_of, dtype=np.uint32)
    start = np.ascontiguousarray(start, dtype=np.int64)
    count = np.ascontiguousarray(count, dtype=np.int32)
    n = file_of.size
    offsets = np.zeros(n, np.int64)
    got = np.zeros(n, np.int32)
    args = (ctx._h, nf, ptrs, lens, n, file_of.ctypes.data, start.ctypes.data, count.ctypes.data, int(bool(clip)))
    if dst is None:
        total = ctx.check(ctx.lib.vpz_decode_excerpts(*args, None, 0, offsets.ctypes.data, got.ctypes.data))
        dst = np.full(total, np.nan, np.float32)   # the call defines every float: short reads are zero-filled
    total = ctx.check(ctx.lib.vpz_decode_excerpts(*args, dst.ctypes.data, dst.size, offsets.ctypes.data, got.ctypes.data))
    return dst[:total], offsets, got


def _device_out(ctx, out, total, dtype, stream):
    """The destination of a *_device call: (buffer, pointer, elements, cudaStream_t handle).  out=None allocates a
    torch CUDA tensor on the context's device; out may be a caller tensor, or a numpy array for the emulated
    library (whose device memory is host memory).  stream=None: torch's current stream for a tensor."""
    if dtype not in ("float32", "int16"):
        raise ValueError("dtype must be 'float32' or 'int16'")
    if out is None:
        import torch
        dev = torch.device("cuda", ctx.device if ctx.device >= 0 else torch.cuda.current_device())
        out = torch.empty(max(total, 1), dtype=getattr(torch, dtype), device=dev)[:total]
    if isinstance(out, np.ndarray):
        if out.dtype != np.dtype(dtype) or not out.flags.c_contiguous:
            raise ValueError("out must be a contiguous %s array" % dtype)
        return out, (out.ctypes.data if out.size else None), out.size, stream
    import torch
    if out.dtype != getattr(torch, dtype) or not out.is_contiguous():
        raise ValueError("out must be a contiguous %s tensor" % dtype)
    if stream is None and out.is_cuda:
        stream = torch.cuda.current_stream(out.device)
    handle = stream.cuda_stream if hasattr(stream, "cuda_stream") else stream
    return out, (out.data_ptr() if out.numel() else None), out.numel(), handle


def _format(dtype, planar):
    return (N.VPZ_OUT_S16 if dtype == "int16" else 0) | (N.VPZ_OUT_PLANAR if planar else 0)


def _vorbis_channels(data):
    """Channel count from a container image's first identification header ("\\x01vorbis", channels at byte 11)."""
    i = bytes(data[:1 << 16]).find(b"\x01vorbis")
    return data[i + 11] if i >= 0 and i + 11 < len(data) else 0


def _conv(fmt, sample_rate, channels):
    """The vpz_out_conv of sample_rate / channels keywords, or None when neither is given (the plain *_device call)."""
    if sample_rate is None and channels is None:
        return None
    return N.OutConv(fmt, int(sample_rate or 0), int(channels or 0))


def decode_files_device(ctx, files, clip=True, dtype="float32", planar=True, out=None, stream=None, sample_rate=None,
                        channels=None):
    """vpz_decode_files_device: decode_files with the PCM left in device memory.

    Returns (buf, offsets, counts): buf is one flat buffer of `dtype` ("float32", or "int16" by the reference
    tests' (int)(x * 32768f) rule); file k starts at element offsets[k] and has counts[k] samples per channel,
    channel-major [C_k][counts[k]] with planar=True, interleaved otherwise.  When every file has the same channel
    count C and length T, ``buf.view(n, C, T)`` is the batch.  out: a caller tensor (contiguous, on the context's
    device) instead of a new one; stream: the torch / CUDA stream the result is used on (default: the current one);
    the call waits for the work queued on it and returns when buf is complete.

    sample_rate / channels (vpz_decode_files_device_conv): every file converted on the GPU to that rate
    (torchaudio.functional.resample's default filter) and to 1 channel (the mean) or 2 (mono duplicated); None or 0
    keeps the stream's own.  counts are then output samples and offsets the converted layout's."""
    keep = [_u8(f) for f in files]
    n = len(keep)
    ptrs = (C.c_void_p * n)(*[k[1] for k in keep])
    lens = (C.c_size_t * n)(*[k[2] for k in keep])
    counts = np.zeros(n, np.int64)
    fmt = _format(dtype, planar)
    conv = _conv(fmt, sample_rate, channels)
    if conv is not None:
        offsets = np.zeros(n, np.int64)
        args = (ctx._h, n, ptrs, lens, int(bool(clip)), C.byref(conv))
        total = None
        if out is None:
            total = ctx.check(ctx.lib.vpz_decode_files_device_conv(*args, None, 0, counts.ctypes.data, None, None))
        buf, ptr, elems, handle = _device_out(ctx, out, total, dtype, stream)
        total = ctx.check(ctx.lib.vpz_decode_files_device_conv(*args, ptr, elems, counts.ctypes.data,
                                                               offsets.ctypes.data, handle))
        return buf[:total], offsets, counts
    args = (ctx._h, n, ptrs, lens, int(bool(clip)), fmt)
    total = None
    if out is None:
        total = ctx.check(ctx.lib.vpz_decode_files_device(*args, None, 0, counts.ctypes.data, None))
    buf, ptr, elems, handle = _device_out(ctx, out, total, dtype, stream)
    total = ctx.check(ctx.lib.vpz_decode_files_device(*args, ptr, elems, counts.ctypes.data, handle))
    chans = np.array([_vorbis_channels(k[0]) for k in keep], np.int64)
    offsets = np.zeros(n, np.int64)
    if n > 1:
        offsets[1:] = np.cumsum(counts * chans)[:-1]
    return buf[:total], offsets, counts


def decode_excerpts_device(ctx, files, file_of, start, count, clip=True, dtype="float32", planar=True, out=None,
                           stream=None, sample_rate=None, channels=None):
    """vpz_decode_excerpts_device: decode_excerpts with the PCM left in device memory.

    Returns (buf, offsets, got) as decode_excerpts does; excerpt i starts at element offsets[i] and holds count[i]
    samples per channel, channel-major with planar=True; samples not delivered are zero.  With one channel count C
    and a uniform count T (a crop batch), ``buf.view(n, C, T)`` is the batch.  dtype, out, stream: as
    decode_files_device.

    sample_rate / channels (vpz_decode_excerpts_device_conv): as decode_files_device; start and count are then
    samples at the output rate, and got counts output samples.  A mixed-rate, mixed-layout corpus cropped to one
    rate, channel count and length is one dense [n, C, T] batch."""
    keep = [_u8(f) for f in files]
    nf = len(keep)
    ptrs = (C.c_void_p * nf)(*[k[1] for k in keep])
    lens = (C.c_size_t * nf)(*[k[2] for k in keep])
    file_of = np.ascontiguousarray(file_of, dtype=np.uint32)
    start = np.ascontiguousarray(start, dtype=np.int64)
    count = np.ascontiguousarray(count, dtype=np.int32)
    n = file_of.size
    offsets = np.zeros(n, np.int64)
    got = np.zeros(n, np.int32)
    fmt = _format(dtype, planar)
    conv = _conv(fmt, sample_rate, channels)
    fn = ctx.lib.vpz_decode_excerpts_device if conv is None else ctx.lib.vpz_decode_excerpts_device_conv
    args = (ctx._h, nf, ptrs, lens, n, file_of.ctypes.data, start.ctypes.data, count.ctypes.data, int(bool(clip)),
            fmt if conv is None else C.byref(conv))
    total = None
    if out is None:
        total = ctx.check(fn(*args, None, 0, offsets.ctypes.data, got.ctypes.data, None))
    buf, ptr, elems, handle = _device_out(ctx, out, total, dtype, stream)
    total = ctx.check(fn(*args, ptr, elems, offsets.ctypes.data, got.ctypes.data, handle))
    return buf[:total], offsets, got


class Corpus:
    """vpz_corpus: container images opened once (page scan, headers, setup tables, seek index, total samples) and
    cut into excerpt batches many times, each call costing only its excerpts' planning and decoding.

    files: list of bytes / uint8 arrays.  copy=False keeps references to the caller's buffers, which must not change
    while the corpus is open; copy=True makes the library keep its own copy.  close() (or dropping the corpus) frees
    its device memory; closing the context closes its open corpora first.
    .channels, .sample_rates and .samples (TotalSamples) are per-file numpy arrays, for drawing crops uniformly."""

    def __init__(self, ctx, files, copy=False):
        self.ctx = ctx
        self._h = None
        keep = [_u8(f) for f in files]
        n = len(keep)
        ptrs = (C.c_void_p * max(n, 1))(*[k[1] for k in keep])
        lens = (C.c_size_t * max(n, 1))(*[k[2] for k in keep])
        h = C.c_void_p()
        ctx.check(ctx.lib.vpz_corpus_open(ctx._h, n, ptrs, lens, int(bool(copy)), C.byref(h)))
        self._h = h
        self._keep = None if copy else keep
        ctx._corpora.add(self)
        self.channels = np.zeros(n, np.int32)
        self.sample_rates = np.zeros(n, np.int32)
        self.samples = np.zeros(n, np.int64)
        ctx.check(ctx.lib.vpz_corpus_info(h, self.channels.ctypes.data, self.sample_rates.ctypes.data,
                                          self.samples.ctypes.data))

    def __len__(self):
        return self.samples.size

    @property
    def device_bytes(self):
        """Bytes of device memory the corpus holds (its images)."""
        return int(self.ctx.lib.vpz_corpus_device_bytes(self._h)) if self._h else 0

    def close(self):
        """Frees the device images and the setup references; Context.close() closes its open corpora first."""
        if self._h:
            self.ctx.lib.vpz_corpus_close(self._h)
            self._h = None
            self._keep = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):   # a dropped corpus gives its device memory back (its context is still open: it closes corpora first)
        try:
            self.close()
        except Exception:
            pass

    def excerpts(self, file_of, start, count, clip=True, dtype="float32", planar=True, out=None, stream=None,
                 sample_rate=None, channels=None):
        """vpz_corpus_excerpts_device: decode_excerpts_device on the corpus's files, same arguments after `files`
        and bitwise the same (buf, offsets, got)."""
        if not self._h:
            raise ValueError("corpus is closed")
        ctx = self.ctx
        file_of = np.ascontiguousarray(file_of, dtype=np.uint32)
        start = np.ascontiguousarray(start, dtype=np.int64)
        count = np.ascontiguousarray(count, dtype=np.int32)
        n = file_of.size
        offsets = np.zeros(n, np.int64)
        got = np.zeros(n, np.int32)
        fmt = _format(dtype, planar)
        conv = N.OutConv(fmt, int(sample_rate or 0), int(channels or 0))
        args = (self._h, n, file_of.ctypes.data, start.ctypes.data, count.ctypes.data, int(bool(clip)), C.byref(conv))
        total = None
        if out is None:
            total = ctx.check(ctx.lib.vpz_corpus_excerpts_device(*args, None, 0, offsets.ctypes.data, got.ctypes.data,
                                                                 None))
        buf, ptr, elems, handle = _device_out(ctx, out, total, dtype, stream)
        total = ctx.check(ctx.lib.vpz_corpus_excerpts_device(*args, ptr, elems, offsets.ctypes.data, got.ctypes.data,
                                                             handle))
        return buf[:total], offsets, got


PAGE_DTYPE = np.dtype([("offset", "<u4"), ("body_len", "<u4"), ("granule", "<i8"), ("serial", "<u4"), ("sequence", "<u4"),
                       ("flags", "u1"), ("segments", "u1"), ("is_resync", "u1"), ("is_continued", "u1"),
                       ("packet_count", "<u2"), ("reserved", "<u2")])


def scan_pages(ctx, datas):
    """vpz_scan_pages: the physical Ogg layer of many container images on the GPU (capture-pattern search, header
    parse, lacing sums, page CRC-32; Ogg/PageReaderBase.cs:41-84,286-361).  Returns a list with, per image,
    (pages: structured array of PAGE_DTYPE, waste_bits, crc_failures)."""
    n = len(datas)
    keep = [np.frombuffer(d, np.uint8) for d in datas]
    ptrs = (C.c_void_p * max(n, 1))(*[k.ctypes.data if k.size else None for k in keep])
    lens = (C.c_size_t * max(n, 1))(*[k.size for k in keep])
    first = np.zeros(n, np.uint32)
    count = np.zeros(n, np.uint32)
    waste = np.zeros(n, np.uint64)
    crcf = np.zeros(n, np.uint32)
    cap = sum(len(d) // 64 + 16 for d in datas) + 1
    pages = np.zeros(cap, PAGE_DTYPE)
    assert PAGE_DTYPE.itemsize == 32
    total = ctx.check(ctx.lib.vpz_scan_pages(ctx._h, n, ptrs, lens, pages.ctypes.data, cap, first.ctypes.data,
                                              count.ctypes.data, waste.ctypes.data, crcf.ctypes.data))
    assert total == int(count.sum())
    return [(pages[int(first[i]):int(first[i]) + int(count[i])].copy(), int(waste[i]), int(crcf[i])) for i in range(n)]


def page_end_granules(ctx, data, on_device):
    """vpz_debug_page_end_granules: the seek index of a container image's first logical stream (entry p = granules
    up to and including page p; PacketProvider.FillPageEndGranuleCache, Ogg/PacketProvider.cs:203-307), built on the
    GPU (raises VpzError(VPZ_E_UNSUPPORTED) for files that keep the host path) or by the host's packet walk."""
    buf = np.frombuffer(data, np.uint8)
    cap = len(data) // 27 + 16
    out = np.zeros(cap, np.int64)
    n = ctx.check(ctx.lib.vpz_debug_page_end_granules(ctx._h, buf.ctypes.data, buf.size, 1 if on_device else 0, out.ctypes.data, cap))
    return out[:n].copy()
