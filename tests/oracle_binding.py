"""ctypes binding of the CPU oracle (oracle/libvorbis_oracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package never imports this.
"""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB_PATH = os.path.join(ORACLE_DIR, "libvorbis_oracle.so")

VO_MAX_CH = 8


def build_oracle(force=False):
    srcs = [os.path.join(ORACLE_DIR, f) for f in os.listdir(ORACLE_DIR) if f.endswith((".c", ".h", ".inc"))]
    if (not force and os.path.exists(LIB_PATH)
            and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in srcs)):
        return LIB_PATH
    subprocess.check_call(["make", "-C", ORACLE_DIR, "-s"])
    return LIB_PATH


class PacketView(C.Structure):
    _fields_ = [("data", C.POINTER(C.c_uint8)), ("len", C.c_int32), ("is_resync", C.c_int32),
                ("is_eos", C.c_int32), ("granule", C.c_int64), ("page_index", C.c_int32),
                ("packet_index", C.c_int32)]


class PacketDump(C.Structure):
    _fields_ = [
        ("status", C.c_int32), ("mode", C.c_int32), ("block_flag", C.c_int32), ("block_size", C.c_int32),
        ("info", C.c_int32 * 6), ("bits_read", C.c_int32), ("is_short", C.c_int32),
        ("scalars", C.POINTER(C.c_int32)), ("scalars_cap", C.c_int32), ("scalars_n", C.c_int32),
        ("post_count", C.c_int32 * VO_MAX_CH),
        ("raw_posts", (C.c_int32 * 64) * VO_MAX_CH),
        ("final_y", (C.c_int32 * 64) * VO_MAX_CH),
        ("step_flags", (C.c_int32 * 64) * VO_MAX_CH),
        ("no_execute", C.c_int32 * VO_MAX_CH),
        ("classes", C.POINTER(C.c_int32)), ("classes_cap", C.c_int32), ("classes_n", C.c_int32),
        ("residue", C.POINTER(C.c_float)), ("spectrum", C.POINTER(C.c_float)), ("imdct", C.POINTER(C.c_float)),
    ]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build_oracle()
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.vo_open.restype = vp
    L.vo_open.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]
    L.vo_close.argtypes = [vp]
    for name in ("vo_channels", "vo_sample_rate", "vo_page_count", "vo_crc_failures", "vo_comment_count",
                 "vo_has_clipped", "vo_is_end_of_stream", "vo_audio_packet_count", "vo_book_count"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = [vp]
    L.vo_block_size.restype = C.c_int
    L.vo_block_size.argtypes = [vp, C.c_int]
    L.vo_bitrate.restype = C.c_int
    L.vo_bitrate.argtypes = [vp, C.c_int]
    for name in ("vo_container_bits", "vo_waste_bits", "vo_sample_position", "vo_total_samples"):
        getattr(L, name).restype = C.c_int64
        getattr(L, name).argtypes = [vp]
    L.vo_page_end_granules.restype = C.c_int
    L.vo_page_end_granules.argtypes = [vp, C.c_void_p, C.c_int]
    L.vo_vendor.restype = C.c_void_p
    L.vo_vendor.argtypes = [vp, C.POINTER(C.c_int)]
    L.vo_comment.restype = C.c_void_p
    L.vo_comment.argtypes = [vp, C.c_int, C.POINTER(C.c_int)]
    L.vo_header_packet.restype = C.c_void_p
    L.vo_header_packet.argtypes = [vp, C.c_int, C.POINTER(C.c_int)]
    L.vo_set_clip.argtypes = [vp, C.c_int]
    L.vo_read.restype = C.c_int
    L.vo_read.argtypes = [vp, C.c_void_p, C.c_int]
    L.vo_read_planar.restype = C.c_int
    L.vo_read_planar.argtypes = [vp, C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.vo_seek.restype = C.c_int
    L.vo_seek.argtypes = [vp, C.c_int64]
    L.vo_audio_packet.restype = C.c_int
    L.vo_audio_packet.argtypes = [vp, C.c_int, C.POINTER(PacketView)]
    L.vo_book_info.restype = C.c_int
    L.vo_book_info.argtypes = [vp, C.c_int] + [C.POINTER(C.c_int)] * 6
    L.vo_book_lengths.restype = C.c_int
    L.vo_book_lengths.argtypes = [vp, C.c_int, C.c_void_p]
    L.vo_book_lookup.restype = C.c_void_p
    L.vo_book_lookup.argtypes = [vp, C.c_int, C.POINTER(C.c_int)]
    L.vo_book_decode.restype = C.c_int
    L.vo_book_decode.argtypes = [vp, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int)]
    L.vo_book_kraft.restype = C.c_double
    L.vo_book_kraft.argtypes = [vp, C.c_int]
    L.vo_decode_packet_dump.restype = C.c_int
    L.vo_decode_packet_dump.argtypes = [vp, C.c_void_p, C.c_int, C.POINTER(PacketDump)]
    L.vo_imdct.restype = C.c_int
    L.vo_imdct.argtypes = [C.c_void_p, C.c_int]
    L.vo_window_slope.argtypes = [C.c_void_p, C.c_int]
    L.vo_inverse_db_table.restype = C.c_void_p
    L.vo_crc_ogg.restype = C.c_uint32
    L.vo_crc_ogg.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32]
    L.vo_packet_info.argtypes = [C.c_int] * 5 + [C.POINTER(C.c_int32)]
    L.vo_bench_decode.restype = C.c_int64
    L.vo_bench_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
    _lib = L
    return L


class OracleError(Exception):
    def __init__(self, code):
        super().__init__("oracle error %d" % code)
        self.code = code


class OracleStream:
    """Mirror of VorbisReader/StreamDecoder over the oracle."""

    def __init__(self, data: bytes):
        L = lib()
        self._buf = np.frombuffer(data, dtype=np.uint8).copy()
        err = C.c_int(0)
        self._h = L.vo_open(self._buf.ctypes.data, self._buf.size, C.byref(err))
        if not self._h:
            raise OracleError(err.value)
        self.channels = L.vo_channels(self._h)
        self.sample_rate = L.vo_sample_rate(self._h)
        self.block_sizes = (L.vo_block_size(self._h, 0), L.vo_block_size(self._h, 1))

    def close(self):
        if self._h:
            lib().vo_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def page_end_granules(self):
        """PacketProvider's page-end granule cache, filled to the end of the stream (raises OracleError)."""
        out = np.zeros(1 << 16, np.int64)
        n = lib().vo_page_end_granules(self._h, out.ctypes.data, out.size)
        if n < 0:
            raise OracleError(n)
        return out[:n].copy()

    # --- properties
    @property
    def total_samples(self):
        return lib().vo_total_samples(self._h)

    @property
    def sample_position(self):
        return lib().vo_sample_position(self._h)

    @property
    def has_clipped(self):
        return bool(lib().vo_has_clipped(self._h))

    @property
    def is_end_of_stream(self):
        return bool(lib().vo_is_end_of_stream(self._h))

    def set_clip(self, clip):
        lib().vo_set_clip(self._h, int(clip))

    def bitrates(self):
        return tuple(lib().vo_bitrate(self._h, i) for i in range(3))

    def vendor(self):
        n = C.c_int(0)
        p = lib().vo_vendor(self._h, C.byref(n))
        return C.string_at(p, n.value)

    def comments(self):
        out = []
        for i in range(lib().vo_comment_count(self._h)):
            n = C.c_int(0)
            p = lib().vo_comment(self._h, i, C.byref(n))
            out.append(C.string_at(p, n.value))
        return out

    def header_packet(self, which):
        n = C.c_int(0)
        p = lib().vo_header_packet(self._h, which, C.byref(n))
        return C.string_at(p, n.value)

    def page_count(self):
        return lib().vo_page_count(self._h)

    def crc_failures(self):
        return lib().vo_crc_failures(self._h)

    def waste_bits(self):
        return lib().vo_waste_bits(self._h)

    # --- decode
    def read(self, buf: np.ndarray):
        assert buf.dtype == np.float32 and buf.flags.c_contiguous
        return lib().vo_read(self._h, buf.ctypes.data, buf.size)

    def read_planar(self, buf: np.ndarray, samples_to_read, channel_stride):
        return lib().vo_read_planar(self._h, buf.ctypes.data, buf.size, samples_to_read, channel_stride)

    def seek(self, pos):
        rc = lib().vo_seek(self._h, int(pos))
        if rc < 0:
            raise OracleError(rc)

    def decode_all(self, chunk_floats=48000):
        """TestApp-style drain (TestApp/Program.cs:42,155): returns [samples, channels] and the
        list of per-call return counts; stops on 0 or on the reference-fault code."""
        ch = self.channels
        chunk_floats -= chunk_floats % ch
        buf = np.empty(chunk_floats, dtype=np.float32)
        out, counts = [], []
        fault = 0
        while True:
            n = self.read(buf)
            if n < 0:
                fault = n
                break
            if n == 0:
                break
            counts.append(n)
            out.append(buf[: n * ch].copy())
        pcm = np.concatenate(out).reshape(-1, ch) if out else np.zeros((0, ch), np.float32)
        return pcm, counts, fault

    # --- packets
    def audio_packets(self):
        L = lib()
        n = L.vo_audio_packet_count(self._h)
        res = []
        v = PacketView()
        for i in range(n):
            L.vo_audio_packet(self._h, i, C.byref(v))
            res.append(dict(data=C.string_at(v.data, v.len) if v.len else b"", is_resync=bool(v.is_resync),
                            is_eos=bool(v.is_eos), granule=v.granule, page_index=v.page_index,
                            packet_index=v.packet_index))
        return res

    # --- books
    def book_count(self):
        return lib().vo_book_count(self._h)

    def book_info(self, b):
        vals = [C.c_int(0) for _ in range(6)]
        lib().vo_book_info(self._h, b, *[C.byref(v) for v in vals])
        keys = ("dims", "entries", "max_bits", "map_type", "prefix_bits", "overflow_count")
        return dict(zip(keys, [v.value for v in vals]))

    def book_lengths(self, b):
        n = self.book_info(b)["entries"]
        a = np.zeros(n, dtype=np.int32)
        lib().vo_book_lengths(self._h, b, a.ctypes.data)
        return a

    def book_lookup(self, b):
        n = C.c_int(0)
        p = lib().vo_book_lookup(self._h, b, C.byref(n))
        if not p or n.value == 0:
            return np.zeros(0, np.float32)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=(n.value,)).copy()

    def book_kraft(self, b):
        return lib().vo_book_kraft(self._h, b)

    def book_decode(self, b, data: bytes, bitpos: int):
        arr = np.frombuffer(data, dtype=np.uint8)
        pos = C.c_int64(bitpos)
        short = C.c_int(0)
        v = lib().vo_book_decode(self._h, b, arr.ctypes.data if arr.size else None, arr.size, C.byref(pos),
                                 C.byref(short))
        return v, pos.value, bool(short.value)

    def dump_packet(self, data: bytes, want_floats=True, scalars_cap=8192, classes_cap=8192):
        """Returns a dict of every integer stage (+ float stages) for one audio packet."""
        d = PacketDump()
        scal = np.zeros(scalars_cap, np.int32)
        cls = np.zeros(classes_cap, np.int32)
        d.scalars = scal.ctypes.data_as(C.POINTER(C.c_int32))
        d.scalars_cap = scalars_cap
        d.classes = cls.ctypes.data_as(C.POINTER(C.c_int32))
        d.classes_cap = classes_cap
        ch = self.channels
        n1 = self.block_sizes[1]
        res = spec = imd = None
        if want_floats:
            res = np.zeros(ch * n1 // 2, np.float32)
            spec = np.zeros(ch * n1 // 2, np.float32)
            imd = np.zeros(ch * n1, np.float32)
            d.residue = res.ctypes.data_as(C.POINTER(C.c_float))
            d.spectrum = spec.ctypes.data_as(C.POINTER(C.c_float))
            d.imdct = imd.ctypes.data_as(C.POINTER(C.c_float))
        arr = np.frombuffer(data, dtype=np.uint8)
        rc = lib().vo_decode_packet_dump(self._h, arr.ctypes.data if arr.size else None, arr.size, C.byref(d))
        out = dict(rc=rc, status=d.status, mode=d.mode, block_flag=d.block_flag, block_size=d.block_size,
                   info=list(d.info), bits_read=d.bits_read, is_short=d.is_short,
                   scalars=scal[: min(d.scalars_n, scalars_cap)].copy(), scalars_n=d.scalars_n,
                   classes=cls[: min(d.classes_n, classes_cap)].copy(), classes_n=d.classes_n,
                   post_count=[d.post_count[c] for c in range(ch)],
                   raw_posts=np.array([list(d.raw_posts[c]) for c in range(ch)], np.int32),
                   final_y=np.array([list(d.final_y[c]) for c in range(ch)], np.int32),
                   step_flags=np.array([list(d.step_flags[c]) for c in range(ch)], np.int32),
                   no_execute=[d.no_execute[c] for c in range(ch)])
        if want_floats and d.status == 0:
            n = d.block_size
            out["residue"] = res[: ch * n // 2].reshape(ch, n // 2).copy()
            out["spectrum"] = spec[: ch * n // 2].reshape(ch, n // 2).copy()
            out["imdct"] = imd[: ch * n].reshape(ch, n).copy()
        return out


def imdct(spectrum: np.ndarray) -> np.ndarray:
    """Mdct.Reverse on n/2 coefficients -> n samples."""
    n = spectrum.size * 2
    buf = np.zeros(n, np.float32)
    buf[: n // 2] = spectrum
    rc = lib().vo_imdct(buf.ctypes.data, n)
    if rc:
        raise OracleError(rc)
    return buf


def window_slope(n: int) -> np.ndarray:
    w = np.zeros(n, np.float32)
    lib().vo_window_slope(w.ctypes.data, n)
    return w


def inverse_db_table() -> np.ndarray:
    p = lib().vo_inverse_db_table()
    return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=(256,)).copy()


def crc_ogg(data: bytes, crc=0) -> int:
    arr = np.frombuffer(data, dtype=np.uint8)
    return lib().vo_crc_ogg(arr.ctypes.data if arr.size else None, arr.size, crc)


def packet_info(size0, size1, block_flag, prev_flag, next_flag):
    a = (C.c_int32 * 6)()
    lib().vo_packet_info(size0, size1, int(block_flag), int(prev_flag), int(next_flag), a)
    return list(a)


_bench_libs = {}


def bench_lib(native=False):
    """The oracle library used for TIMING: the portable -O2 build, or (native=True) the same sources built
    -O3 -march=native on THIS machine (oracle/Makefile `native`; rebuilt on every call site's first use so a
    binary tuned for another CPU is never run).  The native build goes to a temporary directory, removed once
    the library is loaded, so the source tree may be read-only.  None when that build is not possible here."""
    key = bool(native)
    if key in _bench_libs:
        return _bench_libs[key]
    if not native:
        L = lib()
    else:
        tmp = tempfile.mkdtemp(prefix="vpz_oracle_native_")
        try:
            subprocess.check_call(["make", "-C", ORACLE_DIR, "-s", "-B", "native", "NATIVE_DIR=" + tmp],
                                  stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            L = C.CDLL(os.path.join(tmp, "libvorbis_oracle.so"))
        except Exception:
            L = None
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    if L is not None:
        L.vo_bench_decode.restype = C.c_int64
        L.vo_bench_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
        L.vo_bench_excerpts.restype = C.c_int64
        L.vo_bench_excerpts.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_int, C.POINTER(C.c_double)]
    _bench_libs[key] = L
    return L


def bench_decode(files, njobs, nthreads, native=False):
    """Host-core baseline: decodes njobs whole streams (job j = file j % len(files)) on nthreads threads
    inside the oracle, streams handed out by a shared cursor; returns (channel_samples, seconds)."""
    L = bench_lib(native)
    if L is None:
        return None
    keep = [np.frombuffer(f, np.uint8) for f in files]
    ptrs = (C.c_void_p * len(keep))(*[k.ctypes.data for k in keep])
    lens = (C.c_size_t * len(keep))(*[k.size for k in keep])
    sec = C.c_double(0)
    n = L.vo_bench_decode(ptrs, lens, len(keep), njobs, nthreads, C.byref(sec))
    return n, sec.value


def bench_excerpts(files, file_of, start, count, nthreads, native=False):
    """Host-core baseline of the random-access batch: SeekTo(start[i]) + read count[i] samples per channel of
    files[file_of[i]], one open reader per (thread, file); returns (channel_samples delivered, seconds)."""
    L = bench_lib(native)
    if L is None:
        return None
    keep = [np.frombuffer(f, np.uint8) for f in files]
    ptrs = (C.c_void_p * len(keep))(*[k.ctypes.data for k in keep])
    lens = (C.c_size_t * len(keep))(*[k.size for k in keep])
    file_of = np.ascontiguousarray(file_of, np.uint32)
    start = np.ascontiguousarray(start, np.int64)
    count = np.ascontiguousarray(count, np.int32)
    sec = C.c_double(0)
    n = L.vo_bench_excerpts(ptrs, lens, len(keep), int(file_of.size), file_of.ctypes.data, start.ctypes.data,
                            count.ctypes.data, nthreads, C.byref(sec))
    return n, sec.value


def bench_imdct_ola(spectra, flags, channels, size0, size1, nthreads, native=False):
    """Host-core baseline of BASELINE config 3: Mdct.Reverse + OverlapBuffers + interleaved clipped store on the
    synthetic streams (flags [n_streams][n_blocks], spectra back to back); returns (channel_samples, seconds)."""
    L = bench_lib(native)
    if L is None:
        return None
    L.vo_bench_imdct_ola.restype = C.c_int64
    L.vo_bench_imdct_ola.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.POINTER(C.c_double), C.POINTER(C.c_double)]
    spectra = np.ascontiguousarray(spectra, np.float32)
    flags = np.ascontiguousarray(flags, np.uint8)
    sec, chk = C.c_double(0), C.c_double(0)
    n = L.vo_bench_imdct_ola(spectra.ctypes.data, flags.ctypes.data, flags.shape[0], flags.shape[1], channels, size0, size1,
                             nthreads, C.byref(sec), C.byref(chk))
    return n, sec.value, chk.value
