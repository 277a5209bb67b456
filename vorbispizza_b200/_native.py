"""ctypes binding of libvpz.so (include/vpz.h).

The product path is the CUDA library built in-tree at ``vorbispizza_b200/libvpz.so``; there is no
CPU fallback: if the library is missing or no sm_100 GPU is visible, loading / context creation
raises.  ``load(path)`` lets the CPU-only test-suite point the same binding at the emulated test
build (tests/emu/libvpz_emu.so) -- never done by product code.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB = os.path.join(_HERE, "libvpz.so")

VPZ_OK = 0
VPZ_E_INVALID_DATA = -1
VPZ_E_ARGUMENT = -2
VPZ_E_SEEK_RANGE = -3
VPZ_E_PREROLL = -4
VPZ_E_UNSUPPORTED = -5
VPZ_E_CUDA = -6
VPZ_E_NOMEM = -7
VPZ_E_DISPOSED = -8
VPZ_E_INVALID_OP = -9
VPZ_E_NO_DEVICE = -10
VPZ_E_REF_FAULT = -11

DUMP_MAX_CH = 8

VPZ_OUT_S16 = 1      # format bits of the *_device bulk calls; 0 = fp32 interleaved
VPZ_OUT_PLANAR = 2


class SetupInfo(C.Structure):
    _fields_ = [("channels", C.c_int32), ("sample_rate", C.c_int32), ("bitrate_upper", C.c_int32),
                ("bitrate_nominal", C.c_int32), ("bitrate_lower", C.c_int32), ("block_size0", C.c_int32),
                ("block_size1", C.c_int32), ("n_books", C.c_int32), ("n_floors", C.c_int32),
                ("n_residues", C.c_int32), ("n_mappings", C.c_int32), ("n_modes", C.c_int32),
                ("max_codeword_bits", C.c_int32), ("table_bytes", C.c_uint64)]


class OutConv(C.Structure):   # vpz_out_conv
    _fields_ = [("format", C.c_int32), ("sample_rate", C.c_int32), ("channels", C.c_int32)]


class PacketDump(C.Structure):
    _fields_ = [("status", C.c_int32), ("mode", C.c_int32), ("block_size", C.c_int32), ("info", C.c_int32 * 6),
                ("bits_read", C.c_int32), ("exec_mask", C.c_int32), ("no_execute_mask", C.c_int32),
                ("scalars_n", C.c_int32), ("classes_n", C.c_int32), ("post_count", C.c_int32 * DUMP_MAX_CH),
                ("raw_posts", (C.c_int32 * 64) * DUMP_MAX_CH), ("final_y", (C.c_int32 * 64) * DUMP_MAX_CH),
                ("step_flags", (C.c_int32 * 64) * DUMP_MAX_CH)]


# name -> (restype, argtypes); every symbol include/vpz.h declares
_P = C.c_void_p
_SIGS = {
    "vpz_strerror": (C.c_char_p, [C.c_int]),
    "vpz_last_error": (C.c_char_p, [_P]),
    "vpz_version": (C.c_char_p, []),
    "vpz_ctx_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "vpz_ctx_destroy": (None, [_P]),
    "vpz_device_count": (C.c_int, []),
    "vpz_ctx_set": (C.c_int, [_P, C.c_char_p, C.c_int]),
    "vpz_ctx_mark": (C.c_int, [_P, C.c_int]),
    "vpz_ctx_elapsed_ms": (C.c_float, [_P, C.c_int, C.c_int]),
    "vpz_ctx_kernel_launches": (C.c_int64, [_P]),
    "vpz_setup_create": (C.c_int, [_P, _P, C.c_size_t, _P, C.c_size_t, C.POINTER(_P)]),
    "vpz_setup_release": (None, [_P]),
    "vpz_setup_get_info": (C.c_int, [_P, C.POINTER(SetupInfo)]),
    "vpz_packet_info": (C.c_int, [_P, _P, C.c_size_t, C.POINTER(C.c_int32)]),
    "vpz_batch_create": (C.c_int, [_P, C.POINTER(_P)]),
    "vpz_batch_destroy": (None, [_P]),
    "vpz_batch_reset": (C.c_int, [_P]),
    "vpz_batch_add_run": (C.c_int, [_P, _P, _P, _P, C.c_uint32, _P]),
    "vpz_batch_run_samples": (C.c_int64, [_P, C.c_int]),
    "vpz_batch_run_channels": (C.c_int, [_P, C.c_int]),
    "vpz_batch_run_status": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int32)]),
    "vpz_batch_run_packet_samples": (C.c_int, [_P, C.c_int, _P]),
    "vpz_batch_total_floats": (C.c_int64, [_P]),
    "vpz_batch_total_packets": (C.c_int64, [_P]),
    "vpz_batch_total_bytes": (C.c_int64, [_P]),
    "vpz_batch_upload": (C.c_int, [_P]),
    "vpz_batch_decode": (C.c_int, [_P, C.c_int]),
    "vpz_batch_sync": (C.c_int, [_P]),
    "vpz_batch_has_clipped": (C.c_int, [_P]),
    "vpz_batch_read_run": (C.c_int, [_P, C.c_int, _P]),
    "vpz_batch_read_all": (C.c_int, [_P, _P]),
    "vpz_batch_run_offset": (C.c_int64, [_P, C.c_int]),
    "vpz_batch_device_pcm": (_P, [_P]),
    "vpz_batch_last_ms": (C.c_float, [_P, C.c_int, C.POINTER(C.c_int)]),
    "vpz_transfer_bytes": (C.c_uint64, [C.c_int]),
    "vpz_host_alloc": (_P, [C.c_size_t]),
    "vpz_host_free": (None, [_P]),
    "vpz_debug_decode_packet": (C.c_int, [_P, _P, _P, C.c_size_t, C.POINTER(PacketDump), _P, C.c_int32, _P,
                                          C.c_int32, _P, _P, _P]),
    "vpz_synth_create": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_uint32, _P, _P, C.POINTER(_P)]),
    "vpz_reader_open_memory": (C.c_int, [_P, _P, C.c_size_t, C.c_int, C.POINTER(_P)]),
    "vpz_reader_close": (None, [_P]),
    "vpz_reader_stream_count": (C.c_int, [_P]),
    "vpz_reader_stream_index": (C.c_int, [_P]),
    "vpz_reader_switch_stream": (C.c_int, [_P, C.c_int]),
    "vpz_reader_find_next_stream": (C.c_int, [_P]),
    "vpz_reader_can_seek": (C.c_int, [_P]),
    "vpz_reader_channels": (C.c_int, [_P]),
    "vpz_reader_sample_rate": (C.c_int, [_P]),
    "vpz_reader_bitrate": (C.c_int, [_P, C.c_int]),
    "vpz_reader_stream_serial": (C.c_int, [_P]),
    "vpz_reader_total_samples": (C.c_int64, [_P]),
    "vpz_reader_sample_position": (C.c_int64, [_P]),
    "vpz_reader_is_end_of_stream": (C.c_int, [_P]),
    "vpz_reader_has_clipped": (C.c_int, [_P]),
    "vpz_reader_get_clip": (C.c_int, [_P]),
    "vpz_reader_set_clip": (None, [_P, C.c_int]),
    "vpz_reader_container_overhead_bits": (C.c_int64, [_P]),
    "vpz_reader_container_waste_bits": (C.c_int64, [_P]),
    "vpz_reader_vendor": (_P, [_P, C.POINTER(C.c_int)]),
    "vpz_reader_comment_count": (C.c_int, [_P]),
    "vpz_reader_comment": (_P, [_P, C.c_int, C.POINTER(C.c_int)]),
    "vpz_reader_read": (C.c_int, [_P, _P, C.c_int]),
    "vpz_reader_read_planar": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int]),
    "vpz_reader_seek": (C.c_int, [_P, C.c_int64, C.c_int]),
    "vpz_reader_set_lookahead": (C.c_int, [_P, C.c_int]),
    "vpz_reader_audio_packet_count": (C.c_int, [_P]),
    "vpz_reader_audio_packet": (C.c_int, [_P, C.c_int, C.POINTER(_P), C.POINTER(C.c_uint32), C.POINTER(C.c_int64),
                                          C.POINTER(C.c_int32)]),
    "vpz_reader_header_packet": (_P, [_P, C.c_int, C.POINTER(C.c_uint32)]),
    "vpz_reader_setup": (_P, [_P]),
    "vpz_decode_files": (C.c_int64, [_P, C.c_uint32, _P, _P, C.c_int, _P, C.c_size_t, _P]),
    "vpz_decode_files_s16": (C.c_int64, [_P, C.c_uint32, _P, _P, C.c_int, _P, C.c_size_t, _P]),
    "vpz_decode_excerpts": (C.c_int64, [_P, C.c_uint32, _P, _P, C.c_uint32, _P, _P, _P, C.c_int, _P, C.c_size_t, _P, _P]),
    "vpz_decode_files_device": (C.c_int64, [_P, C.c_uint32, _P, _P, C.c_int, C.c_int, _P, C.c_size_t, _P, _P]),
    "vpz_decode_excerpts_device": (C.c_int64, [_P, C.c_uint32, _P, _P, C.c_uint32, _P, _P, _P, C.c_int, C.c_int, _P,
                                               C.c_size_t, _P, _P, _P]),
    "vpz_decode_files_device_conv": (C.c_int64, [_P, C.c_uint32, _P, _P, C.c_int, C.POINTER(OutConv), _P, C.c_size_t,
                                                 _P, _P, _P]),
    "vpz_decode_excerpts_device_conv": (C.c_int64, [_P, C.c_uint32, _P, _P, C.c_uint32, _P, _P, _P, C.c_int,
                                                    C.POINTER(OutConv), _P, C.c_size_t, _P, _P, _P]),
    "vpz_corpus_open": (C.c_int, [_P, C.c_uint32, _P, _P, C.c_int, C.POINTER(_P)]),
    "vpz_corpus_close": (None, [_P]),
    "vpz_corpus_info": (C.c_int64, [_P, _P, _P, _P]),
    "vpz_corpus_device_bytes": (C.c_uint64, [_P]),
    "vpz_corpus_excerpts_device": (C.c_int64, [_P, C.c_uint32, _P, _P, _P, C.c_int, C.POINTER(OutConv), _P, C.c_size_t,
                                               _P, _P, _P]),
    "vpz_debug_page_end_granules":(C.c_int64, [_P, _P, C.c_size_t, C.c_int, _P, C.c_size_t]),
    "vpz_scan_pages": (C.c_int64, [_P, C.c_uint32, _P, _P, _P, C.c_size_t, _P, _P, _P, _P]),
}

EXPORTED_SYMBOLS = tuple(sorted(_SIGS))

_libs = {}


class VpzError(Exception):
    def __init__(self, code, text=""):
        self.code = code
        super().__init__("vpz error %d%s" % (code, (": " + text) if text else ""))


def load(path=None):
    """Loads libvpz.so (default: the in-tree CUDA build) and declares every prototype."""
    path = os.path.abspath(path or DEFAULT_LIB)
    if path in _libs:
        return _libs[path]
    if not os.path.exists(path):
        raise ImportError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  vorbispizza_b200 has no CPU fallback." % path)
    lib = C.CDLL(path)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    _libs[path] = lib
    return lib
