"""vorbispizza_b200 -- B200-native Vorbis decode path behind VorbisPizza's reader API.

Host-side mirror of the reference interface for this path (NVorbis/VorbisReader.cs,
NVorbis/Contracts/IStreamDecoder.cs) on top of the C ABI in include/vpz.h.  All compute happens in
the sm_100a kernels of libvpz.so; importing this package never falls back to a CPU decoder --
loading fails loudly when the library is missing and creating a Context fails when no B200 is
visible.
"""
from ._native import VpzError, load  # noqa: F401
from .api import (  # noqa: F401
    Batch,
    Context,
    Corpus,
    InvalidDataError,
    PreRollPacketError,
    SeekOutOfRangeError,
    SynthBatch,
    VorbisReader,
    decode_excerpts,
    decode_excerpts_device,
    decode_files,
    decode_files_device,
    scan_pages,
)

__all__ = ["Batch", "Context", "Corpus", "SynthBatch", "VorbisReader", "decode_files", "decode_excerpts", "decode_files_device",
           "decode_excerpts_device", "scan_pages", "VpzError", "InvalidDataError",
           "SeekOutOfRangeError", "PreRollPacketError", "load"]
