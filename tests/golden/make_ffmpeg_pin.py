#!/usr/bin/env python3
"""Generates tests/golden/ffmpeg_pin_<name>.npz: 16-bit PCM of the four TestFiles decoded by an INDEPENDENT
native Vorbis decoder (FFmpeg's `vorbis` decoder inside the libavcodec that ships in the
opencv-python-headless wheel of this image), driven through ctypes.

Why: the reference's own tests (NVorbis.Tests/AssetTest.cs:72-194, RepoTests.cs:5-9) pin the decoder
to "|diff| <= 2 LSB at 16 bit, 0 differing packets" against the system libvorbisfile.  Neither .NET
nor libvorbisfile exists here, so the same convention is applied with a different independent
decoder.  The packets fed to FFmpeg come from a minimal Ogg page splitter in THIS file (no oracle
code involved), so the pin is independent of the oracle's container layer as well.

The generated files are committed; tests never need libavcodec or this script at run time.  Each holds
the whole decode of one file as wrapping int16 second differences along time, split into a low-byte and a
high-byte plane (`encode`): these deflate far better than the PCM itself and keep every file under 1 MB;
two wrapping cumulative sums restore the PCM exactly.

Layout knowledge used (FFmpeg 8 / lavc 62 public structs): AVPacket.data @24, .size @32;
AVFrame.extended_data @96, .nb_samples @112, .format @116; AVCodecParameters.codec_type @0,
.codec_id @4, .extradata @16, .extradata_size @24.
"""
import ctypes as C
import glob
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
FILES = ["1test", "2test", "3test", "issue6test"]


def encode(q):
    """q [frames, channels] int16 -> {"lo", "hi"}: the byte planes of its second differences, [channels, frames]."""
    d = np.ascontiguousarray(q.T)
    for _ in range(2):
        d = np.diff(d, axis=1, prepend=np.int16(0)).astype(np.int16)
    u = d.view(np.uint16)
    return {"lo": (u & 0xFF).astype(np.uint8), "hi": (u >> 8).astype(np.uint8)}


def ogg_packets(data):
    """Packets of the first logical stream, assembled across pages (lacing < 255 ends a packet)."""
    pos, serial0, cur, out = 0, None, b"", []
    while pos + 27 <= len(data):
        assert data[pos:pos + 4] == b"OggS", pos
        nseg = data[pos + 26]
        serial = struct.unpack_from("<I", data, pos + 14)[0]
        lac = data[pos + 27:pos + 27 + nseg]
        body = pos + 27 + nseg
        if serial0 is None:
            serial0 = serial
        for v in lac:
            if serial == serial0:
                cur += data[body:body + v]
            body += v
            if v < 255 and serial == serial0:
                out.append(cur)
                cur = b""
        pos = body
    return out


def main():
    import cv2  # noqa: F401  -- importing it loads libavcodec and all of its private dependencies
    libdir = glob.glob(os.path.join(os.path.dirname(np.__file__), "..", "opencv_python_headless.libs"))[0]
    util = C.CDLL(glob.glob(os.path.join(libdir, "libavutil-*"))[0], mode=C.RTLD_GLOBAL)
    for dep in ("libswresample-*",):
        for p in glob.glob(os.path.join(libdir, dep)):
            C.CDLL(p, mode=C.RTLD_GLOBAL)
    avc = C.CDLL(glob.glob(os.path.join(libdir, "libavcodec-*"))[0], mode=C.RTLD_GLOBAL)
    vp = C.c_void_p
    avc.avcodec_find_decoder_by_name.restype = vp
    avc.avcodec_find_decoder_by_name.argtypes = [C.c_char_p]
    avc.avcodec_alloc_context3.restype = vp
    avc.avcodec_alloc_context3.argtypes = [vp]
    avc.avcodec_parameters_alloc.restype = vp
    avc.avcodec_parameters_to_context.argtypes = [vp, vp]
    avc.avcodec_open2.argtypes = [vp, vp, vp]
    avc.av_packet_alloc.restype = vp
    avc.avcodec_send_packet.argtypes = [vp, vp]
    avc.avcodec_receive_frame.argtypes = [vp, vp]
    util.av_frame_alloc.restype = vp
    util.av_frame_unref.argtypes = [vp]
    util.av_mallocz.restype = vp
    util.av_mallocz.argtypes = [C.c_size_t]
    print("lavc version %x" % avc.avcodec_version())
    codec = avc.avcodec_find_decoder_by_name(b"vorbis")
    assert codec, "no native vorbis decoder in this libavcodec"
    for name in FILES:
        data = open(os.path.join(ROOT, "tests", "data", name + ".ogg"), "rb").read()
        pk = ogg_packets(data)
        hdr, audio = pk[:3], pk[3:]
        assert len(hdr[0]) == 30
        extra = b"".join(struct.pack(">H", len(h)) + h for h in hdr)
        ctx = avc.avcodec_alloc_context3(codec)
        par = avc.avcodec_parameters_alloc()
        ex = util.av_mallocz(len(extra) + 64)
        C.memmove(ex, extra, len(extra))
        C.c_int.from_address(par + 0).value = 1          # AVMEDIA_TYPE_AUDIO
        C.c_int.from_address(par + 4).value = 0x15005    # AV_CODEC_ID_VORBIS
        C.c_void_p.from_address(par + 16).value = ex
        C.c_int.from_address(par + 24).value = len(extra)
        assert avc.avcodec_parameters_to_context(ctx, par) >= 0
        rc = avc.avcodec_open2(ctx, codec, None)
        assert rc >= 0, rc
        pkt = avc.av_packet_alloc()
        frame = util.av_frame_alloc()
        chunks = []
        keep = []
        for p in audio:
            buf = C.create_string_buffer(p + b"\0" * 64, len(p) + 64)
            keep.append(buf)
            C.c_void_p.from_address(pkt + 24).value = C.addressof(buf)
            C.c_int.from_address(pkt + 32).value = len(p)
            rc = avc.avcodec_send_packet(ctx, pkt)
            if rc < 0:
                print(name, "send_packet", rc, "len", len(p))
                continue
            while avc.avcodec_receive_frame(ctx, frame) >= 0:
                n = C.c_int.from_address(frame + 112).value
                fmt = C.c_int.from_address(frame + 116).value
                assert fmt == 8, fmt  # AV_SAMPLE_FMT_FLTP
                ext = C.c_void_p.from_address(frame + 96).value
                chans = []
                ch = 0
                while True:
                    ptr = C.c_void_p.from_address(ext + 8 * ch).value
                    if not ptr or ch >= 2 and len(chunks) and ch >= chunks[0].shape[1]:
                        break
                    chans.append(np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_float)), shape=(n,)).copy())
                    ch += 1
                    if ch >= 8:
                        break
                if n:
                    chunks.append(np.stack(chans, axis=1))
                util.av_frame_unref(frame)
        pcm = np.concatenate(chunks)
        q = np.clip((pcm * np.float32(32768.0)).astype(np.int64), -32768, 32767).astype(np.int16)
        print(name, pcm.shape, "rms %.5f" % float(np.sqrt((pcm.astype(np.float64) ** 2).mean())))
        np.savez_compressed(os.path.join(HERE, "ffmpeg_pin_%s.npz" % name), **encode(q))
        print("wrote ffmpeg_pin_%s.npz" % name)


if __name__ == "__main__":
    sys.exit(main())
