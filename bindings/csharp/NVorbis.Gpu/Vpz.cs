// P/Invoke surface of libvpz.so: one declaration per prototype of include/vpz.h (same order).
using System;
using System.IO;
using System.Runtime.InteropServices;

namespace NVorbis.Gpu
{
    [StructLayout(LayoutKind.Sequential)]
    internal struct VpzSetupInfo
    {
        public int Channels, SampleRate, BitrateUpper, BitrateNominal, BitrateLower, BlockSize0, BlockSize1;
        public int Books, Floors, Residues, Mappings, Modes, MaxCodewordBits;
        public ulong TableBytes;
    }

    [StructLayout(LayoutKind.Sequential)]
    internal struct VpzOutConv      // vpz_out_conv
    {
        public int Format, SampleRate, Channels;
    }

    [StructLayout(LayoutKind.Sequential)]
    public struct VpzPageInfo       // vpz_page_info, 32 bytes
    {
        public uint Offset, BodyLength, GranuleLo, GranuleHi, Serial, Sequence;
        public byte Flags, Segments, IsResync, IsContinued;
        public ushort PacketCount, Reserved;
        public long Granule => (long)(((ulong)GranuleHi << 32) | GranuleLo);
    }

    internal static unsafe partial class Vpz
    {
        const string Lib = "vpz";   // libvpz.so next to NVorbis.dll

        // vpz_status (include/vpz.h:36-52)
        internal const int Ok = 0, InvalidData = -1, Argument = -2, SeekRange = -3, PreRoll = -4, Unsupported = -5,
                           Cuda = -6, NoMem = -7, Disposed = -8, InvalidOp = -9, NoDevice = -10, RefFault = -11;

        /// <summary>Negative vpz_status -> the exception the reference throws at the same place.</summary>
        internal static void Check(long rc, IntPtr ctx)
        {
            if (rc >= 0) return;
            string msg = ctx != IntPtr.Zero ? Marshal.PtrToStringUTF8(vpz_last_error(ctx)) ?? "" : "";
            if (msg.Length == 0) msg = Marshal.PtrToStringUTF8(vpz_strerror((int)rc)) ?? "";
            throw (int)rc switch
            {
                InvalidData => new InvalidDataException(msg),            // StreamDecoder.cs:77,84,313,330,338,351,734
                Argument => new ArgumentException(msg),                  // StreamDecoder.cs:423-430,825,842
                SeekRange => new SeekOutOfRangeException(),              // StreamDecoder.cs:861
                PreRoll => new PreRollPacketException(),                 // StreamDecoder.cs:874
                Unsupported => new NotSupportedException(msg),           // block size < 256, > 8 channels, ...
                Disposed => new ObjectDisposedException(nameof(VorbisReader)),   // StreamDecoder.cs:401
                InvalidOp => new InvalidOperationException(msg),         // StreamDecoder.cs:822
                NoDevice => new PlatformNotSupportedException("no sm_100 GPU: libvpz has no CPU path"),
                NoMem => new OutOfMemoryException(msg),
                RefFault => new ArgumentOutOfRangeException(msg),        // what the reference itself throws (SURVEY quirk Q4)
                _ => new ExternalException(msg, (int)rc),
            };
        }

        [LibraryImport(Lib)] internal static partial IntPtr vpz_strerror(int code);
        [LibraryImport(Lib)] internal static partial IntPtr vpz_last_error(IntPtr ctx);
        [LibraryImport(Lib)] internal static partial IntPtr vpz_version();

        // ---- context
        [LibraryImport(Lib)] internal static partial int vpz_ctx_create(int device, out IntPtr ctx);
        [LibraryImport(Lib)] internal static partial void vpz_ctx_destroy(IntPtr ctx);
        [LibraryImport(Lib)] internal static partial int vpz_device_count();
        [LibraryImport(Lib, StringMarshalling = StringMarshalling.Utf8)] internal static partial int vpz_ctx_set(IntPtr ctx, string key, int value);
        [LibraryImport(Lib)] internal static partial int vpz_ctx_mark(IntPtr ctx, int slot);
        [LibraryImport(Lib)] internal static partial float vpz_ctx_elapsed_ms(IntPtr ctx, int slotA, int slotB);
        [LibraryImport(Lib)] internal static partial long vpz_ctx_kernel_launches(IntPtr ctx);

        // ---- setup: StreamDecoder.LoadStreamHeader + LoadBooks (StreamDecoder.cs:213-355)
        [LibraryImport(Lib)] internal static partial int vpz_setup_create(IntPtr ctx, byte* idPkt, nuint idLen, byte* setupPkt, nuint setupLen, out IntPtr setup);
        [LibraryImport(Lib)] internal static partial void vpz_setup_release(IntPtr setup);
        [LibraryImport(Lib)] internal static partial int vpz_setup_get_info(IntPtr setup, out VpzSetupInfo info);
        // Mode.GetPacketInfo (Mode.cs:30-66): info = {Length, LeftUseSize1, LeftStart, LeftEnd, RightStart, RightEnd}
        [LibraryImport(Lib)] internal static partial int vpz_packet_info(IntPtr setup, byte* pkt, nuint len, int* info6);

        // ---- batch: Mode.Decode -> Mapping.DecodePacket -> Mdct.Reverse -> OverlapBuffers -> StoreInterleaved
        [LibraryImport(Lib)] internal static partial int vpz_batch_create(IntPtr ctx, out IntPtr batch);
        [LibraryImport(Lib)] internal static partial void vpz_batch_destroy(IntPtr batch);
        [LibraryImport(Lib)] internal static partial int vpz_batch_reset(IntPtr batch);
        [LibraryImport(Lib)] internal static partial int vpz_batch_add_run(IntPtr batch, IntPtr setup, byte* bytes, uint* offsets, uint nPkts, int* trim);
        [LibraryImport(Lib)] internal static partial long vpz_batch_run_samples(IntPtr batch, int run);
        [LibraryImport(Lib)] internal static partial int vpz_batch_run_channels(IntPtr batch, int run);
        [LibraryImport(Lib)] internal static partial int vpz_batch_run_status(IntPtr batch, int run, out int stopPacket);
        [LibraryImport(Lib)] internal static partial int vpz_batch_run_packet_samples(IntPtr batch, int run, int* counts);
        [LibraryImport(Lib)] internal static partial long vpz_batch_total_floats(IntPtr batch);
        [LibraryImport(Lib)] internal static partial long vpz_batch_total_packets(IntPtr batch);
        [LibraryImport(Lib)] internal static partial long vpz_batch_total_bytes(IntPtr batch);
        [LibraryImport(Lib)] internal static partial int vpz_batch_upload(IntPtr batch);
        [LibraryImport(Lib)] internal static partial int vpz_batch_decode(IntPtr batch, int clip);
        [LibraryImport(Lib)] internal static partial int vpz_batch_sync(IntPtr batch);
        [LibraryImport(Lib)] internal static partial int vpz_batch_has_clipped(IntPtr batch);
        [LibraryImport(Lib)] internal static partial int vpz_batch_read_run(IntPtr batch, int run, float* dst);
        [LibraryImport(Lib)] internal static partial int vpz_batch_read_all(IntPtr batch, float* dst);
        [LibraryImport(Lib)] internal static partial long vpz_batch_run_offset(IntPtr batch, int run);
        [LibraryImport(Lib)] internal static partial IntPtr vpz_batch_device_pcm(IntPtr batch);
        [LibraryImport(Lib)] internal static partial float vpz_batch_last_ms(IntPtr batch, int which, out int launches);
        [LibraryImport(Lib)] internal static partial ulong vpz_transfer_bytes(int which);
        [LibraryImport(Lib)] internal static partial IntPtr vpz_host_alloc(nuint bytes);
        [LibraryImport(Lib)] internal static partial void vpz_host_free(IntPtr p);

        // ---- reader: IVorbisReader / IStreamDecoder over container bytes
        [LibraryImport(Lib)] internal static partial int vpz_reader_open_memory(IntPtr ctx, byte* data, nuint len, int copy, out IntPtr reader);
        [LibraryImport(Lib)] internal static partial void vpz_reader_close(IntPtr reader);
        [LibraryImport(Lib)] internal static partial int vpz_reader_stream_count(IntPtr reader);
        [LibraryImport(Lib)] internal static partial int vpz_reader_stream_index(IntPtr reader);
        [LibraryImport(Lib)] internal static partial int vpz_reader_switch_stream(IntPtr reader, int index);
        [LibraryImport(Lib)] internal static partial int vpz_reader_find_next_stream(IntPtr reader);
        [LibraryImport(Lib)] internal static partial int vpz_reader_can_seek(IntPtr reader);
        [LibraryImport(Lib)] internal static partial int vpz_reader_channels(IntPtr reader);
        [LibraryImport(Lib)] internal static partial int vpz_reader_sample_rate(IntPtr reader);
        [LibraryImport(Lib)] internal static partial int vpz_reader_bitrate(IntPtr reader, int which);
        [LibraryImport(Lib)] internal static partial int vpz_reader_stream_serial(IntPtr reader);
        [LibraryImport(Lib)] internal static partial long vpz_reader_total_samples(IntPtr reader);
        [LibraryImport(Lib)] internal static partial long vpz_reader_sample_position(IntPtr reader);
        [LibraryImport(Lib)] internal static partial int vpz_reader_is_end_of_stream(IntPtr reader);
        [LibraryImport(Lib)] internal static partial int vpz_reader_has_clipped(IntPtr reader);
        [LibraryImport(Lib)] internal static partial int vpz_reader_get_clip(IntPtr reader);
        [LibraryImport(Lib)] internal static partial void vpz_reader_set_clip(IntPtr reader, int clip);
        [LibraryImport(Lib)] internal static partial long vpz_reader_container_overhead_bits(IntPtr reader);
        [LibraryImport(Lib)] internal static partial long vpz_reader_container_waste_bits(IntPtr reader);
        [LibraryImport(Lib)] internal static partial IntPtr vpz_reader_vendor(IntPtr reader, out int len);
        [LibraryImport(Lib)] internal static partial int vpz_reader_comment_count(IntPtr reader);
        [LibraryImport(Lib)] internal static partial IntPtr vpz_reader_comment(IntPtr reader, int i, out int len);
        [LibraryImport(Lib)] internal static partial int vpz_reader_read(IntPtr reader, float* buf, int nfloats);
        [LibraryImport(Lib)] internal static partial int vpz_reader_read_planar(IntPtr reader, float* buf, int nfloats, int samplesToRead, int channelStride);
        [LibraryImport(Lib)] internal static partial int vpz_reader_seek(IntPtr reader, long samplePosition, int origin);
        [LibraryImport(Lib)] internal static partial int vpz_reader_set_lookahead(IntPtr reader, int packets);
        [LibraryImport(Lib)] internal static partial int vpz_reader_audio_packet_count(IntPtr reader);
        [LibraryImport(Lib)] internal static partial int vpz_reader_audio_packet(IntPtr reader, int i, out byte* data, out uint len, out long granule, out int flags);
        [LibraryImport(Lib)] internal static partial byte* vpz_reader_header_packet(IntPtr reader, int which, out uint len);
        [LibraryImport(Lib)] internal static partial IntPtr vpz_reader_setup(IntPtr reader);

        // ---- bulk
        [LibraryImport(Lib)] internal static partial long vpz_decode_files(IntPtr ctx, uint n, byte** datas, nuint* lens, int clip, float* dst, nuint dstFloats, long* sampleCounts);
        [LibraryImport(Lib)] internal static partial long vpz_decode_files_s16(IntPtr ctx, uint n, byte** datas, nuint* lens, int clip, short* dst, nuint dstSamples, long* sampleCounts);
        [LibraryImport(Lib)] internal static partial long vpz_scan_pages(IntPtr ctx, uint n, byte** datas, nuint* lens, VpzPageInfo* pages, nuint pagesCap, uint* first, uint* count, ulong* wasteBits, uint* crcFailures);
        [LibraryImport(Lib)] internal static partial long vpz_decode_excerpts(IntPtr ctx, uint nFiles, byte** datas, nuint* lens, uint n, uint* fileOf, long* start, int* count, int clip, float* dst, nuint dstFloats, long* dstOffsets, int* got);
        // format bits of the *_device calls (0 = fp32 interleaved); dstDev is device memory of the context's GPU, stream a cudaStream_t
        internal const int OutS16 = 1, OutPlanar = 2;
        [LibraryImport(Lib)] internal static partial long vpz_decode_files_device(IntPtr ctx, uint n, byte** datas, nuint* lens, int clip, int format, IntPtr dstDev, nuint dstElems, long* sampleCounts, IntPtr stream);
        [LibraryImport(Lib)] internal static partial long vpz_decode_excerpts_device(IntPtr ctx, uint nFiles, byte** datas, nuint* lens, uint n, uint* fileOf, long* start, int* count, int clip, int format, IntPtr dstDev, nuint dstElems, long* dstOffsets, int* got, IntPtr stream);
        // the same with every item converted to conv->SampleRate / conv->Channels (0: keep) on the GPU (K6)
        [LibraryImport(Lib)] internal static partial long vpz_decode_files_device_conv(IntPtr ctx, uint n, byte** datas, nuint* lens, int clip, VpzOutConv* conv, IntPtr dstDev, nuint dstElems, long* sampleCounts, long* dstOffsets, IntPtr stream);
        [LibraryImport(Lib)] internal static partial long vpz_decode_excerpts_device_conv(IntPtr ctx, uint nFiles, byte** datas, nuint* lens, uint n, uint* fileOf, long* start, int* count, int clip, VpzOutConv* conv, IntPtr dstDev, nuint dstElems, long* dstOffsets, int* got, IntPtr stream);
        // corpus: images opened once (scan, headers, setups, seek index, lengths; images resident on the GPU), excerpts many times
        [LibraryImport(Lib)] internal static partial int vpz_corpus_open(IntPtr ctx, uint n, byte** datas, nuint* lens, int copy, out IntPtr corpus);
        [LibraryImport(Lib)] internal static partial void vpz_corpus_close(IntPtr corpus);
        [LibraryImport(Lib)] internal static partial long vpz_corpus_info(IntPtr corpus, int* channels, int* sampleRate, long* samples);
        [LibraryImport(Lib)] internal static partial ulong vpz_corpus_device_bytes(IntPtr corpus);
        [LibraryImport(Lib)] internal static partial long vpz_corpus_excerpts_device(IntPtr corpus, uint n, uint* fileOf, long* start, int* count, int clip, VpzOutConv* conv, IntPtr dstDev, nuint dstElems, long* dstOffsets, int* got, IntPtr stream);
        [LibraryImport(Lib)] internal static partial long vpz_debug_page_end_granules(IntPtr ctx, byte* data, nuint len, int onDevice, long* dst, nuint cap);
    }
}
