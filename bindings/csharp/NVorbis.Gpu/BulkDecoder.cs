// Bulk calls: many container images per call, pipelined on the GPU (vpz_decode_files / _s16 / vpz_decode_excerpts /
// their _device forms / vpz_scan_pages).  These have no counterpart in the reference's API; they are what a server decoding thousands of
// streams calls instead of one VorbisReader per stream.
using System;
using System.Buffers;
using System.Runtime.InteropServices;

namespace NVorbis.Gpu
{
    public static unsafe class BulkDecoder
    {
        sealed class PinnedImages : IDisposable
        {
            public readonly MemoryHandle[] Handles;
            public readonly IntPtr[] Ptrs;
            public readonly nuint[] Lens;
            public PinnedImages(ReadOnlyMemory<byte>[] files)
            {
                Handles = new MemoryHandle[files.Length];
                Ptrs = new IntPtr[Math.Max(files.Length, 1)];
                Lens = new nuint[Math.Max(files.Length, 1)];
                for (int i = 0; i < files.Length; i++)
                {
                    Handles[i] = files[i].Pin();
                    Ptrs[i] = (IntPtr)Handles[i].Pointer;
                    Lens[i] = (nuint)files[i].Length;
                }
            }
            public void Dispose() { foreach (MemoryHandle h in Handles) h.Dispose(); }
        }

        /// <summary>Every file decoded from its first to its last sample, interleaved, file after file.
        /// Returns the pinned PCM and the samples per channel of each file.</summary>
        public static (PinnedBuffer<float> pcm, long[] sampleCounts) DecodeFiles(GpuContext gpu, ReadOnlyMemory<byte>[] files, bool clip = true)
        {
            using PinnedImages im = new(files);
            long[] counts = new long[files.Length];
            fixed (IntPtr* p = im.Ptrs)
            fixed (nuint* l = im.Lens)
            fixed (long* c = counts)
            {
                long total = Vpz.vpz_decode_files(gpu.Handle, (uint)files.Length, (byte**)p, l, clip ? 1 : 0, null, 0, c);   // size query
                Vpz.Check(total, gpu.Handle);
                PinnedBuffer<float> dst = gpu.AllocPinned<float>(Math.Max(total, 1));
                long got = Vpz.vpz_decode_files(gpu.Handle, (uint)files.Length, (byte**)p, l, clip ? 1 : 0, (float*)dst.Pointer, (nuint)total, c);
                if (got < 0) dst.Dispose();
                Vpz.Check(got, gpu.Handle);
                return (dst, counts);
            }
        }

        /// <summary>The same with 16-bit PCM converted on the GPU by the rule of the reference's tests
        /// (AssetTest.cs:131-132: (int)(x * 32768f), clamped): half the device-to-host bytes.</summary>
        public static (PinnedBuffer<short> pcm, long[] sampleCounts) DecodeFilesInt16(GpuContext gpu, ReadOnlyMemory<byte>[] files, bool clip = true)
        {
            using PinnedImages im = new(files);
            long[] counts = new long[files.Length];
            fixed (IntPtr* p = im.Ptrs)
            fixed (nuint* l = im.Lens)
            fixed (long* c = counts)
            {
                long total = Vpz.vpz_decode_files_s16(gpu.Handle, (uint)files.Length, (byte**)p, l, clip ? 1 : 0, null, 0, c);
                Vpz.Check(total, gpu.Handle);
                PinnedBuffer<short> dst = gpu.AllocPinned<short>(Math.Max(total, 1));
                long got = Vpz.vpz_decode_files_s16(gpu.Handle, (uint)files.Length, (byte**)p, l, clip ? 1 : 0, (short*)dst.Pointer, (nuint)total, c);
                if (got < 0) dst.Dispose();
                Vpz.Check(got, gpu.Handle);
                return (dst, counts);
            }
        }

        /// <summary>Random access in bulk: excerpt i is what `new VorbisReader(files[file]).SeekTo(start)` followed by
        /// ReadSamples until `count` samples per channel delivers (StreamDecoder.cs:817-880, 418-498).  got[i] is the
        /// number of samples per channel delivered, or the negative vpz_status SeekTo raised for that excerpt
        /// (Vpz.SeekRange -> SeekOutOfRangeException, Vpz.PreRoll -> PreRollPacketException); undelivered floats are 0.</summary>
        public static (PinnedBuffer<float> pcm, long[] offsets, int[] got) ReadExcerpts(
            GpuContext gpu, ReadOnlyMemory<byte>[] files, (int file, long start, int count)[] excerpts, bool clip = true)
        {
            using PinnedImages im = new(files);
            int n = excerpts.Length;
            uint[] fileOf = new uint[Math.Max(n, 1)];
            long[] start = new long[Math.Max(n, 1)];
            int[] count = new int[Math.Max(n, 1)];
            for (int i = 0; i < n; i++) (fileOf[i], start[i], count[i]) = ((uint)excerpts[i].file, excerpts[i].start, excerpts[i].count);
            long[] offsets = new long[Math.Max(n, 1)];
            int[] got = new int[Math.Max(n, 1)];
            fixed (IntPtr* p = im.Ptrs)
            fixed (nuint* l = im.Lens)
            fixed (uint* f = fileOf)
            fixed (long* s = start, o = offsets)
            fixed (int* c = count, g = got)
            {
                long total = Vpz.vpz_decode_excerpts(gpu.Handle, (uint)files.Length, (byte**)p, l, (uint)n, f, s, c, clip ? 1 : 0, null, 0, o, g);
                Vpz.Check(total, gpu.Handle);
                PinnedBuffer<float> dst = gpu.AllocPinned<float>(Math.Max(total, 1));
                long rc = Vpz.vpz_decode_excerpts(gpu.Handle, (uint)files.Length, (byte**)p, l, (uint)n, f, s, c, clip ? 1 : 0, (float*)dst.Pointer, (nuint)total, o, g);
                if (rc < 0) dst.Dispose();
                Vpz.Check(rc, gpu.Handle);
                return (dst, offsets, got);
            }
        }

        /// <summary>Elements (fp32, or int16 with int16: true) a DecodeFilesToDevice call of these files writes, and the
        /// samples per channel of each file: the size query, nothing is decoded.</summary>
        public static long DeviceElements(GpuContext gpu, ReadOnlyMemory<byte>[] files, out long[] sampleCounts, bool clip = true)
        {
            using PinnedImages im = new(files);
            sampleCounts = new long[files.Length];
            fixed (IntPtr* p = im.Ptrs)
            fixed (nuint* l = im.Lens)
            fixed (long* c = sampleCounts)
            {
                long total = Vpz.vpz_decode_files_device(gpu.Handle, (uint)files.Length, (byte**)p, l, clip ? 1 : 0, 0, IntPtr.Zero, 0, c, IntPtr.Zero);
                Vpz.Check(total, gpu.Handle);
                return total;
            }
        }

        /// <summary>DecodeFiles with the PCM left in GPU memory: dstDevice is device memory of the context's GPU with room
        /// for dstElements elements (DeviceElements); file k starts at element sum over j &lt; k of samples_j * channels_j,
        /// channel-major [channels][samples] with planar: true, interleaved otherwise; int16: the rule of DecodeFilesInt16,
        /// for every stream.  The call waits for the work queued on `stream` (a cudaStream_t, IntPtr.Zero: the legacy
        /// default stream) and returns when dstDevice is complete.  Returns the samples per channel of each file.</summary>
        public static long[] DecodeFilesToDevice(GpuContext gpu, ReadOnlyMemory<byte>[] files, IntPtr dstDevice, long dstElements,
                                                 bool planar = true, bool int16 = false, bool clip = true, IntPtr stream = default)
        {
            using PinnedImages im = new(files);
            long[] counts = new long[files.Length];
            int format = (planar ? Vpz.OutPlanar : 0) | (int16 ? Vpz.OutS16 : 0);
            fixed (IntPtr* p = im.Ptrs)
            fixed (nuint* l = im.Lens)
            fixed (long* c = counts)
            {
                Vpz.Check(Vpz.vpz_decode_files_device(gpu.Handle, (uint)files.Length, (byte**)p, l, clip ? 1 : 0, format, dstDevice,
                                                      (nuint)dstElements, c, stream), gpu.Handle);
                return counts;
            }
        }

        /// <summary>ReadExcerpts with the PCM left in GPU memory (layout, format and stream as DecodeFilesToDevice; excerpt i
        /// holds count samples per channel at element offsets[i], undelivered samples are 0).  dstDevice == IntPtr.Zero:
        /// only the layout is computed.  Returns the total elements of the layout.</summary>
        public static long ReadExcerptsToDevice(GpuContext gpu, ReadOnlyMemory<byte>[] files, (int file, long start, int count)[] excerpts,
                                                IntPtr dstDevice, long dstElements, out long[] offsets, out int[] got,
                                                bool planar = true, bool int16 = false, bool clip = true, IntPtr stream = default)
        {
            using PinnedImages im = new(files);
            int n = excerpts.Length;
            uint[] fileOf = new uint[Math.Max(n, 1)];
            long[] start = new long[Math.Max(n, 1)];
            int[] count = new int[Math.Max(n, 1)];
            for (int i = 0; i < n; i++) (fileOf[i], start[i], count[i]) = ((uint)excerpts[i].file, excerpts[i].start, excerpts[i].count);
            offsets = new long[Math.Max(n, 1)];
            got = new int[Math.Max(n, 1)];
            int format = (planar ? Vpz.OutPlanar : 0) | (int16 ? Vpz.OutS16 : 0);
            fixed (IntPtr* p = im.Ptrs)
            fixed (nuint* l = im.Lens)
            fixed (uint* f = fileOf)
            fixed (long* s = start, o = offsets)
            fixed (int* c = count, g = got)
            {
                long rc = Vpz.vpz_decode_excerpts_device(gpu.Handle, (uint)files.Length, (byte**)p, l, (uint)n, f, s, c, clip ? 1 : 0, format,
                                                         dstDevice, (nuint)dstElements, o, g, stream);
                Vpz.Check(rc, gpu.Handle);
                return rc;
            }
        }

        /// <summary>DecodeFilesToDevice with every file converted on the GPU to sampleRate (0: each keeps its own; else
        /// 1,000..384,000 Hz, torchaudio.functional.resample's default filter) and channels (0: keep, 1: mean, 2: mono
        /// duplicated, stereo kept).  dstDevice == IntPtr.Zero: only the layout is computed.  sampleCounts receives the
        /// output samples per channel of each file, offsets the element offset of each file.  Returns the total
        /// elements of the layout.</summary>
        public static long DecodeFilesToDevice(GpuContext gpu, ReadOnlyMemory<byte>[] files, int sampleRate, int channels,
                                               IntPtr dstDevice, long dstElements, out long[] sampleCounts, out long[] offsets,
                                               bool planar = true, bool int16 = false, bool clip = true, IntPtr stream = default)
        {
            using PinnedImages im = new(files);
            sampleCounts = new long[Math.Max(files.Length, 1)];
            offsets = new long[Math.Max(files.Length, 1)];
            VpzOutConv conv = new() { Format = (planar ? Vpz.OutPlanar : 0) | (int16 ? Vpz.OutS16 : 0), SampleRate = sampleRate, Channels = channels };
            fixed (IntPtr* p = im.Ptrs)
            fixed (nuint* l = im.Lens)
            fixed (long* c = sampleCounts, o = offsets)
            {
                long rc = Vpz.vpz_decode_files_device_conv(gpu.Handle, (uint)files.Length, (byte**)p, l, clip ? 1 : 0, &conv, dstDevice,
                                                           (nuint)dstElements, c, o, stream);
                Vpz.Check(rc, gpu.Handle);
                return rc;
            }
        }

        /// <summary>ReadExcerptsToDevice with every excerpt converted as DecodeFilesToDevice(.., sampleRate, channels, ..)
        /// converts files; start and count are samples at the output rate, got counts output samples.  Excerpts of one
        /// count then make a dense [n][channels][count] batch (planar) whatever the rates and layouts of the files.</summary>
        public static long ReadExcerptsToDevice(GpuContext gpu, ReadOnlyMemory<byte>[] files, (int file, long start, int count)[] excerpts,
                                                int sampleRate, int channels, IntPtr dstDevice, long dstElements, out long[] offsets,
                                                out int[] got, bool planar = true, bool int16 = false, bool clip = true,
                                                IntPtr stream = default)
        {
            using PinnedImages im = new(files);
            int n = excerpts.Length;
            uint[] fileOf = new uint[Math.Max(n, 1)];
            long[] start = new long[Math.Max(n, 1)];
            int[] count = new int[Math.Max(n, 1)];
            for (int i = 0; i < n; i++) (fileOf[i], start[i], count[i]) = ((uint)excerpts[i].file, excerpts[i].start, excerpts[i].count);
            offsets = new long[Math.Max(n, 1)];
            got = new int[Math.Max(n, 1)];
            VpzOutConv conv = new() { Format = (planar ? Vpz.OutPlanar : 0) | (int16 ? Vpz.OutS16 : 0), SampleRate = sampleRate, Channels = channels };
            fixed (IntPtr* p = im.Ptrs)
            fixed (nuint* l = im.Lens)
            fixed (uint* f = fileOf)
            fixed (long* s = start, o = offsets)
            fixed (int* c = count, g = got)
            {
                long rc = Vpz.vpz_decode_excerpts_device_conv(gpu.Handle, (uint)files.Length, (byte**)p, l, (uint)n, f, s, c, clip ? 1 : 0,
                                                              &conv, dstDevice, (nuint)dstElements, o, g, stream);
                Vpz.Check(rc, gpu.Handle);
                return rc;
            }
        }

        /// <summary>The physical Ogg layer of many images on the GPU (PageReaderBase.ReadNextPage / VerifyPage,
        /// Ogg/PageReaderBase.cs:41-84,286-361; Crc.cs:20-63): the valid pages of every image.</summary>
        public static VpzPageInfo[][] ScanPages(GpuContext gpu, ReadOnlyMemory<byte>[] files, out ulong[] wasteBits, out uint[] crcFailures)
        {
            using PinnedImages im = new(files);
            int n = files.Length;
            long cap = 1;
            foreach (ReadOnlyMemory<byte> m in files) cap += m.Length / 64 + 16;
            VpzPageInfo[] pages = new VpzPageInfo[cap];
            uint[] first = new uint[Math.Max(n, 1)], count = new uint[Math.Max(n, 1)];
            wasteBits = new ulong[Math.Max(n, 1)];
            crcFailures = new uint[Math.Max(n, 1)];
            fixed (IntPtr* p = im.Ptrs)
            fixed (nuint* l = im.Lens)
            fixed (VpzPageInfo* pg = pages)
            fixed (uint* fi = first, ct = count, cf = crcFailures)
            fixed (ulong* wb = wasteBits)
                Vpz.Check(Vpz.vpz_scan_pages(gpu.Handle, (uint)n, (byte**)p, l, pg, (nuint)cap, fi, ct, wb, cf), gpu.Handle);
            VpzPageInfo[][] outp = new VpzPageInfo[n][];
            for (int i = 0; i < n; i++) outp[i] = pages.AsSpan((int)first[i], (int)count[i]).ToArray();
            return outp;
        }
    }
}
