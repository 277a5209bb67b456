// A set of container images opened once on one GPU (vpz_corpus_*): the page scan, headers, setup tables, seek index
// and lengths are built at open and the images stay in GPU memory, so every excerpt batch afterwards costs only its
// own planning and decoding.  The results are those of BulkDecoder.ReadExcerptsToDevice on the same images.
using System;
using System.Buffers;

namespace NVorbis.Gpu
{
    public sealed unsafe class GpuCorpus : IDisposable
    {
        readonly GpuContext _gpu;
        IntPtr _h;

        /// <summary>Per file: channels, sample rate and TotalSamples of a fresh reader on its first logical stream.</summary>
        public int[] Channels { get; }
        public int[] SampleRates { get; }
        public long[] TotalSamples { get; }
        public int Count => TotalSamples.Length;
        /// <summary>Bytes of GPU memory the corpus holds (its images).</summary>
        public ulong DeviceBytes => _h == IntPtr.Zero ? 0 : Vpz.vpz_corpus_device_bytes(_h);

        /// <summary>Opens the images as one corpus of gpu.  The library keeps its own copy of the bytes (copy = 1), so
        /// the managed arrays are pinned only for the duration of the call.  A file ReadExcerptsToDevice would reject
        /// throws the same exception here.  Dispose the corpus before its context.</summary>
        public GpuCorpus(GpuContext gpu, ReadOnlyMemory<byte>[] files)
        {
            _gpu = gpu;
            int n = files.Length;
            MemoryHandle[] pins = new MemoryHandle[n];
            IntPtr[] ptrs = new IntPtr[Math.Max(n, 1)];
            nuint[] lens = new nuint[Math.Max(n, 1)];
            try
            {
                for (int i = 0; i < n; i++)
                {
                    pins[i] = files[i].Pin();
                    ptrs[i] = (IntPtr)pins[i].Pointer;
                    lens[i] = (nuint)files[i].Length;
                }
                fixed (IntPtr* p = ptrs)
                fixed (nuint* l = lens)
                    Vpz.Check(Vpz.vpz_corpus_open(gpu.Handle, (uint)n, (byte**)p, l, 1, out _h), gpu.Handle);
            }
            finally
            {
                foreach (MemoryHandle h in pins) h.Dispose();
            }
            Channels = new int[n];
            SampleRates = new int[n];
            TotalSamples = new long[n];
            fixed (int* c = Channels, r = SampleRates)
            fixed (long* s = TotalSamples)
                Vpz.Check(Vpz.vpz_corpus_info(_h, c, r, s), gpu.Handle);
        }

        /// <summary>BulkDecoder.ReadExcerptsToDevice on the corpus's files (file = index in the corpus): the same layout,
        /// offsets, got, errors and elements, bitwise.  dstDevice == IntPtr.Zero: only the layout is computed.</summary>
        public long ReadExcerptsToDevice((int file, long start, int count)[] excerpts, IntPtr dstDevice, long dstElements,
                                         out long[] offsets, out int[] got, bool planar = true, bool int16 = false,
                                         bool clip = true, IntPtr stream = default)
            => ReadExcerptsToDevice(excerpts, 0, 0, dstDevice, dstElements, out offsets, out got, planar, int16, clip, stream);

        /// <summary>The same with every excerpt converted to sampleRate (0: keep) and channels (0: keep, 1: mean, 2: mono
        /// duplicated) on the GPU, as BulkDecoder.ReadExcerptsToDevice(.., sampleRate, channels, ..) converts them.</summary>
        public long ReadExcerptsToDevice((int file, long start, int count)[] excerpts, int sampleRate, int channels,
                                         IntPtr dstDevice, long dstElements, out long[] offsets, out int[] got,
                                         bool planar = true, bool int16 = false, bool clip = true, IntPtr stream = default)
        {
            if (_h == IntPtr.Zero) throw new ObjectDisposedException(nameof(GpuCorpus));
            int n = excerpts.Length;
            uint[] fileOf = new uint[Math.Max(n, 1)];
            long[] start = new long[Math.Max(n, 1)];
            int[] count = new int[Math.Max(n, 1)];
            for (int i = 0; i < n; i++) (fileOf[i], start[i], count[i]) = ((uint)excerpts[i].file, excerpts[i].start, excerpts[i].count);
            offsets = new long[Math.Max(n, 1)];
            got = new int[Math.Max(n, 1)];
            VpzOutConv conv = new() { Format = (planar ? Vpz.OutPlanar : 0) | (int16 ? Vpz.OutS16 : 0), SampleRate = sampleRate, Channels = channels };
            fixed (uint* f = fileOf)
            fixed (long* s = start, o = offsets)
            fixed (int* c = count, g = got)
            {
                long rc = Vpz.vpz_corpus_excerpts_device(_h, (uint)n, f, s, c, clip ? 1 : 0, &conv, dstDevice, (nuint)dstElements, o, g, stream);
                Vpz.Check(rc, _gpu.Handle);
                return rc;
            }
        }

        public void Dispose()
        {
            if (_h != IntPtr.Zero) Vpz.vpz_corpus_close(_h);
            _h = IntPtr.Zero;
        }
    }
}
