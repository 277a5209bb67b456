/*
 * vpz.h -- C ABI of the B200-native Vorbis decode path (libvpz.so).
 *
 * This is the boundary a VorbisPizza maintainer binds with P/Invoke to replace the managed hot
 * path below StreamDecoder.Read (reference: NVorbis/StreamDecoder.cs:418) and above
 * IPacketProvider.GetNextPacket (NVorbis/Contracts/IPacketProvider.cs:9-48).  Plain pointers and
 * sizes only; no exceptions, callbacks or caller-freed allocations cross it.  Every entry point
 * returns 0 (VPZ_OK) / a non-negative count, or a negative VPZ_E_* code that the managed shim maps
 * to the reference's exception types (see INTEGRATION.md).  There is NO CPU fallback: without a
 * usable sm_100 device every compute entry point fails with VPZ_E_NO_DEVICE / VPZ_E_CUDA.
 *
 * Three layers, lowest first:
 *   1. setup  -- vpz_setup_*  : replaces StreamDecoder.LoadStreamHeader/LoadBooks table building
 *                               (StreamDecoder.cs:213-355); tables are uploaded once per distinct
 *                               (id, setup) header pair.
 *   2. batch  -- vpz_batch_*  : replaces Mode.Decode -> Mapping.DecodePacket -> Mdct.Reverse ->
 *                               OverlapBuffers -> StoreInterleaved (Mode.cs:68, Mapping.cs:98,
 *                               Mdct.cs:15, StreamDecoder.cs:515-592,764-791) for MANY packets of
 *                               MANY streams per call.  This is the IPacketProvider-side seam.
 *   3. reader -- vpz_reader_* : the IStreamDecoder / IVorbisReader-side seam
 *                               (Contracts/IStreamDecoder.cs:9-152, Contracts/IVorbisReader.cs:10-150)
 *                               including the host-side Ogg layer, for callers that hand over the
 *                               container bytes instead of packets.
 * All calls that share one vpz_ctx must come from one host thread at a time.
 */
#ifndef VPZ_H
#define VPZ_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vpz_ctx vpz_ctx;
typedef struct vpz_setup vpz_setup;
typedef struct vpz_batch vpz_batch;
typedef struct vpz_reader vpz_reader;

enum {
  VPZ_OK = 0,
  VPZ_E_INVALID_DATA = -1,  /* System.IO.InvalidDataException (StreamDecoder.cs:77,84,313,330,338,351,734) */
  VPZ_E_ARGUMENT = -2,      /* ArgumentException / ArgumentOutOfRangeException (StreamDecoder.cs:423-430,825,842) */
  VPZ_E_SEEK_RANGE = -3,    /* SeekOutOfRangeException (StreamDecoder.cs:861) */
  VPZ_E_PREROLL = -4,       /* PreRollPacketException (StreamDecoder.cs:874) */
  VPZ_E_UNSUPPORTED = -5,   /* valid Vorbis the GPU path does not cover (> 8 channels, block size < 256, > 64 floor posts) */
  VPZ_E_CUDA = -6,          /* CUDA runtime error; vpz_last_error() has the text */
  VPZ_E_NOMEM = -7,
  VPZ_E_DISPOSED = -8,      /* ObjectDisposedException (StreamDecoder.cs:401) */
  VPZ_E_INVALID_OP = -9,    /* InvalidOperationException (StreamDecoder.cs:822) */
  VPZ_E_NO_DEVICE = -10,    /* no sm_100 GPU visible: the product has no CPU path */
  VPZ_E_REF_FAULT = -11     /* the reference faults here (SURVEY quirk Q4); we stop the stream instead */
};

const char* vpz_strerror(int code);
/* Text of the last failure on this context (valid until the next call on it). */
const char* vpz_last_error(const vpz_ctx* ctx);
/* Library version / build string, e.g. "vpz 0.1 sm_100a". */
const char* vpz_version(void);

/* ---- context: one per GPU ------------------------------------------------------------- */
/* device < 0: the current CUDA device.  Creates the stream, pinned staging and table caches. */
int vpz_ctx_create(int device, vpz_ctx** out);
void vpz_ctx_destroy(vpz_ctx* ctx);
int vpz_device_count(void);
/* Tunables (call before the first batch): key one of "l1_bits" (Huffman first-level table width,
 * default 9), "ola_chunk" (packets per IMDCT work item, default: 16..63 chosen per batch), "k1_warps" (warps per entropy
 * CTA, default 4), "bulk_group" (streams per pipeline group of vpz_decode_files, default 256), "bulk_group_mib" (a group also closes
 * at this many MiB of container images, default 128, at most 384),
 * "host_threads" (size of the host worker pool of the bulk calls, default 0 = all cores up to 32), "bulk_threads"
 * (how many of them vpz_decode_files uses, default 4: the call is bound by the PCM copy, which more staging
 * threads slow down; 0 = all), "bulk_threads_device" (the same for vpz_decode_files_device, default 8: without a
 * PCIe copy the call is bound by the host's scan and planning, and 8 threads measured fastest), "gpu_scan" (bulk
 * path: Ogg page scan + CRC on the GPU, default 1), "force_general" (tests: route every packet through the
 * general kernels). */
int vpz_ctx_set(vpz_ctx* ctx, const char* key, int value);

/* Device-side stopwatch on the context's stream: vpz_ctx_mark records CUDA event `slot` (0..7) on
 * the stream all of this context's kernels and copies are issued on; vpz_ctx_elapsed_ms waits for
 * slot b and returns the milliseconds between two marks (< 0 on error). */
int vpz_ctx_mark(vpz_ctx* ctx, int slot);
float vpz_ctx_elapsed_ms(vpz_ctx* ctx, int slot_a, int slot_b);
/* Number of kernels this library has launched on the context so far. */
int64_t vpz_ctx_kernel_launches(const vpz_ctx* ctx);

/* ---- setup: StreamDecoder.LoadStreamHeader + LoadBooks -------------------------------- */
typedef struct {
  int32_t channels, sample_rate;
  int32_t bitrate_upper, bitrate_nominal, bitrate_lower;
  int32_t block_size0, block_size1;
  int32_t n_books, n_floors, n_residues, n_mappings, n_modes;
  int32_t max_codeword_bits;
  uint64_t table_bytes;      /* size of the device image */
} vpz_setup_info;

/* Parses the identification and setup header packets, builds the GPU tables and uploads them.
 * Identical header pairs share one vpz_setup (content hash); each create needs one release. */
int vpz_setup_create(vpz_ctx* ctx, const uint8_t* id_pkt, size_t id_len, const uint8_t* setup_pkt,
                     size_t setup_len, vpz_setup** out);
void vpz_setup_release(vpz_setup* s);
int vpz_setup_get_info(const vpz_setup* s, vpz_setup_info* info);

/* Mode.GetPacketInfo (Mode.cs:30-66) for one audio packet, from its first bytes: the callback the
 * reference's seek code needs (IPacketGranuleCountProvider, StreamDecoder.cs:882-913).
 * info = {Length, LeftUseSize1, LeftStart, LeftEnd, RightStart, RightEnd}.  Returns 1 when the
 * packet is a decodable audio packet, 0 when the reference would skip it, VPZ_E_INVALID_DATA for
 * an unused mode index (StreamDecoder.cs:732-735). */
int vpz_packet_info(const vpz_setup* s, const uint8_t* pkt, size_t len, int32_t info[6]);

/* ---- batch: many packets of many streams in one pass ---------------------------------- */
int vpz_batch_create(vpz_ctx* ctx, vpz_batch** out);
void vpz_batch_destroy(vpz_batch* b);
/* Forget all runs but keep the buffers (steady-state reuse). */
int vpz_batch_reset(vpz_batch* b);

/* Adds one RUN: a fresh decoder state (as after StreamDecoder.ResetDecoder, StreamDecoder.cs:357)
 * fed `n_pkts` consecutive audio packets.  As in the reference the first decodable packet of a run
 * only seeds the overlap and yields no samples, so a caller continuing a stream passes its previous
 * packet again as the first packet of the next run (this is also the seek pre-roll).
 *   bytes/offsets : packet i is bytes[offsets[i] .. offsets[i+1])
 *   trim          : NULL, or per packet the number of samples to pull RightStart back by
 *                   (end-of-stream granule trim, StreamDecoder.cs:658-666); a negative value
 *                   instead extends the packet's output by that many samples of its raw right
 *                   half (the drain of StreamDecoder.cs:451-455)
 * Returns the run index (>= 0).  Packets the reference would skip (header bit set, empty decode)
 * are skipped; an unused mode index fails the call with VPZ_E_INVALID_DATA. */
int vpz_batch_add_run(vpz_batch* b, vpz_setup* s, const uint8_t* bytes, const uint32_t* offsets,
                      uint32_t n_pkts, const int32_t* trim);
/* Samples per channel run `run` will produce (known before decoding: geometry is in the packet
 * headers), and its channel count. */
int64_t vpz_batch_run_samples(const vpz_batch* b, int run);
int vpz_batch_run_channels(const vpz_batch* b, int run);
/* 0, or VPZ_E_REF_FAULT when the run was cut at submitted packet *stop_packet because the reference
 * itself faults there (overlap longer than the window slope, SURVEY quirk Q4). */
int vpz_batch_run_status(const vpz_batch* b, int run, int32_t* stop_packet);
/* Per-packet sample counts of a run (PacketInfo.SampleCount after trim; 0 for skipped packets and
 * for the seeding packet).  counts has n_pkts entries. */
int vpz_batch_run_packet_samples(const vpz_batch* b, int run, int32_t* counts);
int64_t vpz_batch_total_floats(const vpz_batch* b);
int64_t vpz_batch_total_packets(const vpz_batch* b);
int64_t vpz_batch_total_bytes(const vpz_batch* b);

/* Uploads the queued packets (host -> device) and builds the device work lists. */
int vpz_batch_upload(vpz_batch* b);
/* Launches symbol decode (K1a), spectrum build (K1b: VQ accumulate, coupling, floor) and IMDCT +
 * window + overlap-add + store (K3) on the context's stream.  clip != 0 clamps to +-0.99999994f like Utils.ClipValue (Utils.cs:44-58).
 * Asynchronous; vpz_batch_sync waits.  May be called repeatedly on the same uploaded batch. */
int vpz_batch_decode(vpz_batch* b, int clip);
int vpz_batch_sync(vpz_batch* b);
/* 1 when any sample was clamped in the last decode (HasClipped, StreamDecoder.cs:569-570). */
int vpz_batch_has_clipped(vpz_batch* b);

/* Interleaved float PCM of one run, device -> host.  dst has run_samples * channels floats. */
int vpz_batch_read_run(vpz_batch* b, int run, float* dst);
/* All runs back to back (run order), device -> host; dst has vpz_batch_total_floats floats.
 * dst may be pinned memory from vpz_host_alloc for full PCIe rate. */
int vpz_batch_read_all(vpz_batch* b, float* dst);
/* Float offset of a run inside the batch PCM buffer / the device pointer of that buffer, for
 * consumers that keep PCM on the GPU. */
int64_t vpz_batch_run_offset(const vpz_batch* b, int run);
const float* vpz_batch_device_pcm(const vpz_batch* b);

/* Device time of the last vpz_batch_decode in milliseconds: which = 0 total, 1 entropy stage (K1a +
 * K1b), 11 symbol decode (K1a), 12 spectrum build (K1b), 3 IMDCT/OLA (K3); number of kernel launches
 * in `launches` (may be NULL). */
float vpz_batch_last_ms(vpz_batch* b, int which, int* launches);

/* Bytes this process has copied so far: which = 0 host->device, 1 device->host. */
uint64_t vpz_transfer_bytes(int which);

/* Pinned host memory helpers (cudaHostAlloc / cudaFreeHost). */
void* vpz_host_alloc(size_t bytes);
void vpz_host_free(void* p);

/* ---- stage dumps for parity tests (SURVEY 8c/8d: integer stages must be bit-exact) -------- */
#define VPZ_DUMP_MAX_CH 8
typedef struct {
  int32_t status;
  int32_t mode, block_size;
  int32_t info[6];
  int32_t bits_read;
  int32_t exec_mask;
  int32_t no_execute_mask;
  int32_t scalars_n;
  int32_t classes_n;
  int32_t post_count[VPZ_DUMP_MAX_CH];
  int32_t raw_posts[VPZ_DUMP_MAX_CH][64];
  int32_t final_y[VPZ_DUMP_MAX_CH][64];
  int32_t step_flags[VPZ_DUMP_MAX_CH][64];
} vpz_packet_dump;

/* Decodes ONE audio packet on the GPU with every stage written out.  scalars/classes receive up to
 * *_cap entries (the _n fields of the dump hold the true counts); residue (before coupling) and
 * spectrum (IMDCT input) receive channels*block_size/2 floats, imdct channels*block_size floats
 * (raw, unwindowed transform output); any of the five may be NULL. */
int vpz_debug_decode_packet(vpz_ctx* ctx, vpz_setup* s, const uint8_t* pkt, size_t len,
                            vpz_packet_dump* dump, int32_t* scalars, int32_t scalars_cap,
                            int32_t* classes, int32_t classes_cap, float* residue, float* spectrum,
                            float* imdct);

/* Kernel-only IMDCT + window + overlap-add + interleaved store on caller-provided spectra
 * (BASELINE config 3).  n_streams runs of n_blocks blocks; flags[s*n_blocks+i] bit0 = long block;
 * window flags follow the Vorbis rule (prev/next flag = neighbour is long).  spectra holds, run
 * after run, block after block, channel after channel, block_size/2 floats.  The spectra stay on
 * the device; returns a handle used like a batch whose entropy stage is skipped. */
int vpz_synth_create(vpz_ctx* ctx, int channels, int log2_size0, int log2_size1, uint32_t n_streams,
                     uint32_t n_blocks, const uint8_t* flags, const float* spectra, vpz_batch** out);

/* ---- reader: IVorbisReader / IStreamDecoder surface ------------------------------------- */
/* VorbisReader(Stream) + Initialize() (VorbisReader.cs:37-66) over container bytes in memory.
 * copy != 0: the library keeps its own copy.  Fails with VPZ_E_INVALID_DATA when no Vorbis stream
 * is found (VorbisReader.cs:63). */
int vpz_reader_open_memory(vpz_ctx* ctx, const uint8_t* data, size_t len, int copy, vpz_reader** out);
void vpz_reader_close(vpz_reader* r);

int vpz_reader_stream_count(const vpz_reader* r);        /* Streams.Count */
int vpz_reader_stream_index(const vpz_reader* r);        /* StreamIndex */
int vpz_reader_switch_stream(vpz_reader* r, int index);  /* SwitchStreams (VorbisReader.cs:191-210) */
int vpz_reader_find_next_stream(vpz_reader* r);          /* FindNextStream: 1 found, 0 none */
int vpz_reader_can_seek(const vpz_reader* r);

int vpz_reader_channels(const vpz_reader* r);
int vpz_reader_sample_rate(const vpz_reader* r);
int vpz_reader_bitrate(const vpz_reader* r, int which);  /* 0 upper, 1 nominal, 2 lower */
int vpz_reader_stream_serial(const vpz_reader* r);
int64_t vpz_reader_total_samples(vpz_reader* r);
int64_t vpz_reader_sample_position(const vpz_reader* r);
int vpz_reader_is_end_of_stream(const vpz_reader* r);
int vpz_reader_has_clipped(const vpz_reader* r);
int vpz_reader_get_clip(const vpz_reader* r);
void vpz_reader_set_clip(vpz_reader* r, int clip);       /* ClipSamples, default 1 */
int64_t vpz_reader_container_overhead_bits(const vpz_reader* r);
int64_t vpz_reader_container_waste_bits(const vpz_reader* r);

/* Tags (TagData.cs): vendor string and raw "KEY=value" comments, UTF-8, not NUL terminated. */
const char* vpz_reader_vendor(const vpz_reader* r, int* len);
int vpz_reader_comment_count(const vpz_reader* r);
const char* vpz_reader_comment(const vpz_reader* r, int i, int* len);

/* IStreamDecoder.Read(Span<float>) (StreamDecoder.cs:407): interleaved; nfloats must be a multiple
 * of Channels; returns samples per channel, at most one packet's worth per call, 0 at the end. */
int vpz_reader_read(vpz_reader* r, float* buf, int nfloats);
/* IStreamDecoder.Read(Span<float>, samplesToRead, channelStride) (StreamDecoder.cs:413): planar. */
int vpz_reader_read_planar(vpz_reader* r, float* buf, int nfloats, int samples_to_read, int channel_stride);
/* SeekTo(long, SeekOrigin) (StreamDecoder.cs:817-880); origin 0 Begin, 1 Current, 2 End (Current and
 * End SUBTRACT the offset like the reference, StreamDecoder.cs:833-839). */
int vpz_reader_seek(vpz_reader* r, int64_t sample_position, int origin);
/* How many packets the reader decodes ahead per GPU batch (default 256; 0 = whole stream). */
int vpz_reader_set_lookahead(vpz_reader* r, int packets);

/* Packet access for callers that keep their own Ogg layer but want ours for tests/benchmarks:
 * audio packet i of the current stream as the packet provider hands it out. */
int vpz_reader_audio_packet_count(vpz_reader* r);
int vpz_reader_audio_packet(vpz_reader* r, int i, const uint8_t** data, uint32_t* len, int64_t* granule,
                            int32_t* flags /* bit0 resync, bit1 end of stream */);
const uint8_t* vpz_reader_header_packet(vpz_reader* r, int which, uint32_t* len); /* 0 id, 1 comment, 2 setup */
vpz_setup* vpz_reader_setup(vpz_reader* r);

/* ---- bulk: many whole files, one call (BASELINE config 4 / bench e2e) --------------------- */
/* Parses n container images on the host, queues every stream's packets (replica k of a file may
 * start at a different packet with start_packet[k], wrapping is the caller's business), decodes
 * them in one batch and leaves interleaved PCM in dst (host) when dst != NULL.  sample_counts[k]
 * receives samples per channel of file k.  Returns total floats written or a negative error. */
int64_t vpz_decode_files(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens,
                         int clip, float* dst, size_t dst_floats, int64_t* sample_counts);

/* The same with 16-bit output: every sample is converted on the GPU by the rule the reference's own
 * tests apply to the float output, v = (int)(x * 32768f) clamped to [-32768, 32767] (AssetTest.cs:131-132),
 * after ClipSamples when clip != 0.  Halves the device-to-host bytes.  Block sizes 256 / 2048 and mono /
 * stereo only (VPZ_E_UNSUPPORTED otherwise).  dst_samples / return value: int16 elements. */
int64_t vpz_decode_files_s16(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens,
                             int clip, int16_t* dst, size_t dst_samples, int64_t* sample_counts);

/* ---- physical Ogg layer on the GPU (SURVEY 8(f) row 1) ----------------------------------------------- */
/* One valid Ogg page as PageReaderBase.ReadNextPage / VerifyPage accept it (Ogg/PageReaderBase.cs:41-84,
 * 286-361): found by capture-pattern search, segment table and body inside the data, CRC-32 (Ogg/Crc.cs:20-63)
 * verified, packets counted (Ogg/PageHeader.cs:35-59). */
typedef struct {
  uint32_t offset;          /* of the page in its container image */
  uint32_t body_len;
  uint32_t granule_lo, granule_hi;
  uint32_t serial, sequence;
  uint8_t flags;            /* 1 continuation, 2 BOS, 4 EOS (Contracts/Ogg/PageFlags.cs) */
  uint8_t segments;
  uint8_t is_resync;        /* bytes were skipped in front of this page */
  uint8_t is_continued;     /* the last lacing value is 255 */
  uint16_t packet_count;
  uint16_t reserved;
} vpz_page_info;

/* Scans n container images on the GPU, one warp per image: sync search, header parse, lacing sums, page CRC.
 * The pages of image i are pages[first[i] .. first[i] + count[i]); waste_bits[i] = bits that belong to no
 * valid page (IVorbisReader.ContainerWasteBits before per-stream filtering), crc_failures[i] = candidates whose
 * CRC did not match.  Any output pointer may be NULL.  Returns the total number of pages or a negative error.
 * vpz_decode_files uses the same scan ("gpu_scan" tunable, default 1). */
int64_t vpz_scan_pages(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens,
                       vpz_page_info* pages, size_t pages_cap, uint32_t* first, uint32_t* count,
                       uint64_t* waste_bits, uint32_t* crc_failures);

/* ---- bulk random access: many short excerpts, one call (BASELINE config 5) -------------------- */
/* Excerpt i is what a fresh VorbisReader over container image file_of[i] delivers for
 *     reader.SeekTo(start[i]);  then ReadSamples until count[i] samples per channel have been read
 * (StreamDecoder.SeekTo, StreamDecoder.cs:817-880: one packet of pre-roll, roll forward inside the
 * target packet; ReadSamples: StreamDecoder.cs:418-498).  The host runs the provider side of every
 * SeekTo, the windows of a group of excerpts are decoded in one GPU batch, interleaved PCM goes to
 * dst (host): excerpt i starts at float offset dst_offsets[i] = sum over j < i of count[j] * channels
 * (fixed layout; returned in dst_offsets when non-NULL).  got[i] receives the samples per channel that
 * were delivered (fewer than count[i] at the end of the stream) or the negative vpz_status SeekTo
 * raised (VPZ_E_SEEK_RANGE, VPZ_E_PREROLL, ...); the floats of an excerpt that were not delivered are set
 * to zero.  clip: ClipSamples.  dst == NULL: only the layout is computed.  The samples are gathered on the
 * device (K4) and arrive in dst by one copy per ~2,048 excerpts: pinned dst (vpz_host_alloc) is fastest.
 * Returns the total floats of the layout or a negative error. */
int64_t vpz_decode_excerpts(vpz_ctx* ctx, uint32_t n_files, const uint8_t* const* datas, const size_t* lens,
                            uint32_t n, const uint32_t* file_of, const int64_t* start, const int32_t* count,
                            int clip, float* dst, size_t dst_floats, int64_t* dst_offsets, int32_t* got);

/* ---- bulk calls with the PCM in caller-owned device memory ----------------------------------------- */
/* Format bits of the *_device calls; 0 = fp32 interleaved (the host calls' layout). */
enum { VPZ_OUT_S16 = 1, VPZ_OUT_PLANAR = 2 };

/* vpz_decode_files / vpz_decode_excerpts with the samples written to dst_dev, device (or managed) memory of
 * the context's device, instead of host memory.  What is decoded, sample_counts / got / dst_offsets, the size
 * query (dst_dev == NULL), the errors and ClipSamples are those of the host calls.  Item k (file k, excerpt k)
 * starts at ELEMENT offset dst_offsets[k], the host calls' offsets; dst_elems and the offsets count elements
 * (4 bytes for fp32, 2 for VPZ_OUT_S16).
 *   VPZ_OUT_PLANAR: item k is channel-major, channel c at dst_offsets[k] + c * samples_k (samples_k = sample_counts[k]
 *                   for files, count[k] for excerpts); items of one channel count and one length make a dense
 *                   [n][C][T] array.  Without it, items are interleaved.
 *   VPZ_OUT_S16:    int16 elements, v = (int)(x * 32768f) clamped to [-32768, 32767] after ClipSamples, for every
 *                   stream the fp32 path decodes (any channel count and block size).
 * Samples an excerpt does not deliver (end of stream, failed SeekTo) are zero.  stream: the caller's cudaStream_t
 * (NULL: the legacy default stream); the library's work starts after the work queued on it before the call, and
 * dst_dev is complete when the call returns.  A host, pinned or other-device pointer, a too small dst_elems and
 * unknown format bits fail with VPZ_E_ARGUMENT.  The PCM is placed by one more kernel pass over the batch PCM
 * (K5) instead of a device-to-host copy; "bulk_threads_device" sets the host threads of the files call. */
int64_t vpz_decode_files_device(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens,
                                int clip, int format, void* dst_dev, size_t dst_elems,
                                int64_t* sample_counts, void* stream);
int64_t vpz_decode_excerpts_device(vpz_ctx* ctx, uint32_t n_files, const uint8_t* const* datas, const size_t* lens,
                                   uint32_t n, const uint32_t* file_of, const int64_t* start, const int32_t* count,
                                   int clip, int format, void* dst_dev, size_t dst_elems,
                                   int64_t* dst_offsets, int32_t* got, void* stream);

/* ---- the same with conversion to one sample rate and channel layout ------------------------------------------ */
typedef struct {
  int32_t format;       /* VPZ_OUT_* bits, as for the *_device calls */
  int32_t sample_rate;  /* 0: every stream keeps its rate; else 1,000..384,000 Hz: every item is converted to it */
  int32_t channels;     /* 0: keep; 1: mono = mean of the stream's channels; 2: mono duplicated, stereo kept
                           (more than 2 source channels: VPZ_E_UNSUPPORTED) */
} vpz_out_conv;

/* vpz_decode_files_device / vpz_decode_excerpts_device with every item converted to conv->sample_rate and
 * conv->channels on the device (K6), in the same last pass over the decoded PCM.  Pointer, stream and size checks,
 * the size query, the format bits and the errors are those of the *_device calls; a sample_rate outside
 * 1,000..384,000 (other than 0) or channels outside {0, 1, 2} fail with VPZ_E_ARGUMENT.
 *   Unconverted items (rate 0 or the stream's own, channels 0 or the stream's own) are bitwise what the *_device
 *   call writes.  Mono is the sum of the channels in channel order divided by C (fp32, round to nearest); at equal
 *   rates that is the output.  Rate conversion is torchaudio.functional.resample's default (sinc_interp_hann,
 *   lowpass_filter_width W = 6, rolloff 0.99) in closed form, fi -> fo, base = 0.99 * min(fi, fo):
 *     y[j] = (base / fi) * sum_k x[k] sinc(t) cos^2(pi t / 2W),  t = clamp(base (k / fi - j / fo), -W, W)
 *   with x[k] = 0 outside the delivered samples; with o / n = fi / fo in lowest terms only the 2 width + 2 taps
 *   k in [floor(j o / n) - width, floor(j o / n) + width + 1] can be nonzero, width = ceil(6 o / (0.99 min(o, n))).
 *   ClipSamples applies to the decoded samples, before mixing and the filter; fp32 output is not clipped again,
 *   int16 clamps.  A rate pair whose coefficient table exceeds 2^22 floats fails with VPZ_E_UNSUPPORTED.
 *   So does a stream whose one-output K6 tile needs more shared memory than the device allows per block (e.g. 8
 *   channels to mono from 1,000,000 Hz to 1 kHz), from the size query and the call, before anything is decoded.
 * Files: sample_counts[k] = ceil(n_k fo / fi) for a converted file (n_k: vpz_decode_files' count), dst_offsets
 *   (may be NULL) the prefix sums of sample_counts * C_out (C_out = conv->channels, or the stream's when 0).  The
 *   filter sees zeros outside the file.
 * Excerpts: start / count are output-rate samples.  A converted item reads the source window k_lo =
 *   max(0, floor(start o / n) - width), k_hi = floor((start + count - 1) o / n) + width + 1 exactly as the plain call
 *   reads (k_lo, k_hi - k_lo) (width 0 at equal rates); with d samples delivered (resampled: those before the
 *   stream's TotalSamples; the filter sees zeros from there on, as in the files call, although a reader that seeks
 *   into the last packet delivers it untrimmed) and e = k_lo + d, got = clamp(ceil(e n / o) - start, 0, count), or the negative SeekTo
 *   status.  Output samples from got on are zero.  A source window longer than the plain call takes as a count (INT32_MAX / 8 samples), or a start past
 *   2^40 samples, fails with VPZ_E_ARGUMENT.
 * channels = 2 with a source of more than 2 channels fails with VPZ_E_UNSUPPORTED before anything is decoded. */
int64_t vpz_decode_files_device_conv(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens,
                                     int clip, const vpz_out_conv* conv, void* dst_dev, size_t dst_elems,
                                     int64_t* sample_counts, int64_t* dst_offsets, void* stream);
int64_t vpz_decode_excerpts_device_conv(vpz_ctx* ctx, uint32_t n_files, const uint8_t* const* datas, const size_t* lens,
                                        uint32_t n, const uint32_t* file_of, const int64_t* start, const int32_t* count,
                                        int clip, const vpz_out_conv* conv, void* dst_dev, size_t dst_elems,
                                        int64_t* dst_offsets, int32_t* got, void* stream);

/* ---- corpus: open a set of container images once, cut excerpt batches from it many times --------------------- */
typedef struct vpz_corpus vpz_corpus;
/* Opens n container images as one corpus of the context.  Does once what every excerpt call does per call: the page
 * scan (on the device, or on the host with "gpu_scan" 0), the headers and setup tables (the corpus holds its
 * references until close), the seek index (built on the device for clean single-stream files, by the host's packet
 * walk for the rest) and each file's total samples.  The images are scanned in slices of at most "bulk_group_mib"
 * (the pinned staging never holds the whole corpus); the 4 GiB limit per image stays.  A file the plain excerpt call
 * rejects fails the open with the same code and last-error text, and *out stays NULL.
 *   copy != 0: the library keeps its own copy of the images.  copy == 0: the caller's bytes must stay valid and
 *   unchanged until vpz_corpus_close (vpz_reader_open_memory's rules).
 * A corpus belongs to its context: every call on it is a call on that context (one thread at a time), and it must be
 * closed before the context is destroyed.  The settings in effect at open ("gpu_scan", "bulk_group_mib") apply. */
int vpz_corpus_open(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens, int copy,
                    vpz_corpus** out);
void vpz_corpus_close(vpz_corpus* c);
/* Per file: channels, sample rate, TotalSamples of a fresh reader on its first logical stream (any pointer may be
 * NULL).  Returns the number of files. */
int64_t vpz_corpus_info(const vpz_corpus* c, int32_t* channels, int32_t* sample_rate, int64_t* samples);
/* Bytes of device memory the corpus holds (its images, 16-byte aligned with 16 zero bytes behind each); 0 for NULL. */
uint64_t vpz_corpus_device_bytes(const vpz_corpus* c);
/* vpz_decode_excerpts_device_conv on the corpus's files: same arguments after (n_files, datas, lens), same results.
 * Given the same images the buffer, got, dst_offsets, the size query (dst_dev == NULL), the error codes and
 * ClipSamples are bitwise those of vpz_decode_excerpts_device_conv; with conv = {format, 0, 0} that is also the plain
 * vpz_decode_excerpts_device(format).  A call costs the planning and decoding of its excerpts: nothing of a file is
 * scanned, parsed or indexed again.  NULL c: VPZ_E_ARGUMENT. */
int64_t vpz_corpus_excerpts_device(vpz_corpus* c, uint32_t n, const uint32_t* file_of, const int64_t* start,
                                   const int32_t* count, int clip, const vpz_out_conv* conv, void* dst_dev,
                                   size_t dst_elems, int64_t* dst_offsets, int32_t* got, void* stream);

/* Debug / tests: the page-end granule index SeekTo searches in (PacketProvider.FillPageEndGranuleCache,
 * Ogg/PacketProvider.cs:203-307) of one container image's first logical stream: entry p = granules up to and
 * including page p.  on_device 1: built by the GPU (page scan + one warp per file over its pages), VPZ_E_UNSUPPORTED
 * when the file is not a clean single stream (those keep the host's packet walk); 0: the host's walk.  Returns the
 * number of pages and writes min(pages, cap) entries. */
int64_t vpz_debug_page_end_granules(vpz_ctx* ctx, const uint8_t* data, size_t len, int on_device, int64_t* out, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* VPZ_H */
