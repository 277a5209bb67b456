// engine.h -- host runtime behind the C ABI: context, setup cache, packet batcher, launch plan.
// Device access goes through devapi.h only.
#pragma once
#include <stdint.h>
#include <string.h>

#include <atomic>
#include <condition_variable>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "devapi.h"
#include "setup.h"

struct vpz_ctx;
struct vpz_batch;

struct vpz_setup {
  vpz_ctx* ctx = nullptr;
  vpz::Setup host;
  std::vector<uint8_t> id_pkt, setup_pkt;
  void* d_blob = nullptr;
  int refs = 0;
  uint32_t k1_words_per_warp = 0;   // shared memory K1b needs per warp
  uint32_t rec_words = 0;           // size of one packet's symbol record (K1a -> K1b)
  bool gather_ok = false;           // K1b gather path applies (mono/stereo, residue 1/2, dims divide the partition)
  bool k1a_full = false;            // needs the K1a variant that walks floor 0 / several submaps
  uint32_t k1g_words = 0;           // shared memory of the gather path per warp (words), without the floor segment tables
  uint32_t k1g_seg_stride = 0;      // words of the floor segment table per channel (4 per post + flat tail)
  uint32_t k3_floats_per_ch = 0;    // shared memory K3 needs per channel (generic layout)
  bool fast_sizes = false;          // block sizes 256 / 2048
  bool synthetic = false;           // window/twiddle tables only (vpz_synth_create)
};

namespace vpz {
// Host worker pool for the bulk path: page scans, packet walks and the copy of packet bytes into
// pinned staging are per-stream work with no shared state.
class ThreadPool {
 public:
  explicit ThreadPool(unsigned n);
  ~ThreadPool();
  // Runs fn(0..n-1) on the workers and the calling thread; returns when all are done.
  void parallel_for(size_t n, const std::function<void(size_t)>& fn);
  unsigned size() const { return (unsigned)workers_.size() + 1; }
  // At most k threads (the caller included) take part in the parallel_for calls that follow; 0 = all.
  void set_limit(unsigned k);

 private:
  void worker(unsigned id);
  void drain();
  unsigned limit_ = 0;
  std::vector<std::thread> workers_;
  std::mutex m_;
  std::condition_variable cv_, done_cv_;
  const std::function<void(size_t)>* fn_ = nullptr;
  size_t n_ = 0;
  std::atomic<size_t> next_{0};
  size_t finished_ = 0;
  unsigned generation_ = 0, active_ = 0;
  bool stop_ = false;
};
}  // namespace vpz

namespace vpz {
struct ExcerptBufs;                  // below: buffers of the bulk random-access path (K4)
struct PlaceBufs;                    // below: tiles of the device-output bulk calls (K5)
struct ScanBufs;                     // scan.cpp: staging of the device page scan (K0)
void scan_bufs_destroy(ScanBufs* s);
struct ScanResult {                  // views into the context's scan buffers, valid until the next scan
  uint32_t n = 0;
  const VpzScanFile* files = nullptr;
  const VpzPageRec* pages = nullptr;
  const VpzScanOut* out = nullptr;
  const uint8_t* images = nullptr;   // the staged images on the device: image i at files[i].data_off
};
}  // namespace vpz

struct vpz_ctx {
  int device = 0;
  vpz::dev::Stream* stream = nullptr;
  vpz::dev::Stream* copy_stream = nullptr;   // device->host PCM copies of the bulk pipeline
  vpz::ThreadPool* pool = nullptr;           // created on first bulk call
  vpz::dev::Event* ev[4] = {nullptr, nullptr, nullptr, nullptr};   // start, after K1a, after K1b, after K3
  std::string last_error;
  int l1_bits = VPZ_L1_BITS_DEFAULT;
  int ola_chunk = 63;   // packets per K3 work item (+ the seed packet)
  bool ola_chunk_set = false;   // set by the user: do not adapt it to the batch size (pick_ola_chunk)
  int k1_warps = 4;
  int k1a_smem = 0;        // K1a: 1 = first-level Huffman tables in shared memory (vpz_k1a_symbols_sm; measured slower, k_history.md)
  int force_general = 0;   // tests: 1 = every packet through the general K1b and the generic K3, 2 = also the full K1a
  int gpu_scan = 1;        // bulk path: page scan + CRC on the device (K0); 0 = on the host worker threads
  vpz::ScanBufs* scan = nullptr;
  std::multimap<uint64_t, vpz_setup*> setups;
  std::vector<vpz_setup*> recent;     // setups the context itself holds a reference on (LRU, 64)
  uint32_t* d_counter = nullptr;
  vpz::dev::Event* marks[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int64_t kernel_launches = 0;
  // vpz_decode_files pipeline: groups of streams rotate through these batches so that host planning,
  // H2D + kernels and the D2H of finished PCM overlap; buffers persist between calls
  struct vpz_batch* bulk[3] = {nullptr, nullptr, nullptr};
  vpz::dev::Event* bulk_done[3] = {nullptr, nullptr, nullptr};   // D2H of the batch's PCM finished
  vpz::dev::Event* bulk_ready[3] = {nullptr, nullptr, nullptr};  // kernels of the batch finished
  vpz::ExcerptBufs* xb = nullptr;            // vpz_decode_excerpts: copy segments and dense output of the two groups in flight
  vpz::PlaceBufs* place = nullptr;           // *_device bulk calls: K5 tiles of the groups in flight
  int bulk_group = 256;                      // streams per pipeline group ("bulk_group" tunable)
  int bulk_group_mib = 128;                  // ... and at most this many MiB of container images ("bulk_group_mib")
  int bulk_group_bytes = 0;                  // tests: the same limit in bytes (overrides bulk_group_mib when > 0)
  int host_threads = 0;                      // size of the worker pool; 0: hardware concurrency, capped at 32
  int bulk_threads = 4;                      // of those, how many vpz_decode_files uses ("bulk_threads"; 0: all)
  int bulk_threads_device = 8;               // ... and vpz_decode_files_device ("bulk_threads_device"; 0: all)
};

namespace vpz {

template <typename T>
struct HostBuf {   // growable pinned staging
  T* p = nullptr;
  size_t n = 0, cap = 0;
  ~HostBuf() { dev::host_free(p); }
  bool reserve(size_t want) {
    if (want <= cap) return true;
    size_t nc = cap ? cap : 1024;
    while (nc < want) nc *= 2;
    T* np = static_cast<T*>(dev::host_alloc(nc * sizeof(T)));
    if (!np) return false;
    if (n) memcpy(np, p, n * sizeof(T));
    dev::host_free(p);
    p = np;
    cap = nc;
    return true;
  }
  bool push(const T& v) {
    if (!reserve(n + 1)) return false;
    p[n++] = v;
    return true;
  }
  void clear() { n = 0; }
};

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  ~DevBuf() { dev::free(p); }
  bool reserve(size_t bytes, std::string& err) {
    if (bytes <= cap) return true;
    dev::free(p);
    p = nullptr;
    cap = 0;
    size_t nc = bytes + bytes / 8 + 256;
    p = dev::alloc(nc, err);
    if (!p) return false;
    cap = nc;
    return true;
  }
};

struct ExcerptBufs {
  HostBuf<VpzCopySeg> h_segs[2];
  DevBuf d_segs[2], d_out[2];
  dev::Event* ready[2] = {nullptr, nullptr};   // kernels of the group finished
  dev::Event* done[2] = {nullptr, nullptr};    // its output has reached the caller's buffer
  ~ExcerptBufs() {
    for (int i = 0; i < 2; i++) {
      dev::event_destroy(ready[i]);
      dev::event_destroy(done[i]);
    }
  }
};

struct ConvFilter {   // K6 coefficient table of one rate pair: 2 width + 2 taps x n phases (tap-major), uploaded once
  int fi = 0, fo = 0;
  uint32_t o = 1, n = 1, width = 0;
  std::vector<float> host;
  DevBuf dev;
};

struct PlaceBufs {   // one slot per pipeline batch (vpz_decode_files_device: 3, vpz_decode_excerpts_device: 2)
  HostBuf<VpzPlaceTile> h_tiles[3];
  DevBuf d_tiles[3];
  HostBuf<VpzConvTile> h_ctiles[3];   // the *_conv calls: K6 tiles
  DevBuf d_ctiles[3];
  DevBuf d_scratch[2];                // vpz_decode_excerpts_device_conv: source windows of converted excerpts (K5 -> K6)
  std::vector<std::unique_ptr<ConvFilter>> filters;   // by rate pair, kept across calls
};

struct PktSrc {
  const uint8_t* p;
  uint32_t len;
};

// Everything batch_add_run decides about one run, computed WITHOUT touching the batch so that many
// runs can be planned on worker threads and committed in one go (batch_commit).
struct RunPlan {
  vpz_setup* setup = nullptr;
  std::vector<PktSrc> src;          // decodable packets, in order
  std::vector<uint32_t> byte_off;   // staged offset of each, relative to the run's byte base
  std::vector<uint32_t> ent_off;    // uint16 offset of each packet's entry-index area, relative to the run
  uint64_t ent_total = 0;
  std::vector<VpzPktOla> ola;       // spec_off relative to the run's spectrum base, out_off in samples
  std::vector<int32_t> counts;      // per SUBMITTED packet
  uint64_t staged_bytes = 0, payload_bytes = 0, spec_floats = 0;
  int64_t samples = 0;
  int status = 0;
  int32_t stop_packet = -1;
};

struct Run {
  vpz_setup* setup = nullptr;
  int slot = 0;
  uint32_t first_valid = 0, n_valid = 0;     // range in the batch packet arrays
  std::vector<int32_t> counts;               // per submitted packet
  int64_t samples = 0;
  uint64_t out_base = 0;                     // float offset in the PCM buffer
  int status = 0;                            // 0 or VPZ_E_REF_FAULT (run cut short)
  int32_t stop_packet = -1;                  // submitted-packet index where the run was cut
};

}  // namespace vpz

struct vpz_batch {
  vpz_ctx* ctx = nullptr;
  vpz::HostBuf<uint8_t> bytes;
  vpz::HostBuf<VpzPktIn> pkts_in;
  vpz::HostBuf<VpzPktOla> pkts_ola;
  vpz::HostBuf<VpzOlaItem> items;
  std::vector<vpz::Run> runs;
  std::vector<vpz_setup*> slots;
  uint64_t total_floats = 0, spec_floats = 0;
  uint64_t payload_bytes = 0;
  uint64_t rec_words = 0, ent_total = 0;      // symbol records / entry indices of all packets
  vpz::HostBuf<uint32_t> order;               // K1 packet order (by kernel class, (setup, block size), then byte length)
  std::vector<uint32_t> sort_key;             // per packet: (setup slot * 2 + short) << 13 | length key, written while the batch is filled
  // Kernel paths are chosen per SETUP, not per batch: the order array is cut into three classes
  //   0: simple K1a + gather K1b   1: simple K1a + general K1b   2: full K1a + general K1b
  // and the K3 work items into fast (256 / 2048, <= 2 channels) and generic ones (items_sorted).
  uint32_t n_class[3] = {0, 0, 0};
  vpz::HostBuf<VpzOlaItem> items_sorted;
  uint32_t n_items_fast = 0;
  vpz::DevBuf d_rec, d_ent, d_order;
  int max_channels = 1;
  bool uploaded = false, synthetic = false, decoded = false;
  vpz::DevBuf d_bytes, d_pkts_in, d_pkts_ola, d_items, d_res, d_spec, d_pcm, d_clip, d_setups;
  vpz::HostBuf<const void*> h_setups;
  vpz::HostBuf<uint32_t> h_clip;
  bool clip_fetched = false;
  // corpus calls (vpz_corpus_excerpts_device): set before batch_commit on an empty batch, K7 writes the packet bytes
  // from the corpus's device images.  batch_commit then lays the packets out but stages none of their bytes (their
  // layout size goes to gather_bytes, `bytes` stays empty) and calls gather_fill(plan, byte base of its run) from
  // the thread that fills that plan, which writes the plan's pieces (one per packet and page) into `pieces`;
  // batch_upload uploads the pieces instead of the bytes and launches K7.
  const uint8_t* gather_images = nullptr;
  uint64_t gather_bytes = 0;
  std::function<void(size_t, uint64_t)> gather_fill;
  vpz::HostBuf<VpzGatherPiece> pieces;
  vpz::DevBuf d_pieces;
  float ms_k1 = 0, ms_k1a = 0, ms_k1b = 0, ms_k3 = 0, ms_total = 0;
  int launches = 0;
  // debug plumbing (vpz_debug_decode_packet)
  K1Debug dbg = {nullptr, nullptr, 0, nullptr, 0, nullptr};
  float* dbg_imdct = nullptr;
  vpz_setup* owned_setup = nullptr;  // synthetic batches own their table-only setup
};

namespace vpz {
int setup_create(vpz_ctx* ctx, const uint8_t* id_pkt, size_t id_len, const uint8_t* setup_pkt, size_t setup_len,
                 vpz_setup** out);
// same, with fnv1a64(setup, fnv1a64(id)) already computed (the bulk path hashes on worker threads)
int setup_create_hashed(vpz_ctx* ctx, uint64_t hash, const uint8_t* id_pkt, size_t id_len, const uint8_t* setup_pkt,
                        size_t setup_len, vpz_setup** out);
int setup_create_synthetic(vpz_ctx* ctx, int channels, int lg0, int lg1, vpz_setup** out);
void setup_release(vpz_setup* s);
int batch_add_run(vpz_batch* b, vpz_setup* s, const uint8_t* bytes, const uint32_t* offsets, uint32_t n_pkts,
                  const int32_t* trim);
// Pure planning of one run (thread-safe; `err` receives the text on failure).
int plan_run(vpz_setup* s, const PktSrc* pk, uint32_t n_pkts, const int32_t* trim, RunPlan* out, std::string* err);
// Appends planned runs to the batch: serial prefix sums, then the copies on `pool` (may be NULL).
// first_run receives the index of plans[0]'s run.
int batch_commit(vpz_batch* b, RunPlan* const* plans, size_t n, ThreadPool* pool, int* first_run);
uint32_t pick_ola_chunk(const vpz_ctx* ctx, uint64_t total_packets);
extern double g_trace_ms[4];   // VPZ_TRACE: host milliseconds inside batch_upload / batch_decode (engine.cpp)
int batch_upload(vpz_batch* b);
int batch_decode(vpz_batch* b, int clip, int out16 = 0);   // out16: 16-bit PCM (fast IMDCT kernel only)
int batch_fetch_clip(vpz_batch* b);
void batch_drop_slots(vpz_batch* b);   // releases the setup references the batch's slots hold
// K0: physical Ogg page scan of n container images on the device (scan.cpp)
int scan_pages(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens, ThreadPool* pool, ScanResult* res);
// the same in two halves, two slots (0 / 1): begin stages, uploads and launches without waiting; end collects
int scan_begin(vpz_ctx* ctx, int which, uint32_t n, const uint8_t* const* datas, const size_t* lens, ThreadPool* pool);
int scan_end(vpz_ctx* ctx, int which, ScanResult* res);
// K0g: page-end granule index of files of the slot's last scan (scan.cpp)
int granule_index(vpz_ctx* ctx, int which, const VpzGranFile* gf, uint32_t n, const long long** out);
}  // namespace vpz

// First statement of every extern "C" entry point that may touch the device: the CUDA current device
// is per host thread, and a process may hold one context per GPU.
#define VPZ_USE(ctx) vpz::dev::make_current((ctx)->device)
