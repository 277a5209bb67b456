// engine.cpp -- setup cache, packet batcher and launch plan (host side of the batch layer).
#include "engine.h"

#include <math.h>
#include <string.h>

#include <algorithm>
#include <chrono>

#include "../../include/vpz.h"
#include "bitreader.h"

namespace vpz {

double g_trace_ms[4] = {0, 0, 0, 0};   // VPZ_TRACE: batch_upload sort, batch_upload copies, batch_decode launches, spare
static double trace_now() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// vectors * partitions of one residue instance in a long block (units of K1a / K1b)
static size_t instance_units(const Setup& st, const VpzResidue& r) {
  const VpzSetupHdr* h = st.hdr();
  const int half_max = 1 << (h->log2_size1 - 1);
  const int nvec = r.type == 2 ? 1 : r.nch;
  const int64_t vlen = r.type == 2 ? (int64_t)half_max * r.nch : half_max;
  const int64_t b = std::min<int64_t>(r.begin, vlen), e = std::min<int64_t>(r.end, vlen);
  const int64_t parts = e > b ? (e - b) / r.part_size : 0;
  return (size_t)(parts * nvec);
}
// the largest residue instance of the setup
static size_t max_units(const Setup& st) {
  const VpzSetupHdr* h = st.hdr();
  const VpzResidue* rs = reinterpret_cast<const VpzResidue*>(st.blob.data() + h->residues_off);
  size_t units = 0;
  for (int i = 0; i < h->nresidues; i++) units = std::max(units, instance_units(st, rs[i]));
  return units;
}
// words of the class bytes in a packet's symbol record: the submaps of a mapping follow each other, each
// rounded up to whole words (K1a clears them word-wise)
static size_t max_class_words(const Setup& st) {
  const VpzSetupHdr* h = st.hdr();
  const VpzResidue* rs = reinterpret_cast<const VpzResidue*>(st.blob.data() + h->residues_off);
  const VpzMapping* mp = reinterpret_cast<const VpzMapping*>(st.blob.data() + h->mappings_off);
  size_t words = 0;
  for (int i = 0; i < h->nmappings; i++) {
    size_t w = 0;
    for (int j = 0; j < mp[i].submaps; j++) w += (instance_units(st, rs[mp[i].submap_residue[j]]) + 3) / 4;
    words = std::max(words, w);
  }
  return words;
}

static int fl_type(const Setup& st, int i) {
  const VpzSetupHdr* h = st.hdr();
  return reinterpret_cast<const VpzFloor1*>(st.blob.data() + h->floors_off)[i].floor_type;
}

// Kernel class of a setup (engine.h, vpz_batch::n_class) and whether its K3 items take the fast kernel
static int k1_class(const vpz_ctx* ctx, const vpz_setup* s) {
  if (s->k1a_full || ctx->force_general >= 2) return 2;
  if (!s->gather_ok || ctx->force_general >= 1) return 1;
  return 0;
}
static bool k3_fast(const vpz_ctx* ctx, const vpz_setup* s) {
  return s->fast_sizes && s->host.id.channels <= 2 && ctx->force_general == 0;
}

// K1b shared memory per warp: swizzled residue (one pad word per 32) + unit start offsets
static uint32_t k1_words(const Setup& st) {
  const VpzSetupHdr* h = st.hdr();
  const size_t n = (size_t)h->channels << (h->log2_size1 - 1);
  size_t words = n + (n >> 5) + 1 + (512 + 32) + 512 + 512 + 8 + 8;  // res, ustart, uinfo, uvq, scan
  return (uint32_t)((words + 31) & ~(size_t)31);
}

static int finish_setup(vpz_ctx* ctx, vpz_setup* s) {
  const VpzSetupHdr* h = s->host.hdr();
  s->fast_sizes = h->log2_size0 == 8 && h->log2_size1 == 11;
  s->k3_floats_per_ch = (1u << h->log2_size1) + 3u * (1u << (h->log2_size1 - 2)) + 16u;  // scratch + 3 half-slots
  if (!s->synthetic) {
    const size_t units = max_units(s->host);
    if (units > 512) {  // K1_MAX_UNITS
      ctx->last_error = "more than 512 residue partitions per packet are not on the GPU path";
      return VPZ_E_UNSUPPORTED;
    }
    s->k1_words_per_warp = k1_words(s->host);
    // K1b gather path (k1_symbols.cuh): mono / stereo, residue 1 / 2, VQ dimensions that divide the
    // partition size and, for the interleaved type 2 vector of a stereo stream, are even
    {
      const Setup& st = s->host;
      const int C = h->channels;
      const VpzResidue* rs = reinterpret_cast<const VpzResidue*>(st.blob.data() + h->residues_off);
      const VpzBook* bk = reinterpret_cast<const VpzBook*>(st.blob.data() + h->books_off);
      bool ok = C <= 2 && h->nbooks <= 256 && h->log2_size0 >= 5;
      int max_stages = 1;
      for (int i = 0; i < h->nresidues && ok; i++) {
        if (rs[i].type != 1 && rs[i].type != 2) ok = false;
        // a thread gathers chunks of 8 positions (16 for the interleaved stereo vector): chunks must
        // not straddle partitions and every VQ dimension must be a power of two that divides the chunk
        const int chunk = rs[i].type == 2 && C == 2 ? 16 : 8;
        if ((rs[i].begin % chunk) || (rs[i].part_size % chunk)) ok = false;
        // K1b's phase B scans the entry counts of two stages in one 32-bit prefix sum: 32 units of a stage
        // must stay below 2^16 entries (a unit has at most part_size of them)
        if (rs[i].part_size > 2047) ok = false;
        max_stages = std::max<int>(max_stages, rs[i].max_stages);
        for (int c = 0; c < rs[i].classifications && ok; c++)
          for (int sg = 0; sg < 8 && ok; sg++)
            if (((rs[i].cascade[c] >> sg) & 1) && rs[i].has_books[c]) {
              const int dims = bk[rs[i].books[c][sg]].dims;
              if (dims < 1 || (dims & (dims - 1)) || dims > chunk) ok = false;
            }
      }
      // floor 0 curves and mappings with several submaps live on the general path only
      const VpzMapping* mp = reinterpret_cast<const VpzMapping*>(st.blob.data() + h->mappings_off);
      for (int i = 0; i < h->nmappings; i++) s->k1a_full = s->k1a_full || mp[i].submaps > 1;
      for (int i = 0; i < h->nfloors; i++) s->k1a_full = s->k1a_full || fl_type(st, i) == 0;
      s->gather_ok = ok && !s->k1a_full;
      const size_t U = (units + 31) & ~(size_t)31;
      const size_t half_max = (size_t)1 << (h->log2_size1 - 1);
      // k1b gather layout per warp: urec stages*U*2 + ybuf C*half_max/4 + sg C*4*66 (+ pad, multiple of 32)
      // segments per channel <= posts of the largest floor (+ the flat tail): the segment table is sized for this setup
      const VpzFloor1* fl = reinterpret_cast<const VpzFloor1*>(st.blob.data() + h->floors_off);
      size_t max_posts = 2;
      for (int i = 0; i < h->nfloors; i++) max_posts = std::max<size_t>(max_posts, fl[i].xcount);
      s->k1g_seg_stride = (uint32_t)(4 * (max_posts + 1));
      // without the segment tables: a batch sizes those by the LARGEST floor among its gather setups (batch_decode)
      s->k1g_words = (uint32_t)((size_t)max_stages * U * 2 + (size_t)C * half_max / 4);
    }
    // K1_REC_HDR, K1_SEG_WORDS, classes; a multiple of 4 words so every record starts on a 16-byte boundary
    // + 16 with several submaps: the per-submap entry ends K1a leaves behind the class bytes
    bool multi_sub = false;
    {
      const VpzMapping* mp = reinterpret_cast<const VpzMapping*>(s->host.blob.data() + h->mappings_off);
      for (int i = 0; i < h->nmappings; i++) multi_sub = multi_sub || mp[i].submaps > 1;
    }
    s->rec_words = (uint32_t)((4 + h->channels * 68 + max_class_words(s->host) + 1 + (multi_sub ? 16 : 0) + 3) & ~(size_t)3);
  }
  size_t bytes = s->host.blob.size() * 4;
  s->d_blob = dev::alloc(bytes, ctx->last_error);
  if (!s->d_blob) return VPZ_E_CUDA;
  int rc = dev::h2d(s->d_blob, s->host.blob.data(), bytes, ctx->stream, ctx->last_error);
  if (rc) return rc;
  return dev::stream_sync(ctx->stream, ctx->last_error);
}

int setup_create(vpz_ctx* ctx, const uint8_t* id_pkt, size_t id_len, const uint8_t* setup_pkt, size_t setup_len,
                 vpz_setup** out) {
  return setup_create_hashed(ctx, fnv1a64(setup_pkt, setup_len, fnv1a64(id_pkt, id_len)), id_pkt, id_len, setup_pkt,
                             setup_len, out);
}

int setup_create_hashed(vpz_ctx* ctx, uint64_t h, const uint8_t* id_pkt, size_t id_len, const uint8_t* setup_pkt,
                        size_t setup_len, vpz_setup** out) {
  auto range = ctx->setups.equal_range(h);
  for (auto it = range.first; it != range.second; ++it) {
    vpz_setup* s = it->second;
    if (s->id_pkt.size() == id_len && s->setup_pkt.size() == setup_len &&
        memcmp(s->id_pkt.data(), id_pkt, id_len) == 0 && memcmp(s->setup_pkt.data(), setup_pkt, setup_len) == 0) {
      s->refs++;
      *out = s;
      return VPZ_OK;
    }
  }
  vpz_setup* s = new vpz_setup;
  s->ctx = ctx;
  int rc = s->host.parse(id_pkt, id_len, setup_pkt, setup_len, ctx->l1_bits);
  if (rc) {
    ctx->last_error = s->host.error;
    delete s;
    return rc;
  }
  s->id_pkt.assign(id_pkt, id_pkt + id_len);
  s->setup_pkt.assign(setup_pkt, setup_pkt + setup_len);
  rc = finish_setup(ctx, s);
  if (rc) {
    dev::free(s->d_blob);
    delete s;
    return rc;
  }
  s->refs = 1;
  ctx->setups.insert({h, s});
  // the context keeps recently built tables alive (parse + upload once per distinct setup even
  // when every stream that used it has been closed in between)
  s->refs++;
  ctx->recent.push_back(s);
  if (ctx->recent.size() > 64) {
    vpz_setup* old = ctx->recent.front();
    ctx->recent.erase(ctx->recent.begin());
    setup_release(old);
  }
  *out = s;
  return VPZ_OK;
}

// Tables for kernel-only IMDCT runs on caller-provided spectra: window slopes + twiddles only.
int setup_create_synthetic(vpz_ctx* ctx, int channels, int lg0, int lg1, vpz_setup** out) {
  if (channels < 1 || channels > VPZ_MAX_CH || lg0 < 6 || lg1 < lg0 || lg1 > 13) {
    ctx->last_error = "synthetic setup: channels 1..8, block sizes 64..8192";
    return VPZ_E_ARGUMENT;
  }
  vpz_setup* s = new vpz_setup;
  s->ctx = ctx;
  s->synthetic = true;
  Setup& st = s->host;
  st.id.channels = channels;
  st.id.size0 = 1 << lg0;
  st.id.size1 = 1 << lg1;
  std::vector<uint32_t>& blob = st.blob;
  blob.assign((sizeof(VpzSetupHdr) + 3) / 4, 0u);
  while (blob.size() % 4) blob.push_back(0);
  VpzSetupHdr h;
  memset(&h, 0, sizeof(h));
  h.magic = 0x315A5056u;
  h.channels = (uint8_t)channels;
  h.log2_size0 = (uint8_t)lg0;
  h.log2_size1 = (uint8_t)lg1;
  for (int w = 0; w < 2; w++) {
    int size = 1 << (w ? lg1 : lg0), M = size / 2, H = size / 4;
    std::vector<float> slope((size_t)M), tw((size_t)2 * H), roots((size_t)2 * H);
    window_slope(slope.data(), M);
    for (int n = 0; n < H; n++) {
      double a = -M_PI * ((double)n + 0.125) / (double)M, b = -2.0 * M_PI * (double)n / (double)H;
      tw[2 * n] = (float)cos(a);
      tw[2 * n + 1] = (float)sin(a);
      roots[2 * n] = (float)cos(b);
      roots[2 * n + 1] = (float)sin(b);
    }
    auto put = [&](const std::vector<float>& v) {
      while (blob.size() % 4) blob.push_back(0);
      uint32_t off = (uint32_t)blob.size();
      blob.resize(blob.size() + v.size());
      memcpy(&blob[off], v.data(), v.size() * 4);
      return off;
    };
    h.slope_off[w] = put(slope);
    h.tw_off[w] = put(tw);
    h.fft_off[w] = put(roots);
  }
  h.total_words = (uint32_t)blob.size();
  memcpy(blob.data(), &h, sizeof(h));
  int rc = finish_setup(ctx, s);
  if (rc) {
    dev::free(s->d_blob);
    delete s;
    return rc;
  }
  s->refs = 1;
  *out = s;
  return VPZ_OK;
}

void setup_release(vpz_setup* s) {
  if (!s) return;
  if (--s->refs > 0) return;
  vpz_ctx* ctx = s->ctx;
  for (auto it = ctx->setups.begin(); it != ctx->setups.end(); ++it)
    if (it->second == s) {
      ctx->setups.erase(it);
      break;
    }
  dev::free(s->d_blob);
  delete s;
}

static int slot_of(vpz_batch* b, vpz_setup* s) {
  for (size_t i = 0; i < b->slots.size(); i++)
    if (b->slots[i] == s) return (int)i;
  // the batch holds a reference for as long as the slot exists (vpz_batch_reset / destroy drop it): the
  // caller may release its own handle right after add_run, and the context's LRU may evict the setup
  s->refs++;
  b->slots.push_back(s);
  return (int)b->slots.size() - 1;
}

void batch_drop_slots(vpz_batch* b) {
  for (vpz_setup* s : b->slots)
    if (s != b->owned_setup) setup_release(s);
  b->slots.clear();
}

// ---- host worker pool -----------------------------------------------------------------------
ThreadPool::ThreadPool(unsigned n) {
  for (unsigned i = 1; i < n; i++) workers_.emplace_back([this, i] { worker(i); });
}
ThreadPool::~ThreadPool() {
  {
    std::lock_guard<std::mutex> lk(m_);
    stop_ = true;
  }
  cv_.notify_all();
  for (auto& t : workers_) t.join();
}
void ThreadPool::drain() {
  for (;;) {
    size_t i = next_.fetch_add(1);
    if (i >= n_) break;
    (*fn_)(i);
  }
}
void ThreadPool::set_limit(unsigned k) {
  std::lock_guard<std::mutex> lk(m_);
  limit_ = k;
}
void ThreadPool::worker(unsigned id) {
  unsigned seen = 0;
  for (;;) {
    bool take;
    {
      std::unique_lock<std::mutex> lk(m_);
      cv_.wait(lk, [&] { return stop_ || generation_ != seen; });
      if (stop_) return;
      seen = generation_;
      take = limit_ == 0 || id < limit_;   // the caller is thread 0
    }
    if (take) drain();
    {
      std::lock_guard<std::mutex> lk(m_);
      if (--active_ == 0) done_cv_.notify_all();
    }
  }
}
void ThreadPool::parallel_for(size_t n, const std::function<void(size_t)>& fn) {
  if (n == 0) return;
  if (workers_.empty() || n == 1) {
    for (size_t i = 0; i < n; i++) fn(i);
    return;
  }
  {
    std::lock_guard<std::mutex> lk(m_);
    fn_ = &fn;
    n_ = n;
    next_.store(0);
    active_ = (unsigned)workers_.size();
    generation_++;
  }
  cv_.notify_all();
  drain();
  std::unique_lock<std::mutex> lk(m_);
  done_cv_.wait(lk, [&] { return active_ == 0; });
}

// Plans one run: which packets decode, where their spectra and samples go.  Mirrors the
// bookkeeping of StreamDecoder.ReadNextPacket (StreamDecoder.cs:640-694) for a decoder that starts
// from ResetDecoder state.  Pure: touches neither the batch nor the context.
int plan_run(vpz_setup* s, const PktSrc* pk, uint32_t n_pkts, const int32_t* trim, RunPlan* out, std::string* err) {
  const Setup& st = s->host;
  const int C = st.id.channels;
  out->setup = s;
  out->counts.assign(n_pkts, 0);
  out->src.reserve(n_pkts);
  out->byte_off.reserve(n_pkts);
  out->ent_off.reserve(n_pkts);
  out->ola.reserve(n_pkts);
  bool have_prev = false;
  int prev_rs = 0, prev_re = 0, prev_half = 0;
  int64_t pos = 0;  // samples emitted so far by this run
  uint64_t staged = 0;
  for (uint32_t i = 0; i < n_pkts; i++) {
    const uint8_t* p = pk[i].p;
    const uint32_t len = pk[i].len;
    PacketGeom g = st.packet_geometry(p, len);
    if (g.bad_mode) {
      if (err) *err = "Unused mode index.";  // StreamDecoder.cs:734
      return VPZ_E_INVALID_DATA;
    }
    if (!g.valid) continue;
    int rs = g.right_start;
    if (trim && trim[i] > 0) rs = std::max(rs - trim[i], 0);
    // negative trim: also emit that many samples of the raw right half (the drain of
    // StreamDecoder.cs:451-455 when the end-of-stream packet that follows cannot be decoded)
    if (trim && trim[i] < 0) rs = std::min(rs - trim[i], g.right_end);
    int count = 0;
    if (have_prev && prev_rs < prev_half) {
      // K3 keeps only the low half of the previous block's D (the right half of its output); a
      // RightStart pulled back into the left half happens for the end-of-stream packet only, which
      // has no successor in the reference (StreamDecoder.cs:439-447)
      if (err) *err = "a packet follows one whose RightStart was trimmed into the left half";
      return VPZ_E_ARGUMENT;
    }
    if (have_prev) {
      int L = prev_re - prev_rs;
      int slope_len = (g.left_use_size1 ? st.id.size1 : st.id.size0) / 2;
      if (L > slope_len || L < 0 || g.left_start + L > st.id.size1 || rs < g.left_start) {
        // the reference slices windowSlope.AsSpan(0, L) and throws (SURVEY quirk Q4); the run ends here
        out->status = VPZ_E_REF_FAULT;
        out->stop_packet = (int32_t)i;
        break;
      }
      count = rs - g.left_start;
    }
    // staged layout: 16-byte aligned start (K1a fetches the packet in 16-byte chunks), at least 12 zero bytes
    // after the end (a peek reads up to two words ahead of the cursor)
    const uint64_t end = (staged + len + 12 + 15) & ~(uint64_t)15;
    const int M = g.block_size / 2;
    VpzPktOla ola;
    memset(&ola, 0, sizeof(ola));
    if (len > (1u << 24)) {   // K1b keeps entry indices of a packet in 28 bits (8 * len + 8 of them at most)
      if (err) *err = "audio packet larger than 16 MiB is not on the GPU path";
      return VPZ_E_UNSUPPORTED;
    }
    if (out->spec_floats + (uint64_t)C * M > 0xffffff00ull || end > 0xfffffff0ull || pos > 0x7fffffff) {
      if (err) *err = "run exceeds 2^32 spectrum floats / 4 GiB of packet bytes; split it";
      return VPZ_E_ARGUMENT;
    }
    ola.spec_off = (uint32_t)out->spec_floats;
    ola.out_off = (uint32_t)pos;
    ola.left_start = (uint16_t)g.left_start;
    ola.right_start = (uint16_t)rs;
    ola.right_end = (uint16_t)g.right_end;
    ola.flags = (uint8_t)((g.long_block ? VPZ_OLA_LONG : 0) | (g.left_use_size1 ? VPZ_OLA_LEFT1 : 0) |
                          (have_prev ? 0 : VPZ_OLA_NOOUT));
    out->src.push_back(PktSrc{p, len});
    out->byte_off.push_back((uint32_t)staged);
    // every codeword is at least one bit long: 8 * len bounds the entry indices of the packet
    out->ent_off.push_back((uint32_t)out->ent_total);
    out->ent_total += ((uint64_t)len * 8 + 8 + 3) & ~(uint64_t)3;   // multiple of 4: K1a stores 4 indices at a time
    out->ola.push_back(ola);
    staged = end;
    out->payload_bytes += len;
    out->spec_floats += (uint64_t)C * M;
    out->counts[i] = count;
    pos += count;
    have_prev = true;
    prev_rs = rs;
    prev_re = g.right_end;
    prev_half = M;
  }
  out->staged_bytes = staged;
  out->samples = pos;
  return VPZ_OK;
}

// Packets per K3 work item.  Every item re-transforms its predecessor packet as the overlap seed, so
// long items are cheaper; but the IMDCT kernel runs 12 workers per SM, and a batch with few packets
// should still hand every worker about two items.  A user-set "ola_chunk" is taken as is.
uint32_t pick_ola_chunk(const vpz_ctx* ctx, uint64_t total_packets) {
  if (ctx->ola_chunk_set) return (uint32_t)std::max(1, ctx->ola_chunk);
  const uint64_t workers = (uint64_t)std::max(1, dev::sm_count()) * 12u;
  const uint64_t want = (total_packets + 2 * workers - 1) / (2 * workers);
  return (uint32_t)std::min<uint64_t>(63, std::max<uint64_t>(16, want));
}

int batch_commit(vpz_batch* b, RunPlan* const* plans, size_t n, ThreadPool* pool, int* first_run) {
  vpz_ctx* ctx = b->ctx;
  if (b->synthetic) {
    ctx->last_error = "packet runs cannot be added to a synthetic batch";
    return VPZ_E_INVALID_OP;
  }
  if (first_run) *first_run = (int)b->runs.size();
  if (n == 0) return VPZ_OK;
  uint64_t commit_pkts = 0;
  for (size_t i = 0; i < n; i++) commit_pkts += plans[i]->src.size();
  // one run at a time (batch layer): the batch total is unknown, keep the long items
  const uint32_t chunk = n > 1 ? pick_ola_chunk(ctx, commit_pkts) : (uint32_t)std::max(1, ctx->ola_chunk);
  struct Base {
    uint64_t bytes, spec, out, rec, ent;
    size_t pkt, item;
    int slot;
  };
  std::vector<Base> base(n);
  uint64_t bytes = (b->bytes.n + 3) & ~(size_t)3, spec = b->spec_floats, out = b->total_floats;
  uint64_t rec = b->rec_words, ent = b->ent_total;
  size_t pkt = b->pkts_in.n, item = b->items.n;
  for (size_t i = 0; i < n; i++) {
    const RunPlan& p = *plans[i];
    if (p.setup->synthetic) {
      ctx->last_error = "packet runs cannot use a synthetic setup";
      return VPZ_E_INVALID_OP;
    }
    base[i] = Base{bytes, spec, out, rec, ent, pkt, item, slot_of(b, p.setup)};
    const size_t nv = p.src.size();
    rec += (uint64_t)nv * p.setup->rec_words;
    ent += p.ent_total;
    bytes += p.staged_bytes;
    spec += p.spec_floats;
    out += (uint64_t)p.samples * p.setup->host.id.channels;
    pkt += nv;
    item += nv > 1 ? (nv - 1 + chunk - 1) / chunk : 0;
    b->max_channels = std::max(b->max_channels, p.setup->host.id.channels);
  }
  if (spec > 0xffffff00ull || bytes > 0xfffffff0ull || rec > 0xffffff00ull || ent > 0xffffff00ull) {
    ctx->last_error = "batch exceeds 2^32 spectrum floats / 4 GiB of packet bytes; split it";
    return VPZ_E_ARGUMENT;
  }
  const size_t old_bytes = b->bytes.n;
  const bool gather = b->gather_images != nullptr;   // K7 writes the bytes: nothing to stage
  if ((!gather && !b->bytes.reserve(bytes)) || !b->pkts_in.reserve(pkt) || !b->pkts_ola.reserve(pkt) ||
      !b->items.reserve(item))
    return VPZ_E_NOMEM;
  b->sort_key.resize(pkt);
  if (!gather) memset(b->bytes.p + old_bytes, 0, (size_t)base[0].bytes - old_bytes);
  auto fill = [&](size_t i) {
    const RunPlan& p = *plans[i];
    const Base& bs = base[i];
    const size_t nv = p.src.size();
    uint8_t* dst = gather ? nullptr : b->bytes.p + bs.bytes;
    for (size_t k = 0; k < nv; k++) {
      const uint32_t off = p.byte_off[k], len = p.src[k].len;
      const uint32_t next = k + 1 < nv ? p.byte_off[k + 1] : (uint32_t)p.staged_bytes;
      if (!gather) {
        if (len) memcpy(dst + off, p.src[k].p, len);
        memset(dst + off + len, 0, next - off - len);
      }
      VpzPktIn in;
      in.byte_off = (uint32_t)(bs.bytes + off);
      in.byte_len = len;
      in.spec_off = (uint32_t)(bs.spec + p.ola[k].spec_off);
      in.setup_slot = (uint32_t)bs.slot;
      in.rec_off = (uint32_t)(bs.rec + (uint64_t)k * p.setup->rec_words);
      in.ent_off = (uint32_t)(bs.ent + p.ent_off[k]);
      in.pad[0] = in.pad[1] = 0;
      b->pkts_in.p[bs.pkt + k] = in;
      VpzPktOla ola = p.ola[k];
      ola.spec_off = in.spec_off;
      b->pkts_ola.p[bs.pkt + k] = ola;
      // K1a order key: (setup slot, short block) group, then longest packets first
      b->sort_key[bs.pkt + k] = (((uint32_t)bs.slot * 2u + ((ola.flags & VPZ_OLA_LONG) ? 0u : 1u)) << 13) |
                                (4096u - std::min<uint32_t>(len >> 2, 4096u));
    }
    if (gather) b->gather_fill(i, bs.bytes);
    // K3 work items: packets 1..nv-1 emit; each item re-runs its predecessor as carry seed
    size_t it_idx = bs.item;
    for (size_t k = 1; k < nv; k += chunk) {
      VpzOlaItem it;
      it.first_pkt = (uint32_t)(bs.pkt + k);
      it.n_pkts = (uint32_t)std::min<size_t>(chunk, nv - k);
      it.has_pre = 1;
      it.setup_slot = (uint32_t)bs.slot;
      it.out_base = bs.out;
      b->items.p[it_idx++] = it;
    }
  };
  if (pool && n > 1)
    pool->parallel_for(n, fill);
  else
    for (size_t i = 0; i < n; i++) fill(i);
  if (gather)
    b->gather_bytes = bytes;
  else
    b->bytes.n = bytes;
  b->pkts_in.n = b->pkts_ola.n = pkt;
  b->items.n = item;
  b->spec_floats = spec;
  b->total_floats = out;
  b->rec_words = rec;
  b->ent_total = ent;
  for (size_t i = 0; i < n; i++) {
    RunPlan& p = *plans[i];
    Run run;
    run.setup = p.setup;
    run.slot = base[i].slot;
    run.first_valid = (uint32_t)base[i].pkt;
    run.n_valid = (uint32_t)p.src.size();
    run.counts = std::move(p.counts);
    run.samples = p.samples;
    run.out_base = base[i].out;
    run.status = p.status;
    run.stop_packet = p.stop_packet;
    b->payload_bytes += p.payload_bytes;
    b->runs.push_back(std::move(run));
  }
  b->uploaded = false;
  return VPZ_OK;
}

int batch_add_run(vpz_batch* b, vpz_setup* s, const uint8_t* bytes, const uint32_t* offsets, uint32_t n_pkts,
                  const int32_t* trim) {
  vpz_ctx* ctx = b->ctx;
  if (b->synthetic || s->synthetic) {
    ctx->last_error = "packet runs cannot be added to a synthetic batch";
    return VPZ_E_INVALID_OP;
  }
  std::vector<PktSrc> src(n_pkts);
  for (uint32_t i = 0; i < n_pkts; i++) src[i] = PktSrc{bytes + offsets[i], offsets[i + 1] - offsets[i]};
  RunPlan plan;
  int rc = plan_run(s, src.data(), n_pkts, trim, &plan, &ctx->last_error);
  if (rc) return rc;
  RunPlan* pp = &plan;
  int first = 0;
  rc = batch_commit(b, &pp, 1, nullptr, &first);
  return rc ? rc : first;
}

int batch_upload(vpz_batch* b) {
  vpz_ctx* ctx = b->ctx;
  std::string& err = ctx->last_error;
  dev::Stream* st = ctx->stream;
  const size_t np = b->pkts_ola.n;
  int rc;
  if (!b->synthetic) {
    if (!b->d_bytes.reserve((b->gather_images ? b->gather_bytes : b->bytes.n) + 16, err) || !b->d_pkts_in.reserve(np * sizeof(VpzPktIn), err)) return VPZ_E_CUDA;
    if (b->gather_images) {   // corpus call: K7 gathers the packet bytes from the corpus's device images
      if (!b->d_pieces.reserve(b->pieces.n * sizeof(VpzGatherPiece), err)) return VPZ_E_CUDA;
      if ((rc = dev::h2d(b->d_pieces.p, b->pieces.p, b->pieces.n * sizeof(VpzGatherPiece), st, err))) return rc;
      K7Params kp;
      kp.images = b->gather_images;
      kp.bytes = static_cast<uint8_t*>(b->d_bytes.p);
      kp.pieces = static_cast<const VpzGatherPiece*>(b->d_pieces.p);
      kp.n_pieces = (uint32_t)b->pieces.n;
      if ((rc = dev::launch_k7(kp, st, err))) return rc;
      ctx->kernel_launches++;
    } else if ((rc = dev::h2d(b->d_bytes.p, b->bytes.p, b->bytes.n, st, err))) {
      return rc;
    }
    if ((rc = dev::h2d(b->d_pkts_in.p, b->pkts_in.p, np * sizeof(VpzPktIn), st, err))) return rc;
    if (!b->d_res.reserve(np * sizeof(VpzPktRes), err)) return VPZ_E_CUDA;
    if (!b->d_spec.reserve(b->spec_floats * 4, err)) return VPZ_E_CUDA;
    if (!b->d_rec.reserve(b->rec_words * 4 + 16, err) || !b->d_ent.reserve(b->ent_total * 2 + 16, err) ||
        !b->d_order.reserve(np * 4 + 16, err))
      return VPZ_E_CUDA;
    // K1a order: packets grouped by (setup, block size) and sorted by byte length, longest first,
    // inside a group (two stable counting sorts).  The 32 lanes of a warp then walk the same floor /
    // residue configuration with packets of like size (convergent control flow), the warps resident
    // on an SM share one setup's Huffman tables in L1, and the long packets do not form the tail.
    if (!b->order.reserve(2 * np + 2)) return VPZ_E_NOMEM;
    const double ts0 = trace_now();
    {
      // sort_key = (setup slot * 2 + short block) << 13 | (4096 - min(byte_len / 4, 4096)); it was written by
      // the threads that filled the batch, so the sort reads 4 bytes per packet.  The kernel class of the
      // setup (0 gather, 1 general K1b, 2 full K1a + general K1b) goes on top: every class is one contiguous
      // slice of the order array and gets its own launches.
      const size_t nslots = b->slots.size();
      std::vector<uint32_t> cls_of(nslots);
      for (size_t i = 0; i < nslots; i++) cls_of[i] = (uint32_t)k1_class(ctx, b->slots[i]);
      const size_t ngroups = 3 * 2 * nslots;
      const uint32_t* key = b->sort_key.data();
      auto group_of = [&](size_t i) { return (size_t)cls_of[key[i] >> 14] * 2 * nslots + (key[i] >> 13); };
      b->n_class[0] = b->n_class[1] = b->n_class[2] = 0;
      for (size_t i = 0; i < np; i++) b->n_class[cls_of[key[i] >> 14]]++;
      if (ngroups * 4097 <= ((size_t)1 << 20)) {
        std::vector<uint32_t> bucket(ngroups * 4097 + 2, 0);
        auto k1 = [&](size_t i) { return group_of(i) * 4097 + (key[i] & 8191u); };
        for (size_t i = 0; i < np; i++) bucket[k1(i) + 1]++;
        for (size_t k = 1; k < bucket.size(); k++) bucket[k] += bucket[k - 1];
        for (size_t i = 0; i < np; i++) b->order.p[bucket[k1(i)]++] = (uint32_t)i;
      } else {   // many setups: two stable passes
        uint32_t* tmp = b->order.p + np + 1;
        std::vector<uint32_t> bucket(4098, 0);
        for (size_t i = 0; i < np; i++) bucket[(key[i] & 8191u) + 1]++;
        for (size_t k = 1; k < bucket.size(); k++) bucket[k] += bucket[k - 1];
        for (size_t i = 0; i < np; i++) tmp[bucket[key[i] & 8191u]++] = (uint32_t)i;
        std::vector<uint32_t> gb(ngroups + 2, 0);
        for (size_t i = 0; i < np; i++) gb[group_of(i) + 1]++;
        for (size_t k = 1; k < gb.size(); k++) gb[k] += gb[k - 1];
        for (size_t i = 0; i < np; i++) b->order.p[gb[group_of(tmp[i])]++] = tmp[i];
      }
      b->order.n = np;
    }
    g_trace_ms[0] += trace_now() - ts0;
    if ((rc = dev::h2d(b->d_order.p, b->order.p, np * 4, st, err))) return rc;
  }
  if (!b->d_pkts_ola.reserve(np * sizeof(VpzPktOla), err) || !b->d_items.reserve(b->items.n * sizeof(VpzOlaItem), err) ||
      !b->d_pcm.reserve(b->total_floats * 4, err) || !b->d_clip.reserve(np * 4, err) ||
      !b->d_setups.reserve(b->slots.size() * sizeof(void*), err))
    return VPZ_E_CUDA;
  if ((rc = dev::h2d(b->d_pkts_ola.p, b->pkts_ola.p, np * sizeof(VpzPktOla), st, err))) return rc;
  {
    // K3 work items: the ones of 256 / 2048 mono / stereo setups first (fast kernel), the rest behind them
    if (!b->items_sorted.reserve(b->items.n + 1)) return VPZ_E_NOMEM;
    std::vector<uint8_t> fast_slot(b->slots.size());
    for (size_t i = 0; i < b->slots.size(); i++) fast_slot[i] = k3_fast(ctx, b->slots[i]) ? 1 : 0;
    size_t nf = 0;
    for (size_t i = 0; i < b->items.n; i++) nf += fast_slot[b->items.p[i].setup_slot];
    size_t a = 0, g = nf;
    for (size_t i = 0; i < b->items.n; i++) {
      const VpzOlaItem& it = b->items.p[i];
      b->items_sorted.p[fast_slot[it.setup_slot] ? a++ : g++] = it;
    }
    b->items_sorted.n = b->items.n;
    b->n_items_fast = (uint32_t)nf;
  }
  if ((rc = dev::h2d(b->d_items.p, b->items_sorted.p, b->items.n * sizeof(VpzOlaItem), st, err))) return rc;
  if (!b->h_setups.reserve(b->slots.size() + 1)) return VPZ_E_NOMEM;
  b->h_setups.n = 0;
  for (vpz_setup* s : b->slots) b->h_setups.p[b->h_setups.n++] = s->d_blob;
  if ((rc = dev::h2d(b->d_setups.p, b->h_setups.p, b->h_setups.n * sizeof(void*), st, err))) return rc;
  // no host sync: every source buffer is pinned memory owned by the batch and stays untouched until
  // the next reset, which the caller orders after the stream work (vpz_batch_sync / events)
  b->uploaded = true;
  b->decoded = false;
  return VPZ_OK;
}

int batch_decode(vpz_batch* b, int clip, int out16) {
  vpz_ctx* ctx = b->ctx;
  std::string& err = ctx->last_error;
  dev::Stream* st = ctx->stream;
  if (!b->uploaded) {
    const double tu0 = trace_now();
    int rc = batch_upload(b);
    g_trace_ms[1] += trace_now() - tu0;
    if (rc) return rc;
  }
  const double tl0 = trace_now();
  struct TraceLaunch {
    double t0;
    ~TraceLaunch() { g_trace_ms[2] += trace_now() - t0; }
  } trace_launch{tl0};
  const size_t np = b->pkts_ola.n;
  int rc;
  b->launches = 0;
  dev::event_record(ctx->ev[0], st);
  // one zeroed work-stealing word per launch of this pass: K1a simple 0 / full 1, K1b gather 2 / general 3,
  // K3 fast 4 / generic 5
  if ((rc = dev::fill(ctx->d_counter, 0, 32, st, err))) return rc;
  uint32_t k1w = 0, k1g = 0, k3f = 0, k1seg = 0;
  int gen_channels = 1;
  for (vpz_setup* s : b->slots) {
    if (k1_class(ctx, s) == 0) {
      k1g = std::max(k1g, s->k1g_words);      // urec + floor bytes of the largest setup ...
      k1seg = std::max(k1seg, s->k1g_seg_stride);
    } else {
      k1w = std::max(k1w, s->k1_words_per_warp);
    }
    if (!k3_fast(ctx, s)) {
      k3f = std::max(k3f, s->k3_floats_per_ch);
      gen_channels = std::max(gen_channels, s->host.id.channels);
    }
  }
  if (!b->synthetic && np) {
    K1Params p;
    memset(&p, 0, sizeof(p));
    p.bytes = static_cast<const uint32_t*>(b->d_bytes.p);
    p.pkts = static_cast<const VpzPktIn*>(b->d_pkts_in.p);
    p.res = static_cast<VpzPktRes*>(b->d_res.p);
    p.setups = static_cast<const uint32_t* const*>(b->d_setups.p);
    p.spec = static_cast<float*>(b->d_spec.p);
    p.rec = static_cast<uint32_t*>(b->d_rec.p);
    p.ent = static_cast<uint16_t*>(b->d_ent.p);
    p.dbg = b->dbg;
    p.k1a_smem = ctx->k1a_smem;
    const bool debug = b->dbg.hdr != nullptr;
    const uint32_t* order = static_cast<const uint32_t*>(b->d_order.p);
    const uint32_t n0 = b->n_class[0], n1 = b->n_class[1], n2 = b->n_class[2];
    // K1a: one lane per packet, 4 warps per CTA; the simple variant for classes 0 and 1, the full one for 2
    for (int full = 0; full < 2; full++) {
      const uint32_t cnt = full ? n2 : n0 + n1;
      if (!cnt) continue;
      p.order = order + (full ? n0 + n1 : 0);
      p.n_pkts = cnt;
      p.counter = ctx->d_counter + full;
      const size_t a_blocks = std::min<size_t>(((size_t)cnt + 127) / 128, (size_t)16 * dev::sm_count());
      if ((rc = dev::launch_k1a(p, debug, full != 0, (int)std::max<size_t>(1, a_blocks), st, err))) return rc;
      b->launches++;
      ctx->kernel_launches++;
    }
    dev::event_record(ctx->ev[1], st);
    // K1b: persistent CTAs of 4 warps fed by a counter; gather path = one warp per packet (shared
    // memory per warp), general path = one CTA per packet
    const int warps = 4;
    for (int general = 0; general < 2; general++) {
      const uint32_t cnt = general ? n1 + n2 : n0;
      if (!cnt) continue;
      p.order = order + (general ? n0 : 0);
      p.n_pkts = cnt;
      p.counter = ctx->d_counter + 2 + general;
      p.gather_ok = general ? 0 : 1;
      // ... + two channels of segment tables at the batch-wide stride (the kernel places them behind the
      // setup's own urec / floor bytes, so every part is sized by its own maximum)
      p.smem_words_per_warp = general ? k1w : (uint32_t)((k1g + 2 * (size_t)k1seg + 8 + 31) & ~(size_t)31);
      p.seg_stride = k1seg;
      const size_t smem_block = (size_t)p.smem_words_per_warp * 4 * (general ? 1 : warps) + (general ? 0 : 1024);   // + the dB table
      const size_t per_sm = std::max<size_t>(1, std::min<size_t>(16, (227 * 1024) / (smem_block + 1024)));
      const size_t blocks = std::min<size_t>(general ? cnt : ((size_t)cnt + warps - 1) / warps, per_sm * (size_t)dev::sm_count());
      if ((rc = dev::launch_k1b(p, debug, (int)std::max<size_t>(1, blocks), warps, st, err))) return rc;
      b->launches++;
      ctx->kernel_launches++;
    }
  } else {
    dev::event_record(ctx->ev[1], st);
  }
  dev::event_record(ctx->ev[2], st);
  if (b->items.n) {
    if ((rc = dev::fill(b->d_clip.p, 0xff, np * 4, st, err))) return rc;
    K3Params p;
    memset(&p, 0, sizeof(p));
    p.spec = static_cast<const float*>(b->d_spec.p);
    p.pkts = static_cast<const VpzPktOla*>(b->d_pkts_ola.p);
    p.res = b->synthetic ? nullptr : static_cast<const VpzPktRes*>(b->d_res.p);
    p.setups = static_cast<const uint32_t* const*>(b->d_setups.p);
    p.pcm = static_cast<float*>(b->d_pcm.p);
    p.clip_first = static_cast<uint32_t*>(b->d_clip.p);
    p.clip = clip ? 1 : 0;
    p.dbg_imdct = b->dbg_imdct;
    p.out16 = out16 ? 1 : 0;
    const VpzOlaItem* items = static_cast<const VpzOlaItem*>(b->d_items.p);
    if (b->n_items_fast) {
      p.items = items;
      p.n_items = b->n_items_fast;
      p.counter = ctx->d_counter + 4;
      if ((rc = dev::launch_k3_streams(p, st, err))) return rc;
      b->launches++;
      ctx->kernel_launches++;
    }
    if (b->items.n > b->n_items_fast) {
      p.items = items + b->n_items_fast;
      p.n_items = (uint32_t)(b->items.n - b->n_items_fast);
      p.counter = ctx->d_counter + 5;
      const int ncb = std::min(2, gen_channels);
      // descriptors (K3_DESC_FLOATS) + per channel slot the Stockham buffers and the three D half-slots
      const size_t k3_smem = ((size_t)ncb * k3f + 384) * 4;
      if ((rc = dev::launch_k3(p, ncb, k3_smem, st, err))) return rc;
      b->launches++;
      ctx->kernel_launches++;
    }
  }
  dev::event_record(ctx->ev[3], st);
  b->decoded = true;
  b->clip_fetched = false;
  return VPZ_OK;
}

int batch_fetch_clip(vpz_batch* b) {
  if (b->clip_fetched) return VPZ_OK;
  vpz_ctx* ctx = b->ctx;
  const size_t np = b->pkts_ola.n;
  if (!b->h_clip.reserve(np + 1)) return VPZ_E_NOMEM;
  b->h_clip.n = np;
  int rc = dev::d2h(b->h_clip.p, b->d_clip.p, np * 4, ctx->stream, ctx->last_error);
  if (rc) return rc;
  if ((rc = dev::stream_sync(ctx->stream, ctx->last_error))) return rc;
  b->clip_fetched = true;
  return VPZ_OK;
}

}  // namespace vpz
