// reader.cpp -- the IVorbisReader / IStreamDecoder side of the C ABI (include/vpz.h, "reader" and
// "bulk" layers).
//
// The reference decodes one packet per Read call on the CPU (StreamDecoder.Read,
// StreamDecoder.cs:418-498).  Here a stream is decoded AHEAD in windows of `lookahead` packets: the
// host walks the packet provider, replays the reference's position / end-of-stream bookkeeping on
// the packet headers alone (it never needs PCM values), submits the window to the GPU batch layer
// as one run and parks the interleaved PCM in pinned host memory.  Read() then hands that PCM out
// with exactly the reference's call-by-call behaviour: at most one packet per call, same sample
// counts, same SamplePosition / IsEndOfStream / HasClipped transitions, same error points.
//
// Reference behaviour followed (file:line):
//   VorbisReader.Initialize / ProcessNewStream / SwitchStreams / ReadSamples   VorbisReader.cs:56-85,191-253
//   StreamDecoder.ProcessHeaderPackets / LoadComments                          StreamDecoder.cs:125-260
//   StreamDecoder.Read / ReadNextPacket / DecodeNextPacket / ResetDecoder      StreamDecoder.cs:357-369,418-498,640-762
//   StreamDecoder.SeekTo / GetPacketGranuleCount                               StreamDecoder.cs:817-913
//   StoreInterleaved / StoreContiguous / Utils.ClipValue                       StreamDecoder.cs:515-638, Utils.cs:44-58
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <deque>
#include <memory>
#include <new>
#include <numeric>
#include <thread>
#include <unordered_map>

#include "../../include/vpz.h"
#include "bitreader.h"
#include "engine.h"
#include "ogg.h"

using namespace vpz;

namespace {

enum {  // EndOfStreamFlags.cs
  EOS_NONE = 0,
  EOS_INVALID_PACKET = 1,
  EOS_PACKET_FLAG = 2,
  EOS_INVALID_PREROLL = 4
};

struct Entry {            // one packet handed out by the provider, already planned / decoded
  bool ok = false;        // decoded (DecodeNextPacket returned a buffer)
  bool is_resync = false;
  int eos_flags = 0;
  int err = 0;            // error the reference raises at this packet (or VPZ_E_REF_FAULT)
  int count = 0;          // samples this packet makes available (RightStart - LeftStart, trimmed)
  int tail = 0;           // RightEnd - RightStart (trimmed): overlap length for the next packet
  int64_t granule = -1;
  size_t pcm_off = 0;     // float offset of its samples in the PCM cache
  size_t drain_off = 0;   // float offset of the raw right half (only for a failed end-of-stream packet)
};

// A planned window: entries in provider order plus the packets the GPU has to decode.
struct Window {
  std::vector<Entry> entries;
  std::vector<PktSrc> src;        // submitted packets: views into the container image or `arena`
  std::vector<int32_t> trims;
  std::vector<int> entry_of;      // submitted packet -> entry index (-1: carried-over seed packet)
  std::vector<std::vector<uint8_t>> arena;  // packets assembled across pages (moving an inner vector keeps its buffer: the views stay valid)
  std::vector<std::vector<OggSpan>> arena_spans;   // per arena packet: its bytes on each page of the image (K7's pieces)
  // drain of the last decoded packet's raw right half (see resolve_drain)
  bool drain = false, drain_extra_run = false;
  int drain_tail = 0, drain_entry = -1;
  // filled by plan_submit
  RunPlan plan, drain_plan;
  bool has_plan = false, has_drain_plan = false;
  std::vector<PktSrc> drain_src;
  int32_t drain_trims[2] = {0, 0};
  void add_packet(OggPacket* pk, int32_t trim, int entry) {
    if (!pk->owned.empty()) {
      arena.push_back(std::move(pk->owned));
      arena_spans.push_back(std::move(pk->spans));
      src.push_back(PktSrc{arena.back().data(), (uint32_t)arena.back().size()});
    } else {
      src.push_back(PktSrc{pk->ptr, pk->len});
    }
    trims.push_back(trim);
    entry_of.push_back(entry);
  }
};

}  // namespace

// One logical Vorbis stream of the container = one IStreamDecoder.
struct StreamDec {
  vpz_ctx* ctx = nullptr;
  LogicalStream* ls = nullptr;
  vpz_setup* setup = nullptr;
  std::vector<uint8_t> hdr[3];
  uint64_t setup_hash = 0;
  std::string vendor;
  std::vector<std::string> comments;
  // ---- reference decoder state, consumption side (StreamDecoder.cs:40-49) ----
  bool have_prev = false;        // _prevPacketBuf != null
  int prev_avail = 0;            // _prevPacketEnd - _prevPacketStart
  int prev_tail = 0;             // _prevPacketStop - _prevPacketEnd
  int eos_found = EOS_NONE;
  bool has_position = false;
  int64_t current_position = 0;
  bool has_clipped = false;
  bool clip = true;
  int fault = 0;
  // ---- decode-ahead state ----
  std::vector<Entry> q;
  size_t qh = 0;
  size_t pcm_cur = 0;            // float offset of the next unread sample of the current packet
  HostBuf<float> pcm;            // pinned PCM cache of the current window
  const float* pcm_view = nullptr;  // bulk random access: the window's PCM lives in the batch staging instead
  bool planned_only = false;     // bulk random access: the window was planned and decoded by the caller
  // bulk random access: Read does not copy; it records WHICH floats it would copy (K4 moves them on the device)
  std::vector<VpzCopySeg>* seg_sink = nullptr;
  uint64_t seg_dst = 0;          // float offset of buffer[0] in the group's output
  vpz_batch* batch = nullptr;
  int lookahead = 256;
  std::vector<uint8_t> carry;    // last decoded packet: re-submitted as the seed of the next window
  int32_t carry_trim = 0;
  // SeekTo reads its two packets (pre-roll, target) BEFORE it updates _currentPosition
  // (StreamDecoder.cs:851-879): the planner must see the stale position for those two and the
  // new one afterwards.
  int seek_left = 0;             // packets SeekTo still has to consume
  int64_t seek_pos = 0;          // position the provider reported for the target packet
  // packet table for vpz_reader_audio_packet
  std::vector<OggPacket> table;
  bool table_built = false;

  ~StreamDec() {
    if (batch) vpz_batch_destroy(batch);
    if (setup) setup_release(setup);
  }

  int channels() const { return setup->host.id.channels; }

  // IPacketGranuleCountProvider.GetPacketGranuleCount (StreamDecoder.cs:882-913)
  int granule_count(const OggPacket& pk) const {
    if (pk.is_resync) return 0;
    PacketGeom g = setup->host.packet_geometry(pk.ptr, pk.len);
    if (!g.valid) return 0;
    return g.right_start - g.left_start;
  }

  void reset_decoder() {  // StreamDecoder.ResetDecoder (StreamDecoder.cs:357-369)
    have_prev = false;
    prev_avail = prev_tail = 0;
    eos_found = EOS_NONE;
    has_clipped = false;
    has_position = false;
    q.clear();
    qh = 0;
    carry.clear();
    carry_trim = 0;
  }
};

namespace {

// StreamDecoder.LoadComments (StreamDecoder.cs:242-260)
int parse_comments(StreamDec* d, const std::vector<uint8_t>& pk) {
  static const uint8_t sig[7] = {0x03, 'v', 'o', 'r', 'b', 'i', 's'};
  if (pk.size() < 7 || memcmp(pk.data(), sig, 7) != 0) return VPZ_E_INVALID_DATA;
  BitReader br(pk.data(), pk.size());
  br.skip(56);
  auto read_string = [&](std::string* out) {
    uint32_t n = br.read(32);
    if ((int64_t)n * 8 > br.remaining()) return false;
    out->resize(n);
    for (uint32_t i = 0; i < n; i++) (*out)[i] = (char)br.read(8);
    return true;
  };
  if (!read_string(&d->vendor)) return VPZ_E_INVALID_DATA;
  uint32_t n = br.read(32);
  if ((int64_t)n * 32 > br.remaining()) return VPZ_E_INVALID_DATA;
  d->comments.resize(n);
  for (uint32_t i = 0; i < n; i++)
    if (!read_string(&d->comments[i])) return VPZ_E_INVALID_DATA;
  return VPZ_OK;
}

// StreamDecoder.Initialize -> ProcessHeaderPackets (StreamDecoder.cs:71-165), in two steps so the
// bulk path can run the per-stream part on worker threads:
//   stream_prepare : header packets, id / comment parse, content hash        (no shared state)
//   stream_attach  : setup cache lookup or table build + upload              (touches the context)
int stream_prepare(StreamDec* d, LogicalStream* ls, std::string* err) {
  d->ls = ls;
  for (int i = 0; i < 3; i++) {
    OggPacket pk;
    ls->next_packet(&pk);
    if (!pk.valid) {
      *err = i == 0 ? "First packet is not valid." : "Could not find Vorbis data to decode.";
      return VPZ_E_INVALID_DATA;
    }
    d->hdr[i].assign(pk.ptr, pk.ptr + pk.len);
  }
  IdHeader id;
  int rc = parse_id_header(d->hdr[0].data(), d->hdr[0].size(), &id);
  if (!rc) rc = parse_comments(d, d->hdr[1]);
  if (rc) {
    *err = "Could not find Vorbis data to decode.";
    return rc;
  }
  d->setup_hash = fnv1a64(d->hdr[2].data(), d->hdr[2].size(), fnv1a64(d->hdr[0].data(), d->hdr[0].size()));
  return VPZ_OK;
}

int stream_attach(StreamDec* d, vpz_ctx* ctx) {
  d->ctx = ctx;
  int rc = setup_create_hashed(ctx, d->setup_hash, d->hdr[0].data(), d->hdr[0].size(), d->hdr[2].data(),
                               d->hdr[2].size(), &d->setup);
  if (rc) return rc;
  d->ls->granule_count = [d](const OggPacket& pk) { return d->granule_count(pk); };
  d->current_position = 0;
  d->reset_decoder();
  d->has_position = true;
  return VPZ_OK;
}

int stream_init(StreamDec* d, vpz_ctx* ctx, LogicalStream* ls) {
  int rc = stream_prepare(d, ls, &ctx->last_error);
  return rc ? rc : stream_attach(d, ctx);
}

// Walks the provider for up to `max_packets` packets and replays ReadNextPacket's bookkeeping
// (StreamDecoder.cs:640-694) on the packet headers: which packets decode, the end-of-stream trim of
// RightStart, how many samples each makes available.  Nothing here depends on PCM values, which
// is what lets the GPU decode the whole window in one pass afterwards.
// need > 0: stop once the packets from SeekTo's target packet onwards make `need` samples available.
void plan_window(StreamDec* d, int max_packets, Window* w, int64_t need = 0) {
  const Setup& st = d->setup->host;
  bool have_prev = d->have_prev;
  int prev_tail = d->prev_tail;
  int64_t pos = d->current_position;
  bool has_pos = d->has_position;
  int seek_left = d->seek_left;
  int64_t produced = 0;
  if (need > 0) {   // a short excerpt: a handful of packets, one allocation per array
    w->entries.reserve(12);
    w->src.reserve(12);
    w->trims.reserve(12);
    w->entry_of.reserve(12);
  }
  if (have_prev && !d->carry.empty()) {
    w->src.push_back(PktSrc{d->carry.data(), (uint32_t)d->carry.size()});
    w->trims.push_back(d->carry_trim);
    w->entry_of.push_back(-1);
  }
  for (int n = 0; max_packets <= 0 || n < max_packets; n++) {
    OggPacket pk;
    d->ls->next_packet(&pk);
    Entry e;
    if (!pk.valid) {  // StreamDecoder.cs:703-711
      e.eos_flags = EOS_INVALID_PACKET;
      w->entries.push_back(e);
      break;
    }
    e.eos_flags = pk.is_eos ? EOS_PACKET_FLAG : EOS_NONE;
    e.is_resync = pk.is_resync;
    if (pk.is_resync) has_pos = false;
    PacketGeom g = st.packet_geometry(pk.ptr, pk.len);
    if (g.bad_mode) {  // the exception leaves DecodeNextPacket before _eosFound is updated
      e.eos_flags = EOS_NONE;
      e.err = VPZ_E_INVALID_DATA;
      w->entries.push_back(e);
      continue;
    }
    if (!g.valid) {
      w->entries.push_back(e);
      if (e.eos_flags || seek_left > 0) break;  // a failed packet ends SeekTo early
      continue;
    }
    const int L = prev_tail;
    int rs = g.right_start;
    int32_t trim = 0;
    if (pk.granule != -1 && e.eos_flags != EOS_NONE) {  // StreamDecoder.cs:658-666
      int diff = (int)(pos + L - pk.granule);
      if (diff > 0) {
        trim = diff;
        rs = std::max(rs - diff, 0);
      }
    }
    if (have_prev) {
      const int slope_len = (g.left_use_size1 ? st.id.size1 : st.id.size0) / 2;
      if (L > slope_len || L < 0 || g.left_start + L > st.id.size1 || rs < g.left_start) {
        e.err = VPZ_E_REF_FAULT;  // OverlapBuffers would throw (SURVEY quirk Q4)
        w->entries.push_back(e);
        break;
      }
    }
    e.ok = true;
    e.count = have_prev ? rs - g.left_start : 0;
    e.tail = g.right_end - rs;
    e.granule = pk.granule;
    w->add_packet(&pk, trim, (int)w->entries.size());
    w->entries.push_back(e);
    have_prev = true;
    prev_tail = e.tail;
    if (seek_left <= 1) produced += e.count;
    if (seek_left > 0) {
      // inside SeekTo: no position pick-up; after the target packet the position becomes
      // samplePosition + (count - rollForward) = provider position + count
      if (--seek_left == 0) pos = d->seek_pos + e.count;
    } else {
      if (pk.granule != -1 && !has_pos) {  // StreamDecoder.cs:459-463
        has_pos = true;
        pos = pk.granule - e.count;
      }
      pos += e.count;
    }
    if (e.eos_flags) break;
    if (need > 0 && seek_left == 0 && produced >= need) break;
  }
}

// StreamDecoder.cs:451-455: when the end-of-stream packet itself fails to decode, Read drains the
// previous packet's raw (unwindowed) right half.  If that previous packet P belongs to this window
// it simply gets a negative trim, so it emits [LeftStart, RightEnd) in place.  If P is the seed
// carried over from the previous window (it emits nothing here), an extra run [P, P(trim = -tail)]
// makes the second copy emit the same range and the last `tail` samples are taken from it.
void resolve_drain(StreamDec* d, Window* w) {
  if (w->entries.empty() || w->entry_of.empty()) return;
  const Entry& last = w->entries.back();
  if (last.ok || last.err || !(last.eos_flags & EOS_PACKET_FLAG)) return;
  const size_t k = w->entry_of.size() - 1;
  const int ei = w->entry_of[k];
  const int tail = ei >= 0 ? w->entries[(size_t)ei].tail : d->prev_tail;
  if (tail <= 0) return;
  w->drain = true;
  w->drain_tail = tail;
  w->drain_entry = (int)w->entries.size() - 1;
  if (ei >= 0) {
    w->trims[k] = -tail;  // P is never an end-of-stream packet itself, so its trim was 0
  } else {
    w->drain_extra_run = true;
    w->drain_src = {w->src[k], w->src[k]};
    w->drain_trims[0] = 0;
    w->drain_trims[1] = -tail;
  }
}

// Plans the GPU runs of the window (pure per-stream work: safe on worker threads).
int plan_submit(StreamDec* d, Window* w, std::string* err) {
  bool emits = false;
  for (int e : w->entry_of) emits |= e >= 0;
  if (!w->src.empty() && emits) {
    int rc = plan_run(d->setup, w->src.data(), (uint32_t)w->src.size(), w->trims.data(), &w->plan, err);
    if (rc) return rc;
    w->has_plan = true;
  }
  if (w->drain_extra_run) {
    int rc = plan_run(d->setup, w->drain_src.data(), 2, w->drain_trims, &w->drain_plan, err);
    if (rc) return rc;
    w->has_drain_plan = true;
  }
  return VPZ_OK;
}

// After the runs are committed to a batch: turns per-run sample counts into offsets inside the
// buffer the PCM of the batch is (or will be) copied to.  `shift` is added to every offset.
int place_window(StreamDec* d, vpz_batch* b, Window* w, int run, int drain_run, size_t shift) {
  const int C = d->channels();
  if (run >= 0) {
    const Run& r = b->runs[(size_t)run];
    size_t off = (size_t)r.out_base + shift;
    for (size_t k = 0; k < w->entry_of.size(); k++) {
      const int ei = w->entry_of[k];
      const int cnt = r.counts[k];
      if (ei >= 0) {
        Entry& e = w->entries[(size_t)ei];
        if (r.status == VPZ_E_REF_FAULT && (int32_t)k >= r.stop_packet) {
          e.ok = false;
          e.err = VPZ_E_REF_FAULT;
          continue;
        }
        const bool drained = w->drain && !w->drain_extra_run && k + 1 == w->entry_of.size();
        if (cnt != e.count + (drained ? w->drain_tail : 0)) {
          d->ctx->last_error = "internal: window plan and batch plan disagree";
          return VPZ_E_INVALID_OP;
        }
        e.pcm_off = off;
        if (drained) w->entries[(size_t)w->drain_entry].drain_off = off + (size_t)e.count * C;
      }
      off += (size_t)cnt * C;
    }
  }
  if (drain_run >= 0) {
    const Run& r = b->runs[(size_t)drain_run];
    w->entries[(size_t)w->drain_entry].drain_off = (size_t)r.out_base + shift + (size_t)(r.samples - w->drain_tail) * C;
  }
  return VPZ_OK;
}

// Commits the planned runs of one window to batch b.
int commit_window(vpz_batch* b, Window* w, int* run, int* drain_run) {
  *run = *drain_run = -1;
  RunPlan* plans[2];
  size_t n = 0;
  if (w->has_plan) plans[n++] = &w->plan;
  if (w->has_drain_plan) plans[n++] = &w->drain_plan;
  int first = 0;
  int rc = batch_commit(b, plans, n, nullptr, &first);
  if (rc) return rc;
  if (w->has_plan) *run = first++;
  if (w->has_drain_plan) *drain_run = first;
  return VPZ_OK;
}

// Plans, decodes and caches the next window of the stream (the reader path: one stream, own batch).
int decode_ahead(StreamDec* d) {
  vpz_ctx* ctx = d->ctx;
  if (!d->batch) {
    int rc = vpz_batch_create(ctx, &d->batch);
    if (rc) return rc;
  }
  Window w;
  plan_window(d, d->lookahead, &w);
  resolve_drain(d, &w);
  int rc = plan_submit(d, &w, &ctx->last_error);
  if (rc) return rc;
  vpz_batch_reset(d->batch);
  int run, drain_run;
  if ((rc = commit_window(d->batch, &w, &run, &drain_run))) return rc;
  size_t total = (size_t)d->batch->total_floats;
  if (total) {
    if (!d->pcm.reserve(total)) return VPZ_E_NOMEM;
    // the reader clips while copying into the caller's buffer (partial reads need per-sample HasClipped)
    if ((rc = batch_decode(d->batch, 0))) return rc;
    if ((rc = vpz_batch_read_all(d->batch, d->pcm.p))) return rc;
  }
  if ((rc = place_window(d, d->batch, &w, run, drain_run, 0))) return rc;
  // remember the last decoded packet as the seed of the next window
  for (int k = (int)w.entry_of.size() - 1; k >= 0; k--) {
    if (w.entry_of[(size_t)k] < 0) break;  // only the seed itself was submitted
    if (w.entries[(size_t)w.entry_of[(size_t)k]].ok) {
      std::vector<uint8_t> next(w.src[(size_t)k].p, w.src[(size_t)k].p + w.src[(size_t)k].len);
      d->carry.swap(next);
      d->carry_trim = w.trims[(size_t)k];
      break;
    }
  }
  d->q = std::move(w.entries);
  d->qh = 0;
  return VPZ_OK;
}

// StreamDecoder.ReadNextPacket (StreamDecoder.cs:640-694), consumption side
bool read_next_packet(StreamDec* d, int64_t* sample_position, int* err) {
  *sample_position = -1;
  if (d->qh == d->q.size() && d->planned_only) {  // the caller planned exactly what it reads
    d->eos_found |= EOS_INVALID_PACKET;
    return false;
  }
  if (d->qh == d->q.size()) {
    int rc = decode_ahead(d);
    if (rc) {
      *err = rc;
      return false;
    }
    if (d->q.empty()) {
      d->eos_found |= EOS_INVALID_PACKET;
      return false;
    }
  }
  const Entry& e = d->q[d->qh++];
  if (d->seek_left > 0) d->seek_left--;
  if (e.err) {
    if (e.is_resync) d->has_position = false;
    *err = e.err;
    return false;
  }
  d->eos_found |= e.eos_flags;
  if (e.is_resync) d->has_position = false;
  if (!e.ok) {
    if ((e.eos_flags & EOS_PACKET_FLAG) && d->have_prev) {
      // caller applies _prevPacketEnd = _prevPacketStop; point at the raw right half
      d->pcm_cur = e.drain_off;
    }
    return false;
  }
  *sample_position = e.granule;
  d->prev_avail = d->have_prev ? e.count : 0;
  d->prev_tail = e.tail;
  d->pcm_cur = e.pcm_off;
  d->have_prev = true;
  return true;
}

inline float clip_value(float v, bool* clipped) {  // Utils.ClipValue (Utils.cs:44-58)
  if (v > 0.99999994f) {
    *clipped = true;
    return 0.99999994f;
  }
  if (v < -0.99999994f) {
    *clipped = true;
    return -0.99999994f;
  }
  return v;
}

// StreamDecoder.Read (StreamDecoder.cs:418-498)
int stream_read(StreamDec* d, float* buffer, int nfloats, int samples_to_read, int channel_stride, bool interleave) {
  const int C = d->channels();
  if (d->fault) return d->fault;
  if (nfloats < 0 || nfloats % C != 0) return VPZ_E_ARGUMENT;
  if ((int64_t)nfloats < (int64_t)samples_to_read * C) return VPZ_E_ARGUMENT;
  if (!buffer && nfloats && !d->seg_sink) return VPZ_E_ARGUMENT;
  int idx = 0;
  while (idx == 0) {
    if (d->prev_avail == 0) {
      if (d->eos_found != EOS_NONE) {
        d->have_prev = false;
        break;
      }
      int64_t sp = -1;
      int err = 0;
      if (!read_next_packet(d, &sp, &err)) {
        if (err) {
          if (err == VPZ_E_REF_FAULT) {  // the reference throws here; this path ends the stream instead
            d->fault = err;
            d->eos_found |= EOS_INVALID_PACKET;
            d->have_prev = false;
            d->prev_avail = d->prev_tail = 0;
          }
          return err;
        }
        if (d->eos_found & EOS_PACKET_FLAG) {  // StreamDecoder.cs:451-455
          d->prev_avail = d->prev_tail;
          d->prev_tail = 0;
        }
      }
      if (sp != -1 && !d->has_position) {
        d->has_position = true;
        d->current_position = sp - d->prev_avail - idx;
      }
    }
    int copy_len = std::min(samples_to_read - idx, d->prev_avail);
    if (copy_len <= 0) {
      if (samples_to_read - idx <= 0) break;  // the reference spins forever on a zero-length request
      if (d->prev_avail < 0) return VPZ_E_REF_FAULT;
      continue;
    }
    const float* src = (d->pcm_view ? d->pcm_view : d->pcm.p) + d->pcm_cur;
    bool clipped = false;
    if (d->seg_sink) {
      VpzCopySeg sg;
      sg.src = d->pcm_cur;
      sg.dst = d->seg_dst + (uint64_t)idx * C;
      sg.n = (uint32_t)copy_len * (uint32_t)C;
      sg.pad = 0;
      d->seg_sink->push_back(sg);
    } else if (interleave) {
      float* dst = buffer + (size_t)idx * C;
      const size_t n = (size_t)copy_len * C;
      if (d->clip) {
        for (size_t i = 0; i < n; i++) dst[i] = clip_value(src[i], &clipped);
      } else {
        memcpy(dst, src, n * sizeof(float));
      }
    } else {
      for (int ch = 0; ch < C; ch++) {
        float* dst = buffer + (size_t)ch * channel_stride + idx;
        if (d->clip) {
          for (int i = 0; i < copy_len; i++) dst[i] = clip_value(src[(size_t)i * C + ch], &clipped);
        } else {
          for (int i = 0; i < copy_len; i++) dst[i] = src[(size_t)i * C + ch];
        }
      }
    }
    d->has_clipped |= clipped;
    idx += copy_len;
    d->pcm_cur += (size_t)copy_len * C;
    d->prev_avail -= copy_len;
    d->current_position += copy_len;
  }
  return idx;
}

int64_t stream_total_samples(StreamDec* d, int* err) { return d->ls->total_granules(err); }

// StreamDecoder.SeekTo (StreamDecoder.cs:817-880) in two halves.  seek_begin: the packet provider
// repositions (pre-roll of one packet) and the decoder is reset; seek_finish: SeekTo consumes the
// pre-roll and the target packet and rolls forward inside the target.  Between the two the window that
// starts at the pre-roll packet gets planned and decoded -- by decode_ahead on the reader path, by the
// caller for a whole batch of excerpts on the bulk random-access path.
int seek_begin(StreamDec* d, int64_t sample_position, int64_t* pos_out) {
  int err = 0;
  // the provider cursor has run ahead of the consumer; SeekTo repositions it anyway
  int64_t pos = d->ls->seek_to(sample_position, 1, &err);
  if (err) return err;
  d->reset_decoder();
  d->fault = 0;
  d->has_position = true;
  d->seek_left = 2;
  d->seek_pos = pos;
  *pos_out = pos;
  return VPZ_OK;
}

int seek_finish(StreamDec* d, int64_t sample_position, int64_t pos) {
  int err = 0;
  int roll_forward = (int)(sample_position - pos);
  struct SeekDone {
    StreamDec* d;
    ~SeekDone() { d->seek_left = 0; }
  } seek_done{d};
  int64_t sp;
  if (!read_next_packet(d, &sp, &err)) {
    if (err) return err;
    d->eos_found |= EOS_INVALID_PREROLL;
    int64_t max_granule = stream_total_samples(d, &err);
    if (err) return err;
    if (sample_position > max_granule) return VPZ_E_SEEK_RANGE;
    d->prev_avail = 0;
    d->current_position = sample_position;
    return VPZ_OK;
  }
  if (!read_next_packet(d, &sp, &err)) {
    if (err == VPZ_E_REF_FAULT) d->fault = err;
    if (err) return err;
    d->reset_decoder();
    d->eos_found |= EOS_INVALID_PACKET;
    return VPZ_E_PREROLL;
  }
  d->prev_avail -= roll_forward;
  d->pcm_cur += (size_t)roll_forward * d->channels();
  d->current_position = sample_position;
  return VPZ_OK;
}

// StreamDecoder.SeekTo (StreamDecoder.cs:817-880)
int stream_seek(StreamDec* d, int64_t sample_position, int origin) {
  if (!d->ls->can_seek()) return VPZ_E_INVALID_OP;
  if (sample_position < 0) return VPZ_E_ARGUMENT;
  int err = 0;
  switch (origin) {
    case 0: break;
    case 1: sample_position = d->current_position - sample_position; break;
    case 2: {
      int64_t total = stream_total_samples(d, &err);
      if (err) return err;
      sample_position = total - sample_position;
      break;
    }
    default: return VPZ_E_ARGUMENT;
  }
  int64_t pos = 0;
  int rc = seek_begin(d, sample_position, &pos);
  return rc ? rc : seek_finish(d, sample_position, pos);
}

void build_table(StreamDec* d) {
  if (d->table_built) return;
  LogicalStream walker;  // a second cursor over the same pages; the decode cursor is left alone
  walker.serial = d->ls->serial;
  walker.pages = d->ls->pages;
  OggPacket pk;
  for (int i = 0; i < 3; i++) walker.next_packet(&pk);
  for (;;) {
    walker.next_packet(&pk);
    if (!pk.valid) break;
    d->table.push_back(std::move(pk));
  }
  d->table_built = true;
}

}  // namespace

struct vpz_reader {
  vpz_ctx* ctx = nullptr;
  std::vector<uint8_t> own;
  OggContainer cont;
  std::vector<StreamDec*> decs;   // Streams
  size_t next_logical = 0;        // next logical stream FindNextStream will look at
  int cur = 0;                    // StreamIndex
  ~vpz_reader() {
    for (StreamDec* d : decs) delete d;
  }
  StreamDec* dec() const { return decs[(size_t)cur]; }
};

namespace {
// ContainerReader.FindNextStream + VorbisReader.ProcessNewStream: 1 found, 0 none, <0 error
int find_next(vpz_reader* r) {
  if (r->next_logical >= r->cont.streams.size()) return 0;
  LogicalStream* ls = r->cont.streams[r->next_logical++];
  std::unique_ptr<StreamDec> d(new (std::nothrow) StreamDec);
  if (!d) return VPZ_E_NOMEM;
  int rc = stream_init(d.get(), r->ctx, ls);
  if (rc) return rc;
  r->decs.push_back(d.release());
  return 1;
}
}  // namespace

extern "C" {

int vpz_reader_open_memory(vpz_ctx* ctx, const uint8_t* data, size_t len, int copy, vpz_reader** out) {
  if (ctx) VPZ_USE(ctx);
  if (!ctx || !out || (!data && len)) return VPZ_E_ARGUMENT;
  *out = nullptr;
  vpz_reader* r = new (std::nothrow) vpz_reader;
  if (!r) return VPZ_E_NOMEM;
  r->ctx = ctx;
  if (copy) {
    r->own.assign(data, data + len);
    data = r->own.data();
  }
  // "gpu_scan" 2: the physical Ogg layer of single readers runs on the device too (the default keeps it on
  // the host there: one image is one warp of work, not worth a launch and two copies)
  int rc = VPZ_OK;
  bool scanned = false;
  if (ctx->gpu_scan >= 2) {
    ScanResult sr;
    rc = scan_pages(ctx, 1, &data, &len, nullptr, &sr);
    if (rc == VPZ_OK && !sr.out[0].overflow) {
      rc = r->cont.scan_from_records(data, len, sr.pages + sr.files[0].page_base, sr.out[0].n_pages,
                                     ((uint64_t)sr.out[0].waste_hi << 32) | sr.out[0].waste_lo, sr.out[0].crc_failures);
      scanned = true;
    }
  }
  if (rc == VPZ_OK && !scanned) rc = r->cont.scan(data, len);
  if (rc == VPZ_OK) {
    rc = find_next(r);
    if (rc == 0) rc = VPZ_E_INVALID_DATA;
    if (rc == 1) rc = VPZ_OK;
  }
  if (rc) {
    if (rc == VPZ_E_INVALID_DATA && ctx->last_error.empty())
      ctx->last_error = "Could not load the specified container.";  // VorbisReader.cs:63
    delete r;
    return rc;
  }
  *out = r;
  return VPZ_OK;
}

void vpz_reader_close(vpz_reader* r) {
  if (!r) return;
  VPZ_USE(r->ctx);
  delete r;
}

int vpz_reader_stream_count(const vpz_reader* r) { return r ? (int)r->decs.size() : VPZ_E_ARGUMENT; }
int vpz_reader_stream_index(const vpz_reader* r) { return r ? r->cur : VPZ_E_ARGUMENT; }

int vpz_reader_switch_stream(vpz_reader* r, int index) {  // VorbisReader.SwitchStreams
  if (!r) return VPZ_E_ARGUMENT;
  if (index < 0 || (size_t)index >= r->decs.size()) return VPZ_E_ARGUMENT;
  if (index == r->cur) return 0;
  StreamDec* nd = r->decs[(size_t)index];
  StreamDec* od = r->dec();
  nd->clip = od->clip;
  r->cur = index;
  return (nd->channels() != od->channels() || nd->setup->host.id.sample_rate != od->setup->host.id.sample_rate) ? 1 : 0;
}

int vpz_reader_find_next_stream(vpz_reader* r) {
  if (!r) return VPZ_E_ARGUMENT;
  VPZ_USE(r->ctx);
  return find_next(r);
}
int vpz_reader_can_seek(const vpz_reader* r) { return r ? (r->dec()->ls->can_seek() ? 1 : 0) : VPZ_E_ARGUMENT; }

int vpz_reader_channels(const vpz_reader* r) { return r ? r->dec()->channels() : VPZ_E_ARGUMENT; }
int vpz_reader_sample_rate(const vpz_reader* r) { return r ? r->dec()->setup->host.id.sample_rate : VPZ_E_ARGUMENT; }
int vpz_reader_bitrate(const vpz_reader* r, int which) {
  if (!r) return VPZ_E_ARGUMENT;
  const IdHeader& id = r->dec()->setup->host.id;
  return which == 0 ? id.br_upper : which == 1 ? id.br_nominal : id.br_lower;
}
int vpz_reader_stream_serial(const vpz_reader* r) { return r ? (int)r->dec()->ls->serial : VPZ_E_ARGUMENT; }

int64_t vpz_reader_total_samples(vpz_reader* r) {
  if (!r) return VPZ_E_ARGUMENT;
  int err = 0;
  int64_t n = stream_total_samples(r->dec(), &err);
  return err ? err : n;
}
int64_t vpz_reader_sample_position(const vpz_reader* r) { return r ? r->dec()->current_position : VPZ_E_ARGUMENT; }
int vpz_reader_is_end_of_stream(const vpz_reader* r) {  // StreamDecoder.cs:1001
  if (!r) return VPZ_E_ARGUMENT;
  const StreamDec* d = r->dec();
  return (d->eos_found != EOS_NONE && !d->have_prev) ? 1 : 0;
}
int vpz_reader_has_clipped(const vpz_reader* r) { return r ? (r->dec()->has_clipped ? 1 : 0) : VPZ_E_ARGUMENT; }
int vpz_reader_get_clip(const vpz_reader* r) { return r ? (r->dec()->clip ? 1 : 0) : VPZ_E_ARGUMENT; }
void vpz_reader_set_clip(vpz_reader* r, int clip) {
  if (r) r->dec()->clip = clip != 0;
}
int64_t vpz_reader_container_overhead_bits(const vpz_reader* r) {
  if (!r) return VPZ_E_ARGUMENT;
  int64_t n = 0;
  for (const LogicalStream* ls : r->cont.streams) n += ls->container_bits;
  return n;
}
int64_t vpz_reader_container_waste_bits(const vpz_reader* r) { return r ? r->cont.waste_bits : VPZ_E_ARGUMENT; }

const char* vpz_reader_vendor(const vpz_reader* r, int* len) {
  if (!r) return nullptr;
  if (len) *len = (int)r->dec()->vendor.size();
  return r->dec()->vendor.data();
}
int vpz_reader_comment_count(const vpz_reader* r) { return r ? (int)r->dec()->comments.size() : VPZ_E_ARGUMENT; }
const char* vpz_reader_comment(const vpz_reader* r, int i, int* len) {
  if (!r || i < 0 || (size_t)i >= r->dec()->comments.size()) return nullptr;
  if (len) *len = (int)r->dec()->comments[(size_t)i].size();
  return r->dec()->comments[(size_t)i].data();
}

int vpz_reader_read(vpz_reader* r, float* buf, int nfloats) {
  if (!r) return VPZ_E_ARGUMENT;
  VPZ_USE(r->ctx);
  StreamDec* d = r->dec();
  return stream_read(d, buf, nfloats, nfloats / d->channels(), 0, true);
}
int vpz_reader_read_planar(vpz_reader* r, float* buf, int nfloats, int samples_to_read, int channel_stride) {
  if (!r || samples_to_read < 0) return VPZ_E_ARGUMENT;
  VPZ_USE(r->ctx);
  return stream_read(r->dec(), buf, nfloats, samples_to_read, channel_stride, false);
}
int vpz_reader_seek(vpz_reader* r, int64_t sample_position, int origin) {
  if (!r) return VPZ_E_ARGUMENT;
  VPZ_USE(r->ctx);
  return stream_seek(r->dec(), sample_position, origin);
}
int vpz_reader_set_lookahead(vpz_reader* r, int packets) {
  if (!r || packets < 0) return VPZ_E_ARGUMENT;
  r->dec()->lookahead = packets;
  return VPZ_OK;
}

int vpz_reader_audio_packet_count(vpz_reader* r) {
  if (!r) return VPZ_E_ARGUMENT;
  build_table(r->dec());
  return (int)r->dec()->table.size();
}
int vpz_reader_audio_packet(vpz_reader* r, int i, const uint8_t** data, uint32_t* len, int64_t* granule,
                            int32_t* flags) {
  if (!r) return VPZ_E_ARGUMENT;
  StreamDec* d = r->dec();
  build_table(d);
  if (i < 0 || (size_t)i >= d->table.size()) return VPZ_E_ARGUMENT;
  const OggPacket& pk = d->table[(size_t)i];
  if (data) *data = pk.ptr;
  if (len) *len = pk.len;
  if (granule) *granule = pk.granule;
  if (flags) *flags = (pk.is_resync ? 1 : 0) | (pk.is_eos ? 2 : 0);
  return VPZ_OK;
}
const uint8_t* vpz_reader_header_packet(vpz_reader* r, int which, uint32_t* len) {
  if (!r || which < 0 || which > 2) return nullptr;
  if (len) *len = (uint32_t)r->dec()->hdr[which].size();
  return r->dec()->hdr[which].data();
}
vpz_setup* vpz_reader_setup(vpz_reader* r) { return r ? r->dec()->setup : nullptr; }

// ---- bulk: many whole files, pipelined in groups ---------------------------------------------------
// Host work (page scan + CRC, header lookup, packet walk, window plan, copy into pinned staging) runs
// on the worker pool group by group; while the GPU decodes group g (H2D, K1, K3 on the compute
// stream) and the copy stream moves the PCM of group g-1 to the caller's buffer, the host already
// plans group g+1.  Three batches rotate so no buffer is reused before its copies have finished.
namespace {
struct BulkJob {
  OggContainer cont;
  StreamDec dec;
  Window win;
  int rc = 0;
  std::string err;
};
}  // namespace

}  // extern "C"

// ---- device output (vpz_decode_files_device, vpz_decode_excerpts_device) --------------------------
// The bulk pipelines stay as they are; only the last step of a group differs: instead of a device->host copy of
// the group's PCM, K5 places tiles of the batch PCM into the caller's device buffer on the compute stream.
namespace {
struct DevOut {
  void* p = nullptr;       // the caller's device buffer (NULL: size query)
  int format = 0;          // VPZ_OUT_* bits
  void* stream = nullptr;  // the caller's cudaStream_t
  const vpz_out_conv* conv = nullptr;   // the *_conv calls: target rate and channels (K6)
  int64_t* offsets = nullptr;           // vpz_decode_files_device_conv: element offset of every file (may be NULL)
};

size_t tile_count(uint64_t samples) { return (size_t)((samples + VPZ_TILE_SAMPLES - 1) / VPZ_TILE_SAMPLES); }

// samples [first, first + n) of an item (element base `base`, `len` samples per channel, `ch` channels) from the
// batch PCM at float offset src (VPZ_TILE_ZERO: zeros), cut into tiles; returns the end of the written tiles
VpzPlaceTile* put_tiles(VpzPlaceTile* out, uint64_t src, uint64_t base, uint64_t len, uint64_t first, uint64_t n, uint32_t ch) {
  for (uint64_t s = 0; s < n; s += VPZ_TILE_SAMPLES) {
    VpzPlaceTile t;
    t.src = src == VPZ_TILE_ZERO ? src : src + s * ch;
    t.base = base;
    t.len = len;
    t.first = first + s;
    t.n = (uint32_t)std::min<uint64_t>(VPZ_TILE_SAMPLES, n - s);
    t.ch = ch;
    *out++ = t;
  }
  return out;
}
void append_tiles(std::vector<VpzPlaceTile>& v, uint64_t src, uint64_t base, uint64_t len, uint64_t first, uint64_t n, uint32_t ch) {
  const size_t at = v.size();
  v.resize(at + tile_count(n));
  put_tiles(v.data() + at, src, base, len, first, n, ch);
}

// Checks the destination and orders the context's stream behind the work already queued on the caller's stream
// (a tensor from a caching allocator may still be in use there); *ev is destroyed by device_output_end
int device_output_begin(vpz_ctx* ctx, const DevOut& o, dev::Event** ev) {
  if (o.format & ~(VPZ_OUT_S16 | VPZ_OUT_PLANAR)) {
    ctx->last_error = "unknown output format bits";
    return VPZ_E_ARGUMENT;
  }
  if (!o.p) return VPZ_OK;   // size query
  int rc = dev::check_device_ptr(o.p, ctx->device, ctx->last_error);
  if (rc) return rc;
  if (!ctx->place) {
    ctx->place = new (std::nothrow) PlaceBufs;
    if (!ctx->place) return VPZ_E_NOMEM;
  }
  *ev = dev::event_create();
  if (!*ev) {
    ctx->last_error = "cudaEventCreate failed";
    return VPZ_E_CUDA;
  }
  dev::event_record_external(*ev, o.stream);
  dev::stream_wait_event(ctx->stream, *ev);
  return VPZ_OK;
}
// Nothing of the call stays queued behind it: the destination is complete when the call returns
int64_t device_output_end(vpz_ctx* ctx, dev::Event* ev, int64_t rc) {
  if (!ev) return rc;
  std::string err;
  int r2 = dev::stream_sync(ctx->stream, err);
  dev::event_destroy(ev);
  if (r2 && rc >= 0) {
    ctx->last_error = err;
    return r2;
  }
  return rc;
}

// Uploads the tiles of pipeline slot `slot` and launches K5 on the context's stream.  Tiles [0, n_dst) go to the
// caller's buffer; the rest (vpz_decode_excerpts_device_conv) to the slot's scratch, as fp32 interleaved.
int place_tiles(vpz_ctx* ctx, int slot, const vpz_batch* b, const DevOut& o, int clip, size_t n_dst = SIZE_MAX) {
  PlaceBufs& pb = *ctx->place;
  const size_t n = pb.h_tiles[slot].n;
  if (!n) return VPZ_OK;
  if (!pb.d_tiles[slot].reserve(n * sizeof(VpzPlaceTile), ctx->last_error)) return VPZ_E_CUDA;
  int rc = dev::h2d(pb.d_tiles[slot].p, pb.h_tiles[slot].p, n * sizeof(VpzPlaceTile), ctx->stream, ctx->last_error);
  if (rc) return rc;
  n_dst = std::min(n_dst, n);
  K5Params kp;
  kp.pcm = static_cast<const float*>(b->d_pcm.p);
  kp.out = o.p;
  kp.tiles = static_cast<const VpzPlaceTile*>(pb.d_tiles[slot].p);
  kp.n_tiles = (uint32_t)n_dst;
  kp.planar = (o.format & VPZ_OUT_PLANAR) ? 1 : 0;
  kp.out16 = (o.format & VPZ_OUT_S16) ? 1 : 0;
  kp.clip = clip ? 1 : 0;
  rc = dev::launch_k5(kp, ctx->stream, ctx->last_error);
  if (!rc && n_dst) ctx->kernel_launches++;
  if (rc || n_dst == n) return rc;
  kp.out = pb.d_scratch[slot].p;
  kp.tiles += n_dst;
  kp.n_tiles = (uint32_t)(n - n_dst);
  kp.planar = 0;
  kp.out16 = 0;
  rc = dev::launch_k5(kp, ctx->stream, ctx->last_error);
  if (!rc) ctx->kernel_launches++;
  return rc;
}

// ---- conversion to one rate and channel layout (the *_conv calls, K6) ------------------------------------------
int conv_check(vpz_ctx* ctx, const vpz_out_conv* cv) {
  if (!cv || (cv->sample_rate != 0 && (cv->sample_rate < 1000 || cv->sample_rate > 384000)) || cv->channels < 0 ||
      cv->channels > 2) {
    ctx->last_error = cv ? "conversion: sample_rate must be 0 or 1000..384000, channels 0, 1 or 2" : "conversion: NULL";
    return VPZ_E_ARGUMENT;
  }
  return VPZ_OK;
}

int64_t floor_div(int64_t a, int64_t b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

// What K6 does to the items of one stream (rate fi, C channels)
struct ItemConv {
  bool on = false;                 // converted; otherwise K5 places the item unchanged
  const ConvFilter* f = nullptr;   // the rate pair's table once uploaded (NULL at equal rates and in a size query)
  bool filter = false;             // rates differ
  uint32_t o = 1, n = 1, width = 0;
  uint32_t C = 0, Cout = 0, mix = VPZ_MIX_KEEP;
  uint32_t m = 0;                  // output samples per tile
  uint32_t smem_floats = 0;        // shared memory of the largest tile
  int64_t out_len(int64_t src) const { return filter ? (src * n + o - 1) / o : src; }   // ceil(src fo / fi)
  // source window [k_lo, k_hi) of output samples [start, start + count)
  void window(int64_t start, int64_t count, int64_t* k_lo, int64_t* k_hi) const {
    if (!filter) {
      *k_lo = start;
      *k_hi = start + count;
      return;
    }
    *k_lo = std::max<int64_t>(0, floor_div(start * o, n) - width);
    *k_hi = std::max(*k_lo, floor_div((start + count - 1) * o, n) + width + 1);
  }
};

// The coefficient table of fi -> fo, made and uploaded on first use and kept in the context: tap-major, entry
// [i][p] weighs source frame k = floor(p o / n) - width + i, i < 2 width + 2, of output p (torchaudio.functional.resample's sinc_interp_hann,
// W = 6, rolloff 0.99, evaluated in float64)
int conv_filter(vpz_ctx* ctx, int fi, int fo, const ConvFilter** out) {
  PlaceBufs& pb = *ctx->place;
  for (const auto& f : pb.filters)
    if (f->fi == fi && f->fo == fo) {
      *out = f.get();
      return VPZ_OK;
    }
  std::unique_ptr<ConvFilter> f(new (std::nothrow) ConvFilter);
  if (!f) return VPZ_E_NOMEM;
  const uint32_t g = (uint32_t)std::gcd(fi, fo);
  f->fi = fi;
  f->fo = fo;
  f->o = (uint32_t)fi / g;
  f->n = (uint32_t)fo / g;
  const double W = 6.0, base = 0.99 * std::min(f->o, f->n), pi = 3.14159265358979323846;
  f->width = (uint32_t)std::ceil(W * f->o / base);
  const uint32_t taps = 2 * f->width + 2;
  f->host.resize((size_t)f->n * taps);
  for (uint32_t p = 0; p < f->n; p++) {
    const int64_t k0 = (int64_t)p * f->o / f->n - f->width;
    for (uint32_t i = 0; i < taps; i++) {
      double t = base * ((double)(k0 + i) / f->o - (double)p / f->n);
      t = std::min(W, std::max(-W, t));
      const double w = std::cos(t * pi / (2 * W));
      const double sinc = t == 0 ? 1.0 : std::sin(pi * t) / (pi * t);
      f->host[(size_t)i * f->n + p] = (float)(base / f->o * sinc * w * w);
    }
  }
  if (!f->dev.reserve(f->host.size() * 4, ctx->last_error)) return VPZ_E_CUDA;
  int rc = dev::h2d(f->dev.p, f->host.data(), f->host.size() * 4, ctx->stream, ctx->last_error);
  if (rc) return rc;
  *out = f.get();
  pb.filters.push_back(std::move(f));
  return VPZ_OK;
}

// Plans the items of a stream (rate fi, C channels); build: also fetch the table (the call writes samples)
int conv_plan(vpz_ctx* ctx, const vpz_out_conv& cv, int fi, int C, bool build, ItemConv* ic) {
  *ic = ItemConv();
  ic->C = (uint32_t)C;
  ic->Cout = cv.channels ? (uint32_t)cv.channels : (uint32_t)C;
  if (C > 2 && cv.channels == 2) {
    ctx->last_error = "conversion: channels = 2 from a stream of more than 2 channels";
    return VPZ_E_UNSUPPORTED;
  }
  const int fo = cv.sample_rate ? cv.sample_rate : fi;
  ic->mix = ic->Cout == ic->C ? VPZ_MIX_KEEP : ic->Cout == 1 ? VPZ_MIX_MEAN : VPZ_MIX_DUP;
  ic->filter = fo != fi;
  ic->on = ic->filter || ic->mix != VPZ_MIX_KEEP;
  if (!ic->on) return VPZ_OK;
  if (ic->filter) {
    if (fi <= 0) {
      ctx->last_error = "conversion: stream without a sample rate";
      return VPZ_E_UNSUPPORTED;
    }
    const uint32_t g = (uint32_t)std::gcd(fi, fo);
    ic->o = (uint32_t)fi / g;
    ic->n = (uint32_t)fo / g;
    ic->width = (uint32_t)std::ceil(6.0 * ic->o / (0.99 * std::min(ic->o, ic->n)));
    if ((uint64_t)ic->n * (2 * ic->width + 2) > K6_MAX_TAB_FLOATS) {
      ctx->last_error = "conversion: the coefficient table of " + std::to_string(fi) + " -> " + std::to_string(fo) +
                        " Hz exceeds 2^22 floats";
      return VPZ_E_UNSUPPORTED;
    }
    if (build) {
      int rc = conv_filter(ctx, fi, fo, &ic->f);
      if (rc) return rc;
    }
  }
  // tile size: the staged span (frames x staged floats per frame) within K6_SMEM_BUDGET where one output allows it
  const uint32_t per_frame = ic->mix == VPZ_MIX_MEAN ? ic->C + 1 : ic->C;
  const uint64_t budget = K6_SMEM_BUDGET / 4 / per_frame;
  auto span = [&](uint64_t m) { return ic->filter ? ((ic->n - 1) + (m - 1) * ic->o) / ic->n + 2 * ic->width + 2 : m; };
  uint64_t m = K6_MAX_OUTS;
  if (ic->filter) {
    const uint64_t fixed = 2 * ic->width + 3;
    m = budget > fixed ? std::min<uint64_t>(m, (budget - fixed) * ic->n / ic->o + 1) : 1;
  } else {
    m = std::min<uint64_t>(m, budget);
  }
  while (m > 1 && span(m) > budget) m--;
  ic->m = (uint32_t)m;
  ic->smem_floats = (uint32_t)(span(m) * per_frame);
  // a one-output tile that still does not fit (thousands of taps times many staged channels) fails here, before
  // anything is decoded, and so does the size query; launch_k6 keeps the same check as a backstop
  if ((size_t)ic->smem_floats * 4 > dev::max_smem_per_block()) {
    ctx->last_error = "conversion: a K6 tile of " + std::to_string(fi) + " -> " + std::to_string(fo) + " Hz from " +
                      std::to_string(C) + " channels needs " + std::to_string((size_t)ic->smem_floats * 4) +
                      " bytes of shared memory, more than the device's " + std::to_string(dev::max_smem_per_block());
    return VPZ_E_UNSUPPORTED;
  }
  return VPZ_OK;
}

size_t conv_tile_count(const ItemConv& ic, uint64_t len) { return (size_t)((len + ic.m - 1) / ic.m); }

// K6 tiles of one item: `len` output samples (element base `base`), output sample 0 is j = j_first of the stream;
// its source is `src_len` frames at float offset src, source frame 0 is k = k_first; outputs from `valid` on are zero
VpzConvTile* put_conv_tiles(VpzConvTile* out, const ItemConv& ic, uint64_t src, int64_t k_first, uint64_t src_len,
                            uint64_t base, uint64_t len, int64_t j_first, uint64_t valid) {
  for (uint64_t s = 0; s < len; s += ic.m) {
    VpzConvTile t;
    memset(&t, 0, sizeof(t));
    const uint32_t n = (uint32_t)std::min<uint64_t>(ic.m, len - s);
    const int64_t j0 = j_first + (int64_t)s;
    t.src = src;
    t.base = base;
    t.len = len;
    t.first = s;
    t.n = n;
    t.valid = valid > s ? (uint32_t)std::min<uint64_t>(valid - s, n) : 0;
    t.src_len = (uint32_t)src_len;
    t.ch_src = (uint8_t)ic.C;
    t.ch_out = (uint8_t)ic.Cout;
    t.mix = (uint8_t)ic.mix;
    if (ic.filter) {
      const int64_t a = j0 * ic.o;
      t.taps = ic.f->dev.p ? static_cast<const float*>(ic.f->dev.p) : nullptr;
      t.ro = ic.o;
      t.rn = ic.n;
      t.width = ic.width;
      t.p0 = (uint32_t)(j0 % ic.n);
      t.r0 = (uint32_t)(a % ic.n);
      t.s_first = a / ic.n - ic.width - k_first;
      t.span = (t.r0 + (n - 1) * ic.o) / ic.n + 2 * ic.width + 2;
    } else {
      t.ro = t.rn = 1;
      t.s_first = j0 - k_first;
      t.span = n;
    }
    *out++ = t;
  }
  return out;
}

// Uploads the K6 tiles of slot `slot` and launches K6 from src into the caller's buffer
int convert_tiles(vpz_ctx* ctx, int slot, const void* src, const DevOut& o) {
  PlaceBufs& pb = *ctx->place;
  const size_t n = pb.h_ctiles[slot].n;
  if (!n) return VPZ_OK;
  uint32_t smem = 0;
  for (size_t i = 0; i < n; i++) {
    const VpzConvTile& t = pb.h_ctiles[slot].p[i];
    smem = std::max<uint32_t>(smem, t.span * (t.ch_src + (t.mix == VPZ_MIX_MEAN ? 1u : 0u)));
  }
  if (!pb.d_ctiles[slot].reserve(n * sizeof(VpzConvTile), ctx->last_error)) return VPZ_E_CUDA;
  int rc = dev::h2d(pb.d_ctiles[slot].p, pb.h_ctiles[slot].p, n * sizeof(VpzConvTile), ctx->stream, ctx->last_error);
  if (rc) return rc;
  K6Params kp;
  kp.src = static_cast<const float*>(src);
  kp.out = o.p;
  kp.tiles = static_cast<const VpzConvTile*>(pb.d_ctiles[slot].p);
  kp.n_tiles = (uint32_t)n;
  kp.smem_floats = smem;
  kp.planar = (o.format & VPZ_OUT_PLANAR) ? 1 : 0;
  kp.out16 = (o.format & VPZ_OUT_S16) ? 1 : 0;
  rc = dev::launch_k6(kp, ctx->stream, ctx->last_error);
  if (!rc) ctx->kernel_launches++;
  return rc;
}

// Channels and rate from the identification header on the first page of a container image (0, 0 when it is not
// where a well-formed file has it: the decode reports that file's error)
void peek_id_header(const uint8_t* d, size_t len, int* channels, int* rate) {
  *channels = *rate = 0;
  if (!d || len < 27 || memcmp(d, "OggS", 4)) return;
  const size_t body = 27 + (size_t)d[26];
  if (body + 16 > len || memcmp(d + body, "\x01vorbis", 7)) return;
  *channels = d[body + 11];
  *rate = (int)((uint32_t)d[body + 12] | (uint32_t)d[body + 13] << 8 | (uint32_t)d[body + 14] << 16 | (uint32_t)d[body + 15] << 24);
}
}  // namespace

// out16: dst holds int16 elements (same element offsets), produced on the GPU by K3
// dout: the caller's device buffer instead (dst is its address): K3 writes fp32, K5 places and converts
static int64_t decode_files_impl(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens, int clip,
                                 float* dst, size_t dst_floats, int64_t* sample_counts, int out16,
                                 const DevOut* dout = nullptr) {
  if (!ctx || (n && (!datas || !lens))) return VPZ_E_ARGUMENT;
  VPZ_USE(ctx);
  if (!ctx->pool) {
    unsigned t = ctx->host_threads > 0 ? (unsigned)ctx->host_threads
                                       : std::max(1u, std::min(std::thread::hardware_concurrency(), 32u));
    ctx->pool = new (std::nothrow) ThreadPool(t);
    if (!ctx->pool) return VPZ_E_NOMEM;
  }
  ThreadPool* pool = ctx->pool;
  // The call is bound by the PCM copy, and the copy gets SLOWER the more host threads stage packets beside it
  // (16-core box, 4,096 streams: 2 / 4 / 8 / 16 threads = 169 / 167 / 171 / 178 ms; with 2 the 16-bit path turns
  // host-bound): a few threads are the optimum, "bulk_threads" (default 4).  The device-output call has no PCIe
  // copy to slow down: "bulk_threads_device".
  struct PoolLimit {
    ThreadPool* p;
    PoolLimit(ThreadPool* pool_, unsigned k) : p(pool_) { p->set_limit(k); }
    ~PoolLimit() { p->set_limit(0); }
  } pool_limit(pool, (unsigned)std::max(0, dout ? ctx->bulk_threads_device : ctx->bulk_threads));
  const bool trace = getenv("VPZ_TRACE") != nullptr;
  double t_scan = 0, t_init = 0, t_plan = 0, t_commit = 0, t_launch = 0, t_wait = 0;
  auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  double t0 = now(), t1;
  const uint32_t G = (uint32_t)std::max(1, ctx->bulk_group);
  // Group boundaries.  The first groups are small (G/8, G/4, G/2): nothing can be copied back before the first
  // group has been scanned, planned and decoded, and the call is bound by the PCM copy, so a short head start
  // is worth more than full-size batches there.
  std::vector<uint32_t> bounds;
  bounds.push_back(0);
  // A group also closes when its images reach "bulk_group_mib" (128 MiB): a batch addresses its entry-index area
  // (about 8x the compressed bytes) and its spectra (about 11 floats per compressed byte of typical music) with
  // 32 bits, and three batches of that size stay far inside the device memory.  One file alone may be larger
  // (up to ~384 MiB, hours of audio, before batch_commit refuses it).
  const uint64_t kGroupBytes = ctx->bulk_group_bytes > 0 ? (uint64_t)ctx->bulk_group_bytes : (uint64_t)ctx->bulk_group_mib << 20;
  for (uint32_t first = 0, g = 0; first < n; g++) {
    uint32_t want = G;
    if (dst && g < 3 && G >= 8) want = G >> (3 - g);
    uint32_t cnt = 0;
    uint64_t bytes = 0;
    while (cnt < want && first + cnt < n && (cnt == 0 || bytes + lens[first + cnt] <= kGroupBytes))
      bytes += lens[first + cnt++];
    first += cnt;
    bounds.push_back(first);
  }
  const uint32_t n_groups = (uint32_t)bounds.size() - 1;
  std::vector<std::unique_ptr<BulkJob>> held[3];  // jobs stay alive while their batch may still be in flight
  bool used[3] = {false, false, false};
  int64_t total = 0;
  int rc = VPZ_OK;
  uint32_t group = 0;
  // K0 runs one group AHEAD on its own stream: while the workers plan group g, the images of group g+1 are
  // already on their way to the device and through the page scan
  if (ctx->gpu_scan && n_groups)
    rc = scan_begin(ctx, 0, bounds[1], datas, lens, pool);
  t1 = now(); t_scan += t1 - t0;
  for (; group < n_groups && !rc; group++) {
    const uint32_t first = bounds[group], cnt = bounds[group + 1] - first;
    const int slot = (int)(group % 3);
    t0 = now();
    if (dst && used[slot]) {
      if ((rc = dev::event_sync(ctx->bulk_done[slot], ctx->last_error))) break;
    }
    t1 = now(); t_wait += t1 - t0; t0 = t1;
    std::vector<std::unique_ptr<BulkJob>>& jobs = held[slot];
    jobs.clear();
    jobs.resize(cnt);
    // 1. page scan: capture patterns, lacing sums and page CRCs on the device (K0, one warp per image), the
    //    per-serial filing of the page records on the worker threads; "gpu_scan" 0 = all of it on the host
    ScanResult sr;
    if (ctx->gpu_scan) {
      if (group + 1 < n_groups) {
        const uint32_t nf = bounds[group + 1], nc = bounds[group + 2] - nf;
        if ((rc = scan_begin(ctx, (int)((group + 1) & 1), nc, datas + nf, lens + nf, pool))) break;
      }
      if ((rc = scan_end(ctx, (int)(group & 1), &sr))) break;
    }
    pool->parallel_for(cnt, [&](size_t i) {
      jobs[i].reset(new BulkJob);
      BulkJob& j = *jobs[i];
      if (ctx->gpu_scan && !sr.out[i].overflow) {
        const VpzScanOut& o = sr.out[i];
        j.rc = j.cont.scan_from_records(datas[first + i], lens[first + i], sr.pages + sr.files[i].page_base, o.n_pages,
                                        ((uint64_t)o.waste_hi << 32) | o.waste_lo, o.crc_failures);
      } else {
        j.rc = j.cont.scan(datas[first + i], lens[first + i]);   // host scan (a file of unusually many tiny pages)
      }
      if (!j.rc) j.rc = stream_prepare(&j.dec, j.cont.streams[0], &j.err);
    });
    t1 = now(); t_scan += t1 - t0; t0 = t1;
    // 2. headers + setup cache (shared, serial: identical header pairs collapse onto one device image)
    for (uint32_t i = 0; i < cnt && !rc; i++) {
      BulkJob& j = *jobs[i];
      if (j.rc) ctx->last_error = j.err;
      rc = j.rc ? j.rc : stream_attach(&j.dec, ctx);
    }
    if (rc) break;
    t1 = now(); t_init += t1 - t0; t0 = t1;
    // 3. packet walk + window plan + run plan -- parallel, per-stream state only
    pool->parallel_for(cnt, [&](size_t i) {
      BulkJob& j = *jobs[i];
      plan_window(&j.dec, 0, &j.win);
      resolve_drain(&j.dec, &j.win);
      j.rc = plan_submit(&j.dec, &j.win, &j.err);
    });
    t1 = now(); t_plan += t1 - t0; t0 = t1;
    std::vector<RunPlan*> plans;
    plans.reserve(cnt);
    uint64_t group_floats = 0, group_out = 0;   // batch PCM floats; elements of the destination
    std::vector<ItemConv> conv(dout && dout->conv ? cnt : 0);
    for (uint32_t i = 0; i < cnt; i++) {
      BulkJob& j = *jobs[i];
      if (j.rc) {
        rc = j.rc;
        ctx->last_error = j.err;
        break;
      }
      int64_t samples = j.win.has_plan ? j.win.plan.samples : 0, out = samples;
      uint32_t ch = (uint32_t)j.dec.channels();
      if (!conv.empty()) {
        if ((rc = conv_plan(ctx, *dout->conv, j.dec.setup->host.id.sample_rate, (int)ch, dst != nullptr, &conv[i]))) break;
        out = conv[i].out_len(samples);
        ch = conv[i].Cout;
        if (dout->offsets) dout->offsets[first + i] = total + (int64_t)group_out;
      }
      if (sample_counts) sample_counts[first + i] = out;
      group_floats += (uint64_t)samples * j.dec.channels();
      group_out += (uint64_t)out * ch;
      if (j.win.has_plan) plans.push_back(&j.win.plan);
    }
    if (rc) break;
    if (!dst) {  // size query: nothing is decoded
      total += (int64_t)group_out;
      continue;
    }
    if ((uint64_t)total + group_out > dst_floats) {
      ctx->last_error = "destination buffer too small";
      rc = VPZ_E_ARGUMENT;
      break;
    }
    if (!ctx->bulk[slot] && (rc = vpz_batch_create(ctx, &ctx->bulk[slot]))) break;
    if (!ctx->bulk_done[slot]) {   // (the batches are shared with vpz_decode_excerpts, which may have made them first)
      ctx->bulk_done[slot] = dev::event_create();
      ctx->bulk_ready[slot] = dev::event_create();
      if (!ctx->bulk_done[slot] || !ctx->bulk_ready[slot]) {
        rc = VPZ_E_CUDA;
        break;
      }
    }
    vpz_batch* b = ctx->bulk[slot];
    vpz_batch_reset(b);
    // 4. copy packet bytes + descriptors into pinned staging -- parallel
    if ((rc = batch_commit(b, plans.data(), plans.size(), pool, nullptr))) break;
    if (b->total_floats != group_floats) {
      ctx->last_error = "internal: group plan and batch plan disagree";
      rc = VPZ_E_INVALID_OP;
      break;
    }
    if (dout && group_floats) {
      // 4b. K5 tiles: file i of the group is the batch PCM at its offset in the group (runs are committed in
      //     file order), placed at element total + that offset.  The _conv call: a converted file gets K6 tiles
      //     instead, placed at its offset in the converted layout (oo).
      std::vector<uint64_t> off(cnt + 1, 0), oo(cnt + 1, 0);
      std::vector<size_t> first_tile(cnt + 1, 0), first_ctile(cnt + 1, 0);
      for (uint32_t i = 0; i < cnt; i++) {
        const BulkJob& j = *jobs[i];
        const int64_t samples = j.win.has_plan ? j.win.plan.samples : 0;
        const bool on = !conv.empty() && conv[i].on;
        off[i + 1] = off[i] + (uint64_t)samples * j.dec.channels();
        oo[i + 1] = oo[i] + (on ? (uint64_t)conv[i].out_len(samples) * conv[i].Cout : (uint64_t)samples * j.dec.channels());
        first_tile[i + 1] = first_tile[i] + (on ? 0 : tile_count((uint64_t)samples));
        first_ctile[i + 1] = first_ctile[i] + (on ? conv_tile_count(conv[i], (uint64_t)conv[i].out_len(samples)) : 0);
      }
      HostBuf<VpzPlaceTile>& ht = ctx->place->h_tiles[slot];
      HostBuf<VpzConvTile>& hc = ctx->place->h_ctiles[slot];
      if (!ht.reserve(first_tile[cnt]) || !hc.reserve(first_ctile[cnt])) {
        rc = VPZ_E_NOMEM;
        break;
      }
      ht.n = first_tile[cnt];
      hc.n = first_ctile[cnt];
      pool->parallel_for(cnt, [&](size_t i) {
        const BulkJob& j = *jobs[i];
        const uint64_t samples = j.win.has_plan ? (uint64_t)j.win.plan.samples : 0;
        if (!conv.empty() && conv[i].on) {
          const uint64_t out = (uint64_t)conv[i].out_len((int64_t)samples);
          put_conv_tiles(hc.p + first_ctile[i], conv[i], off[i], 0, samples, (uint64_t)total + oo[i], out, 0, out);
        } else {
          put_tiles(ht.p + first_tile[i], off[i], (uint64_t)total + oo[i], samples, 0, samples, (uint32_t)j.dec.channels());
        }
      });
    }
    t1 = now(); t_commit += t1 - t0; t0 = t1;
    if (group_floats && dout) {
      // 5. H2D + K1 + K3 + K5 (batch PCM -> the caller's device buffer) on the compute stream
      if ((rc = batch_decode(b, clip, 0))) break;
      if ((rc = place_tiles(ctx, slot, b, *dout, 0))) break;   // (K3 has clipped)
      if (dout->conv && (rc = convert_tiles(ctx, slot, b->d_pcm.p, *dout))) break;
    } else if (group_floats) {
      // 5. H2D + K1 + K3 on the compute stream, then the PCM of this group on the copy stream
      if ((rc = batch_decode(b, clip, out16))) break;
      dev::event_record(ctx->bulk_ready[slot], ctx->stream);
      dev::stream_wait_event(ctx->copy_stream, ctx->bulk_ready[slot]);
      if (out16)
        rc = dev::d2h(reinterpret_cast<int16_t*>(dst) + total, b->d_pcm.p, group_floats * 2, ctx->copy_stream, ctx->last_error);
      else
        rc = dev::d2h(dst + total, b->d_pcm.p, group_floats * 4, ctx->copy_stream, ctx->last_error);
      if (rc) break;
    }
    dev::event_record(ctx->bulk_done[slot], dout ? ctx->stream : ctx->copy_stream);
    t1 = now(); t_launch += t1 - t0; t0 = t1;
    used[slot] = true;
    total += (int64_t)group_out;
  }
  // drain the pipeline (also on errors: buffers must not be in flight when the jobs are freed)
  for (int s = 0; s < 3; s++)
    if (used[s]) {
      int r2 = dev::event_sync(ctx->bulk_done[s], ctx->last_error);
      if (!rc) rc = r2;
    }
  if (dst) {
    int r2 = dev::stream_sync(ctx->stream, ctx->last_error);
    if (!rc) rc = r2;
    for (int s = 0; s < 3; s++)
      if (ctx->bulk[s]) vpz_batch_reset(ctx->bulk[s]);  // drop setup references; device buffers stay allocated
  }
  if (trace) {
    fprintf(stderr, "vpz_decode_files%s: %u files, %u groups: scan %.1f init %.1f plan %.1f commit %.1f launch %.1f wait %.1f drain %.1f ms\n",
            dout ? "_device" : "", n, group, t_scan, t_init, t_plan, t_commit, t_launch, t_wait, now() - t0);
    fprintf(stderr, "  inside launch (cumulative): order sort %.1f, upload incl. sort %.1f, kernel launches %.1f ms\n",
            vpz::g_trace_ms[0], vpz::g_trace_ms[1], vpz::g_trace_ms[2]);
  }
  return rc ? rc : total;
}

extern "C" {

int64_t vpz_decode_files(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens, int clip,
                         float* dst, size_t dst_floats, int64_t* sample_counts) {
  return decode_files_impl(ctx, n, datas, lens, clip, dst, dst_floats, sample_counts, 0);
}

int64_t vpz_decode_files_s16(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens, int clip,
                             int16_t* dst, size_t dst_samples, int64_t* sample_counts) {
  return decode_files_impl(ctx, n, datas, lens, clip, reinterpret_cast<float*>(dst), dst_samples, sample_counts, 1);
}

int64_t vpz_decode_files_device(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens, int clip,
                                int format, void* dst_dev, size_t dst_elems, int64_t* sample_counts, void* stream) {
  if (!ctx || (n && (!datas || !lens))) return VPZ_E_ARGUMENT;
  VPZ_USE(ctx);
  DevOut o;
  o.p = dst_dev;
  o.format = format;
  o.stream = stream;
  dev::Event* ev = nullptr;
  int rc = device_output_begin(ctx, o, &ev);
  if (rc) return device_output_end(ctx, ev, rc);
  return device_output_end(ctx, ev, decode_files_impl(ctx, n, datas, lens, clip, static_cast<float*>(dst_dev), dst_elems,
                                                      sample_counts, 0, &o));
}

int64_t vpz_decode_files_device_conv(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens, int clip,
                                     const vpz_out_conv* conv, void* dst_dev, size_t dst_elems, int64_t* sample_counts,
                                     int64_t* dst_offsets, void* stream) {
  if (!ctx || (n && (!datas || !lens))) return VPZ_E_ARGUMENT;
  VPZ_USE(ctx);
  int rc = conv_check(ctx, conv);
  if (rc) return rc;
  // streams the conversion refuses fail the call before anything is decoded
  for (uint32_t i = 0; i < n; i++) {
    int ch, rate;
    peek_id_header(datas[i], lens[i], &ch, &rate);
    ItemConv ic;
    if (ch > 0 && rate > 0 && (rc = conv_plan(ctx, *conv, rate, ch, false, &ic))) return rc;
  }
  DevOut o;
  o.p = dst_dev;
  o.format = conv->format;
  o.stream = stream;
  o.conv = conv;
  o.offsets = dst_offsets;
  dev::Event* ev = nullptr;
  rc = device_output_begin(ctx, o, &ev);
  if (rc) return device_output_end(ctx, ev, rc);
  return device_output_end(ctx, ev, decode_files_impl(ctx, n, datas, lens, clip, static_cast<float*>(dst_dev), dst_elems,
                                                      sample_counts, 0, &o));
}


// ---- bulk random access (BASELINE config 5): many short excerpts, SeekTo + Read each --------------
// Every excerpt behaves like a fresh reader on its file that calls SeekTo(start) and then reads `count`
// samples per channel.  The host runs the provider side of SeekTo for all excerpts (page search, one
// packet of pre-roll), plans each excerpt's window (plan_window with the seek state, so the stale-position
// trim of quirk Q5 and the end-of-stream rules are the reader's own), the GPU decodes the windows of
// a group of excerpts in one batch, and the consumer side of SeekTo / Read (seek_finish, stream_read)
// runs against that batch's PCM.  Groups are double-buffered: the host delivers group g-1 while the
// GPU decodes group g.
namespace {
struct ExcerptFile {
  OggContainer cont;
  StreamDec master;
  int rc = 0;
  std::string err;
};
struct ExcerptJob {
  uint32_t index = 0;          // position in the caller's arrays
  std::unique_ptr<Window> win; // made by the planning worker, dropped by the replaying one (a Window is ~600 bytes)
  int64_t pos = 0;             // granule position the provider reported for the target packet
  int status = 0;              // error of the provider side of SeekTo
  int run = -1, drain_run = -1;
  size_t pieces[2] = {0, 0};   // corpus call: K7 pieces of the window's plan / drain plan, SIZE_MAX: not in the image
};
struct ExcerptTask {           // consecutive excerpts of one file, handled by one worker with its own cursor
  uint32_t file = 0;
  size_t first = 0, count = 0; // range in the sorted job array
  std::unique_ptr<LogicalStream> ls;
  std::unique_ptr<StreamDec> dec;
};
}  // namespace

// A file may take the device seek index when it holds ONE logical stream whose pages are in perfect order: then
// every packet FillPageEndGranuleCache (Ogg/PacketProvider.cs:203-307) walks is valid and K0g's page-parallel
// walk (k0_pages.cuh) adds up the same numbers.  Anything else keeps the host's lazy cache (ogg.cpp).
static bool clean_single_stream(const ExcerptFile& f, const VpzPageRec* r, uint32_t n) {
  if (f.cont.streams.size() != 1 || n == 0 || f.cont.streams[0]->pages.size() != n) return false;
  bool data = false;
  int64_t last_granule = -1;
  for (uint32_t i = 0; i < n; i++) {
    if (r[i].is_resync || r[i].serial != r[0].serial) return false;
    if (i > 0 && r[i].seq != r[i - 1].seq + 1) return false;
    const bool continuation = (r[i].flags & 1) != 0;
    if (continuation != (i > 0 && r[i - 1].is_continued)) return false;
    if (continuation && r[i].is_continued && r[i].packet_count == 1) return false;   // a packet over three pages
    if ((r[i].flags & 4) && i + 1 != n) return false;                                 // pages behind the end of the stream
    const int64_t g = (int64_t)(((uint64_t)r[i].granule_hi << 32) | r[i].granule_lo);
    if (g != -1) {
      if (g < last_granule) return false;
      last_granule = g;
      data |= g > 0;
    }
  }
  return data && !r[n - 1].is_continued;
}

// Opens the files of a random-access batch: page scan (K0, or the host with "gpu_scan" 0), headers and setup
// tables, and the page-end granule index SeekTo searches in (K0g for clean files; files_on_device counts them).
// scan: the device scan's result (its staged images stay on the device until the next scan), when there was one.
static int open_excerpt_files(vpz_ctx* ctx, uint32_t n_files, const uint8_t* const* datas, const size_t* lens,
                              std::vector<std::unique_ptr<ExcerptFile>>& files, uint32_t* files_on_device,
                              ScanResult* scan = nullptr) {
  ThreadPool* pool = ctx->pool;
  ScanResult sr;
  const bool dev_scan = ctx->gpu_scan != 0 && n_files > 0;
  if (dev_scan) {
    int rc = scan_begin(ctx, 0, n_files, datas, lens, pool);
    if (!rc) rc = scan_end(ctx, 0, &sr);
    if (rc) return rc;
  }
  pool->parallel_for(n_files, [&](size_t i) {
    files[i].reset(new ExcerptFile);
    ExcerptFile& f = *files[i];
    if (dev_scan && !sr.out[i].overflow) {
      const VpzScanOut& o = sr.out[i];
      f.rc = f.cont.scan_from_records(datas[i], lens[i], sr.pages + sr.files[i].page_base, o.n_pages,
                                      ((uint64_t)o.waste_hi << 32) | o.waste_lo, o.crc_failures);
    } else {
      f.rc = f.cont.scan(datas[i], lens[i]);
    }
    if (!f.rc) f.rc = stream_prepare(&f.master, f.cont.streams[0], &f.err);
  });
  for (uint32_t i = 0; i < n_files; i++) {
    ExcerptFile& f = *files[i];
    if (f.rc) {
      ctx->last_error = f.err;
      return f.rc;
    }
    int rc = stream_attach(&f.master, ctx);
    if (rc) return rc;
  }
  uint32_t on_device = 0;
  if (dev_scan) {
    std::vector<VpzGranFile> gf;
    std::vector<uint32_t> which;
    for (uint32_t i = 0; i < n_files; i++) {
      ExcerptFile& f = *files[i];
      if (sr.out[i].overflow || !clean_single_stream(f, sr.pages + sr.files[i].page_base, sr.out[i].n_pages)) continue;
      const Setup& st = f.master.setup->host;
      if (st.modes.size() > 64) continue;
      VpzGranFile g;
      memset(&g, 0, sizeof(g));
      g.data_off = sr.files[i].data_off;
      g.page_base = sr.files[i].page_base;
      g.n_pages = sr.out[i].n_pages;
      for (size_t m = 0; m < st.modes.size(); m++)
        if (st.modes[m].block_flag) (m < 32 ? g.mode_flags_lo : g.mode_flags_hi) |= 1u << (m & 31);
      g.mode_bits = (uint8_t)st.mode_bits;
      g.nmodes = (uint8_t)st.modes.size();
      int l0 = 0, l1 = 0;
      while ((1 << l0) < st.id.size0) l0++;
      while ((1 << l1) < st.id.size1) l1++;
      g.log2_size0 = (uint8_t)l0;
      g.log2_size1 = (uint8_t)l1;
      gf.push_back(g);
      which.push_back(i);
    }
    const long long* idx = nullptr;
    if (!gf.empty()) {
      int rc = granule_index(ctx, 0, gf.data(), (uint32_t)gf.size(), &idx);
      if (rc) return rc;
    }
    for (size_t k = 0; k < gf.size(); k++) {
      LogicalStream* ls = files[which[k]]->master.ls;
      if (!ls->get_page((int64_t)gf[k].n_pages - 1)) continue;   // the host refuses the page list: its own path reports it
      ls->page_end_granules.assign(idx + gf[k].page_base, idx + gf[k].page_base + gf[k].n_pages);
      on_device++;
    }
  }
  for (uint32_t i = 0; i < n_files; i++) {
    int err = 0;
    files[i]->master.ls->total_granules(&err);   // host cache: walks every page once; the copies of the cursor inherit it
    if (err) return err;
  }
  if (files_on_device) *files_on_device = on_device;
  if (scan && dev_scan) *scan = sr;
  return VPZ_OK;
}

}  // extern "C"

// ---- corpus: the files of the excerpt calls opened once ----------------------------------------------------------
// vpz_corpus_open runs open_excerpt_files (page scan, headers, setup tables, seek index, total samples) once and keeps
// the images in device memory; every vpz_corpus_excerpts_device call then starts at the excerpt planning with the
// same opened files the plain call would have built, and K7 gathers its packet bytes from the device images.  The
// calls only read the files: each planning task copies a file's packet cursor, the masters stay as open left them, so
// one call leaves nothing behind for the next.
struct vpz_corpus {
  vpz_ctx* ctx = nullptr;
  std::vector<std::vector<uint8_t>> copies;   // copy != 0: the library's own images
  std::vector<std::unique_ptr<ExcerptFile>> files;
  std::vector<int64_t> samples;               // TotalSamples per file
  uint8_t* d_img = nullptr;                   // the images on the device: 16-byte aligned, >= 16 zero bytes behind each
  uint64_t d_bytes = 0;
  std::vector<uint64_t> dev_off;              // per file: offset of its image in d_img
  ~vpz_corpus() {
    if (ctx) VPZ_USE(ctx);
    files.clear();                            // gives the setup tables back to the context
    dev::free(d_img);
  }
};

// K7's pieces of one packet of a window: a view of the file's image is one piece, a packet assembled across pages one
// per page (its spans); n_pieces returns 0 when the packet is not in the image (the group then stages it on the host).
static const std::vector<OggSpan>* packet_spans(const Window& w, const uint8_t* p) {
  for (size_t a = 0; a < w.arena.size(); a++)
    if (w.arena[a].data() == p) return &w.arena_spans[a];
  return nullptr;
}
static bool in_image(const OggContainer& c, const uint8_t* p, uint32_t len) {
  return len == 0 || (p >= c.data && p + len <= c.data + c.len);
}
static size_t n_pieces(const OggContainer& c, const Window& w, const PktSrc& ps) {
  if (in_image(c, ps.p, ps.len)) return 1;
  const std::vector<OggSpan>* sp = packet_spans(w, ps.p);
  if (!sp || sp->empty()) return 0;
  for (const OggSpan& x : *sp)
    if (!in_image(c, x.p, x.len)) return 0;
  return sp->size();
}
static size_t plan_pieces(const OggContainer& c, const Window& w, const RunPlan& plan) {
  size_t n = 0;
  for (const PktSrc& ps : plan.src) {
    const size_t k = n_pieces(c, w, ps);
    if (!k) return SIZE_MAX;
    n += k;
  }
  return n;
}
// writes the pieces of `plan` (committed at byte `base` of the batch) from `pc` on; returns the packets over pages
static size_t put_pieces(const OggContainer& c, uint64_t img, const Window& w, const RunPlan& plan, uint64_t base,
                         VpzGatherPiece* pc) {
  size_t multi = 0;
  for (size_t q = 0; q < plan.src.size(); q++) {
    const PktSrc& ps = plan.src[q];
    uint32_t off = (uint32_t)(base + plan.byte_off[q]);
    if (in_image(c, ps.p, ps.len)) {
      *pc++ = VpzGatherPiece{ps.len ? img + (uint64_t)(ps.p - c.data) : img, off, ps.len};
      continue;
    }
    const std::vector<OggSpan>& sp = *packet_spans(w, ps.p);
    for (size_t i = 0; i < sp.size(); i++) {
      *pc++ = VpzGatherPiece{sp[i].len ? img + (uint64_t)(sp[i].p - c.data) : img, off,
                             sp[i].len | (i + 1 < sp.size() ? VPZ_PIECE_MORE : 0u)};
      off += sp[i].len;
    }
    multi++;
  }
  return multi;
}

// dout: the caller's device buffer instead of dst (dst is its address): K5 places the segments and zero-fills.
// corpus: its files (vpz_corpus_open) instead of datas / lens, and K7 instead of the packet bytes' staging.
static int64_t decode_excerpts_impl(vpz_ctx* ctx, uint32_t n_files, const uint8_t* const* datas, const size_t* lens,
                                    uint32_t n, const uint32_t* file_of, const int64_t* start, const int32_t* count,
                                    int clip, float* dst, size_t dst_floats, int64_t* dst_offsets, int32_t* got,
                                    const DevOut* dout, vpz_corpus* corpus = nullptr) {
  if (!ctx->pool) {
    unsigned t = ctx->host_threads > 0 ? (unsigned)ctx->host_threads
                                       : std::max(1u, std::min(std::thread::hardware_concurrency(), 32u));
    ctx->pool = new (std::nothrow) ThreadPool(t);
    if (!ctx->pool) return VPZ_E_NOMEM;
  }
  ThreadPool* pool = ctx->pool;
  const bool trace = getenv("VPZ_TRACE") != nullptr;
  auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  double t_files = 0, t_tasks = 0, t_plan = 0, t_commit = 0, t_launch = 0, t_wait = 0, t_deliver = 0, tt0 = now(), tt1;
  // ---- files: page scan, headers, setup tables, seek index (once per file) ---------------------------
  std::vector<std::unique_ptr<ExcerptFile>> own_files;
  std::vector<std::unique_ptr<ExcerptFile>>& files = corpus ? corpus->files : own_files;
  if (!corpus) {
    own_files.resize(n_files);
    int rc = open_excerpt_files(ctx, n_files, datas, lens, own_files, nullptr);
    if (rc) return rc;
  }
  tt1 = now(); t_files = tt1 - tt0; tt0 = tt1;
  // ---- the _conv call: what K6 does to each file's excerpts, and every converted excerpt's source window, which
  //      the rest of the call decodes as the plain call decodes an excerpt (start / count below are the windows)
  const vpz_out_conv* cv = dout ? dout->conv : nullptr;
  std::vector<ItemConv> fconv(cv ? n_files : 0);
  const int64_t* ostart = start;   // the caller's excerpts (output samples)
  const int32_t* ocount = count;
  std::vector<int64_t> xstart;
  std::vector<int32_t> xcount;
  // the filter of a resampled excerpt sees its file as the files call decodes it: TotalSamples samples, zeros after
  // them.  (A reader that seeks into the last packet delivers that packet untrimmed; the plain call and the
  // equal-rate mix keep those samples, the filter must not see them.)
  std::vector<int64_t> fend(cv ? n_files : 0, INT64_MAX);
  if (cv) {
    for (uint32_t f = 0; f < n_files; f++) {
      const StreamDec& m = files[f]->master;
      int rc = conv_plan(ctx, *cv, m.setup->host.id.sample_rate, m.channels(), dst != nullptr, &fconv[f]);
      if (rc) return rc;
      int err = 0;
      const int64_t total = fconv[f].filter ? m.ls->total_granules(&err) : -1;   // (cached by open_excerpt_files)
      if (!err && total >= 0) fend[f] = total;
    }
    xstart.resize(n);
    xcount.resize(n);
    for (uint32_t i = 0; i < n; i++) {
      if (file_of[i] >= n_files || start[i] < 0 || count[i] < 0) return VPZ_E_ARGUMENT;
      const ItemConv& ic = fconv[file_of[i]];
      int64_t lo = start[i], hi = start[i] + count[i];
      // (far beyond any stream: start * o stays inside 64 bits)
      if (ic.on && start[i] > ((int64_t)1 << 40)) {
        ctx->last_error = "conversion: start out of range";
        return VPZ_E_ARGUMENT;
      }
      if (ic.on) ic.window(start[i], count[i], &lo, &hi);
      if (hi - lo > INT32_MAX / VPZ_MAX_CH) {
        ctx->last_error = "conversion: source window too long";
        return VPZ_E_ARGUMENT;
      }
      xstart[i] = lo;
      xcount[i] = (int32_t)(hi - lo);
    }
    start = xstart.data();
    count = xcount.data();
  }
  // elements of excerpt i in the destination
  auto item_elems = [&](uint32_t i) {
    return cv ? (int64_t)ocount[i] * fconv[file_of[i]].Cout : (int64_t)count[i] * files[file_of[i]]->master.channels();
  };
  // ---- layout of the destination -------------------------------------------------------------------
  int64_t total = 0;
  for (uint32_t i = 0; i < n; i++) {
    // (count * channels is handed to Read as an int, like Span<float>.Length in the reference)
    if (file_of[i] >= n_files || start[i] < 0 || count[i] < 0 || count[i] > INT32_MAX / VPZ_MAX_CH) return VPZ_E_ARGUMENT;
    if (dst_offsets) dst_offsets[i] = total;
    total += item_elems(i);
  }
  if (!dst) return total;
  if ((uint64_t)total > dst_floats) {
    ctx->last_error = "destination buffer too small";
    return VPZ_E_ARGUMENT;
  }
  // ---- groups and tasks ---------------------------------------------------------------------------------
  // A GROUP is a contiguous range of the caller's excerpts (so its samples are one contiguous range of dst:
  // one device->host copy per group), up to 2,048 excerpts or 2^28 floats.  Inside a group the excerpts are
  // sorted by file and cut into TASKS of at most 32: consecutive excerpts of one file, planned by one worker
  // with its own packet cursor.
  std::vector<int64_t> own_offsets;
  if (!dst_offsets) {
    own_offsets.resize(n);
    int64_t acc = 0;
    for (uint32_t i = 0; i < n; i++) {
      own_offsets[i] = acc;
      acc += item_elems(i);
    }
    dst_offsets = own_offsets.data();
  }
  struct Group {
    uint32_t i0, i1;       // excerpts
    size_t t0, t1;         // tasks
    int64_t base, floats;  // range of dst
  };
  std::vector<Group> groups;
  for (uint32_t i = 0; i < n;) {
    Group g;
    g.i0 = i;
    g.base = dst_offsets[i];
    int64_t fl = 0;
    const uint32_t cap = groups.size() < 3 ? 256u << groups.size() : 2048u;   // short first groups: the GPU starts early
    while (i < n && i - g.i0 < cap && (i == g.i0 || fl < ((int64_t)1 << 28))) {
      fl += (int64_t)count[i] * files[file_of[i]]->master.channels();
      i++;
    }
    g.i1 = i;
    g.floats = fl;
    g.t0 = g.t1 = 0;
    groups.push_back(g);
  }
  std::vector<ExcerptJob> jobs(n);
  std::vector<ExcerptTask> tasks;
  {
    std::vector<uint32_t> order(n);
    for (uint32_t i = 0; i < n; i++) order[i] = i;
    for (Group& g : groups) {
      std::stable_sort(order.begin() + g.i0, order.begin() + g.i1, [&](uint32_t a, uint32_t b) { return file_of[a] < file_of[b]; });
      g.t0 = tasks.size();
      for (size_t i = g.i0; i < g.i1;) {
        size_t j = i;
        const uint32_t f = file_of[order[i]];
        while (j < g.i1 && j - i < 32 && file_of[order[j]] == f) j++;
        ExcerptTask t;
        t.file = f;
        t.first = i;
        t.count = j - i;
        tasks.push_back(std::move(t));
        i = j;
      }
      g.t1 = tasks.size();
    }
    for (uint32_t i = 0; i < n; i++) jobs[i].index = order[i];
  }
  for (ExcerptTask& t : tasks) files[t.file]->master.setup->refs++;   // one reference per task decoder (serial: plain counters)
  struct TaskRefs {   // a task whose decoder was never made (an error on the way) gives its reference back here
    std::vector<ExcerptTask>& tasks;
    std::vector<std::unique_ptr<ExcerptFile>>& files;
    ~TaskRefs() {
      for (ExcerptTask& t : tasks)
        if (!t.dec) setup_release(files[t.file]->master.setup);
    }
  } task_refs{tasks, files};
  tt1 = now(); t_tasks = tt1 - tt0; tt0 = tt1;
  // Provider side of SeekTo + window plan of every excerpt of tasks [t0, t1): each task works on its own copy of
  // the file's packet cursor (which inherits the file's page-end granule cache)
  auto plan_tasks = [&](size_t t0, size_t t1) {
    pool->parallel_for(t1 - t0, [&](size_t k) {
      ExcerptTask& t = tasks[t0 + k];
      t.dec.reset(new StreamDec);
      StreamDec* d = t.dec.get();
      d->ctx = ctx;
      d->setup = files[t.file]->master.setup;
      d->clip = clip != 0;
      d->planned_only = true;
      t.ls.reset(new LogicalStream(*files[t.file]->master.ls));
      d->ls = t.ls.get();
      d->ls->granule_count = [d](const OggPacket& pk) { return d->granule_count(pk); };
      for (size_t q = 0; q < t.count; q++) {
        ExcerptJob& j = jobs[t.first + q];
        const int64_t sp = start[j.index];
        d->current_position = 0;   // a fresh reader (the stale position enters SeekTo's end-of-stream trim, quirk Q5)
        d->has_clipped = false;
        j.status = seek_begin(d, sp, &j.pos);
        if (j.status) continue;
        j.win.reset(new Window);
        plan_window(d, 0, j.win.get(), (sp - j.pos) + (int64_t)count[j.index]);
        d->seek_left = 0;
        resolve_drain(d, j.win.get());
        std::string err;
        int rc = plan_submit(d, j.win.get(), &err);
        if (rc) j.status = rc;
        if (!rc && corpus) {   // K7's pieces of the window (SIZE_MAX: a packet outside the image)
          const OggContainer& c = files[t.file]->cont;
          if (j.win->has_plan) j.pieces[0] = plan_pieces(c, *j.win, j.win->plan);
          if (j.win->has_drain_plan) j.pieces[1] = plan_pieces(c, *j.win, j.win->drain_plan);
        }
      }
    });
  };
  // ---- the groups through two batches -------------------------------------------------------------------
  // Per group: commit the windows to a batch; replay the consumer side of SeekTo / Read for every excerpt
  // WITHOUT samples (it only depends on the packets' sample counts) to get got[] and the copy segments; then
  // on the device H2D + K1a + K1b + K3 + K4 (segments -> the group's dense output) and one copy of that output
  // into dst on the copy stream.  The host never touches a sample; while the GPU works on group g the host
  // commits and replays group g + 1.
  if (!ctx->xb) {
    ctx->xb = new (std::nothrow) ExcerptBufs;
    if (!ctx->xb) return VPZ_E_NOMEM;
  }
  ExcerptBufs& xb = *ctx->xb;
  int rc = VPZ_OK;
  bool used[2] = {false, false};
  std::vector<std::vector<VpzCopySeg>> task_segs;
  std::vector<std::vector<VpzPlaceTile>> task_tiles, task_xtiles;   // K5 into dst / into the scratch (_conv)
  std::vector<std::vector<VpzConvTile>> task_ctiles;                 // K6 (_conv)
  std::vector<uint64_t> xoff(cv ? n : 0);                             // float offset of a converted excerpt's window in the scratch
  uint64_t gathered_bytes = 0, gathered_pieces = 0;                   // K7 (corpus call): staged bytes written, pieces,
  uint64_t gathered_multi = 0, gathered_groups = 0;                   // packets over pages, groups it gathered
  for (size_t gi = 0; gi < groups.size() && !rc; gi++) {
    const Group& g = groups[gi];
    const int slot = (int)(gi & 1);
    tt0 = now();
    if (!ctx->bulk[slot]) {
      if ((rc = vpz_batch_create(ctx, &ctx->bulk[slot]))) break;
    }
    if (!xb.done[slot]) {
      xb.done[slot] = dev::event_create();
      xb.ready[slot] = dev::event_create();
      if (!xb.done[slot] || !xb.ready[slot]) {
        rc = VPZ_E_CUDA;
        break;
      }
    }
    if (used[slot] && (rc = dev::event_sync(xb.done[slot], ctx->last_error))) break;   // group gi - 2 has left the slot
    tt1 = now(); t_wait += tt1 - tt0; tt0 = tt1;
    vpz_batch* b = ctx->bulk[slot];
    vpz_batch_reset(b);
    plan_tasks(g.t0, g.t1);   // while the GPU still works on the previous group
    tt1 = now(); t_plan += tt1 - tt0; tt0 = tt1;
    std::vector<RunPlan*> plans;
    std::vector<std::pair<ExcerptJob*, int>> owner;   // plan -> (job, 0 run / 1 drain run)
    for (size_t ti = g.t0; ti < g.t1; ti++)
      for (size_t q = 0; q < tasks[ti].count; q++) {
        ExcerptJob& j = jobs[tasks[ti].first + q];
        if (j.status) continue;
        if (j.win->has_plan) {
          plans.push_back(&j.win->plan);
          owner.push_back({&j, 0});
        }
        if (j.win->has_drain_plan) {
          plans.push_back(&j.win->drain_plan);
          owner.push_back({&j, 1});
        }
      }
    // corpus call: K7 gathers the packet bytes from the corpus's device images instead of the host staging them,
    // when every packet of the group lies in its file's image (a view, or assembled from views of several pages);
    // batch_commit's fill threads write each plan's pieces
    bool gather = corpus && corpus->d_img && b->bytes.n == 0;
    std::vector<size_t> piece_at(gather ? plans.size() + 1 : 0);   // per plan: its first piece
    for (size_t k = 0; k < plans.size() && gather; k++) {
      const size_t np = owner[k].first->pieces[owner[k].second];
      gather = np != SIZE_MAX;
      piece_at[k + 1] = piece_at[k] + (gather ? np : 0);
    }
    std::atomic<size_t> multi{0};
    if (gather) {
      if (!b->pieces.reserve(piece_at.back())) {
        rc = VPZ_E_NOMEM;
        break;
      }
      b->pieces.n = piece_at.back();
      b->gather_images = corpus->d_img;
      b->gather_fill = [&](size_t k, uint64_t base) {
        const ExcerptJob& j = *owner[k].first;
        const uint32_t f = file_of[j.index];
        multi += put_pieces(files[f]->cont, corpus->dev_off[f], *j.win, *plans[k], base, b->pieces.p + piece_at[k]);
      };
    }
    int first = 0;
    if ((rc = batch_commit(b, plans.data(), plans.size(), pool, &first))) break;
    for (size_t k = 0; k < owner.size(); k++) (owner[k].second ? owner[k].first->drain_run : owner[k].first->run) = first + (int)k;
    if (gather) {
      b->gather_fill = nullptr;
      gathered_bytes += b->gather_bytes;
      gathered_pieces += piece_at.back();
      gathered_multi += multi;
      gathered_groups++;
    }
    tt1 = now(); t_commit += tt1 - tt0; tt0 = tt1;
    // consumer side, samples untouched: SeekTo's two packets, then Read until `count` samples or the end
    task_segs.assign(g.t1 - g.t0, std::vector<VpzCopySeg>());
    if (dout) task_tiles.assign(g.t1 - g.t0, std::vector<VpzPlaceTile>());
    uint64_t scratch = 0;
    if (cv) {
      task_xtiles.assign(g.t1 - g.t0, std::vector<VpzPlaceTile>());
      task_ctiles.assign(g.t1 - g.t0, std::vector<VpzConvTile>());
      for (uint32_t i = g.i0; i < g.i1; i++)
        if (fconv[file_of[i]].on) {
          xoff[i] = scratch;
          scratch += (uint64_t)count[i] * fconv[file_of[i]].C;
        }
      if (scratch && !ctx->place->d_scratch[slot].reserve(scratch * 4, ctx->last_error)) {
        rc = VPZ_E_CUDA;
        break;
      }
    }
    // a converted excerpt i whose window delivered `have` samples (status: SeekTo's error, or 0): zeros behind them
    // in the scratch, got by the output rate, K6 tiles from the scratch into dst
    auto conv_item = [&](size_t k, uint32_t i, int have, int status) {
      const ItemConv& ic = fconv[file_of[i]];
      append_tiles(task_xtiles[k], VPZ_TILE_ZERO, xoff[i], count[i], have, count[i] - have, ic.C);
      int64_t g_out = status;
      if (!status) {
        const int64_t e = start[i] + have;   // the window starts at k_lo = start[i]
        g_out = (ic.filter ? (e * ic.n + ic.o - 1) / ic.o : e) - ostart[i];
        g_out = std::max<int64_t>(0, std::min<int64_t>(g_out, ocount[i]));
      }
      if (got) got[i] = (int32_t)g_out;
      std::vector<VpzConvTile>& v = task_ctiles[k];
      const size_t at = v.size();
      v.resize(at + conv_tile_count(ic, (uint64_t)ocount[i]));
      put_conv_tiles(v.data() + at, ic, xoff[i], start[i], (uint64_t)count[i], (uint64_t)dst_offsets[i],
                     (uint64_t)ocount[i], ostart[i], status ? 0 : (uint64_t)g_out);
    };
    pool->parallel_for(g.t1 - g.t0, [&](size_t k) {
      ExcerptTask& t = tasks[g.t0 + k];
      StreamDec* d = t.dec.get();
      std::vector<VpzCopySeg>& segs = task_segs[k];
      segs.reserve(t.count * 8);
      for (size_t q = 0; q < t.count; q++) {
        ExcerptJob& j = jobs[t.first + q];
        const uint32_t i = j.index;
        const bool conv_on = cv && fconv[t.file].on;
        if (j.status) {
          if (got) got[i] = j.status;
          if (conv_on) conv_item(k, i, 0, j.status);
          else if (dout) append_tiles(task_tiles[k], VPZ_TILE_ZERO, dst_offsets[i], count[i], 0, count[i], files[t.file]->master.channels());
          continue;
        }
        int prc = place_window(d, b, j.win.get(), j.run, j.drain_run, 0);
        if (prc) {
          if (got) got[i] = prc;
          if (conv_on) conv_item(k, i, 0, prc);
          else if (dout) append_tiles(task_tiles[k], VPZ_TILE_ZERO, dst_offsets[i], count[i], 0, count[i], files[t.file]->master.channels());
          continue;
        }
        d->current_position = 0;
        d->reset_decoder();
        d->fault = 0;
        d->has_position = true;
        d->seek_left = 2;
        d->seek_pos = j.pos;
        d->q = std::move(j.win->entries);
        d->qh = 0;
        d->seg_sink = &segs;
        const size_t mark = segs.size();
        int src = seek_finish(d, start[i], j.pos);
        int have = 0;
        const int C = d->channels();
        if (!src) {
          while (have < count[i]) {
            d->seg_dst = (uint64_t)(dst_offsets[i] - g.base) + (uint64_t)have * C;
            int r = stream_read(d, nullptr, (count[i] - have) * C, count[i] - have, 0, true);
            if (r <= 0) break;
            have += r;
          }
        } else {
          segs.resize(mark);
        }
        d->seg_sink = nullptr;
        if (got) got[i] = src ? src : have;
        if (conv_on) {   // the window's segments (resampled: those inside the file) into the scratch, then K6
          const uint64_t item = (uint64_t)(dst_offsets[i] - g.base);
          const int inside = (int)std::min<int64_t>(have, std::max<int64_t>(0, fend[t.file] - start[i]));
          for (size_t sg = mark; sg < segs.size(); sg++) {
            const uint64_t first = (segs[sg].dst - item) / C;
            if (first < (uint64_t)inside)
              append_tiles(task_xtiles[k], segs[sg].src, xoff[i], count[i], first,
                           std::min<uint64_t>(segs[sg].n / C, (uint64_t)inside - first), C);
          }
          conv_item(k, i, src ? 0 : inside, src);
        } else if (dout) {   // the segments (samples [0, have)), then zeros up to count
          const uint64_t item = (uint64_t)(dst_offsets[i] - g.base);
          for (size_t sg = mark; sg < segs.size(); sg++)
            append_tiles(task_tiles[k], segs[sg].src, dst_offsets[i], count[i], (segs[sg].dst - item) / C, segs[sg].n / C, C);
          append_tiles(task_tiles[k], VPZ_TILE_ZERO, dst_offsets[i], count[i], have, count[i] - have, C);
        }
        j.win.reset();   // release the packet views / arena
      }
    });
    size_t n_segs = 0;
    for (const auto& v : task_segs) n_segs += v.size();
    if (!xb.h_segs[slot].reserve(n_segs)) {
      rc = VPZ_E_NOMEM;
      break;
    }
    {
      size_t at = 0;
      for (const auto& v : task_segs) {
        if (!v.empty()) memcpy(xb.h_segs[slot].p + at, v.data(), v.size() * sizeof(VpzCopySeg));
        at += v.size();
      }
      xb.h_segs[slot].n = n_segs;
    }
    size_t n_dst_tiles = 0;   // K5 tiles into dst; the scratch's (task_xtiles) follow them
    if (dout) {
      size_t n_tiles = 0;
      for (const auto& v : task_tiles) n_dst_tiles += v.size();
      n_tiles = n_dst_tiles;
      for (const auto& v : task_xtiles) n_tiles += v.size();
      HostBuf<VpzPlaceTile>& ht = ctx->place->h_tiles[slot];
      if (!ht.reserve(n_tiles)) {
        rc = VPZ_E_NOMEM;
        break;
      }
      size_t at = 0;
      for (const auto* vv : {&task_tiles, &task_xtiles})
        for (const auto& v : *vv) {
          if (!v.empty()) memcpy(ht.p + at, v.data(), v.size() * sizeof(VpzPlaceTile));
          at += v.size();
        }
      ht.n = n_tiles;
      if (cv) {
        size_t n_ct = 0;
        for (const auto& v : task_ctiles) n_ct += v.size();
        HostBuf<VpzConvTile>& hc = ctx->place->h_ctiles[slot];
        if (!hc.reserve(n_ct)) {
          rc = VPZ_E_NOMEM;
          break;
        }
        at = 0;
        for (const auto& v : task_ctiles) {
          if (!v.empty()) memcpy(hc.p + at, v.data(), v.size() * sizeof(VpzConvTile));
          at += v.size();
        }
        hc.n = n_ct;
      }
    }
    tt1 = now(); t_deliver += tt1 - tt0; tt0 = tt1;
    if (dout) {
      // H2D + K1a + K1b + K3 (unclipped) + K5: the segments and zeros straight into the caller's device buffer
      if (g.floats > 0 || (cv && ctx->place->h_ctiles[slot].n)) {
        if (b->total_floats && (rc = batch_decode(b, 0))) break;
        if ((rc = place_tiles(ctx, slot, b, *dout, clip, n_dst_tiles))) break;
        if (cv && (rc = convert_tiles(ctx, slot, ctx->place->d_scratch[slot].p, *dout))) break;
      }
      dev::event_record(xb.done[slot], ctx->stream);
      used[slot] = true;
      tt1 = now(); t_launch += tt1 - tt0; tt0 = tt1;
      continue;
    }
    if (g.floats > 0) {
      if (!xb.d_out[slot].reserve((size_t)g.floats * 4, ctx->last_error) ||
          !xb.d_segs[slot].reserve(std::max<size_t>(n_segs, 1) * sizeof(VpzCopySeg), ctx->last_error)) {
        rc = VPZ_E_CUDA;
        break;
      }
      // the reader clips while it copies: K3 decodes unclipped, K4 clips what it hands out
      if (b->total_floats && (rc = batch_decode(b, 0))) break;
      // samples no packet delivers (short reads at the end of a stream, failed seeks) read as zero
      if ((rc = dev::fill(xb.d_out[slot].p, 0, (size_t)g.floats * 4, ctx->stream, ctx->last_error))) break;
      if (n_segs) {
        if ((rc = dev::h2d(xb.d_segs[slot].p, xb.h_segs[slot].p, n_segs * sizeof(VpzCopySeg), ctx->stream, ctx->last_error))) break;
        K4Params kp;
        kp.pcm = static_cast<const float*>(b->d_pcm.p);
        kp.out = static_cast<float*>(xb.d_out[slot].p);
        kp.segs = static_cast<const VpzCopySeg*>(xb.d_segs[slot].p);
        kp.n_segs = (uint32_t)n_segs;
        kp.clip = clip ? 1 : 0;
        if ((rc = dev::launch_k4(kp, ctx->stream, ctx->last_error))) break;
        ctx->kernel_launches++;
      }
      dev::event_record(xb.ready[slot], ctx->stream);
      dev::stream_wait_event(ctx->copy_stream, xb.ready[slot]);
      if ((rc = dev::d2h(dst + g.base, xb.d_out[slot].p, (size_t)g.floats * 4, ctx->copy_stream, ctx->last_error))) break;
    }
    dev::event_record(xb.done[slot], ctx->copy_stream);
    used[slot] = true;
    tt1 = now(); t_launch += tt1 - tt0; tt0 = tt1;
  }
  tt0 = now();
  for (int s2 = 0; s2 < 2; s2++)
    if (used[s2]) {
      int r2 = dev::event_sync(xb.done[s2], ctx->last_error);
      if (!rc) rc = r2;
    }
  int r2 = dev::stream_sync(ctx->stream, ctx->last_error);
  if (!rc) rc = r2;
  t_wait += now() - tt0;
  if (trace) {
    fprintf(stderr, "vpz_decode_excerpts%s: %u excerpts, %zu tasks, %zu groups: files %.1f tasks %.1f plan %.1f commit %.1f replay %.1f launch %.1f wait %.1f ms",
            corpus ? "_corpus" : dout ? "_device" : "", n, tasks.size(), groups.size(), t_files, t_tasks, t_plan, t_commit, t_deliver, t_launch, t_wait);
    if (corpus)
      fprintf(stderr, "; K7 gathered %llu bytes in %llu pieces (%llu packets over pages) in %llu of %zu groups",
              (unsigned long long)gathered_bytes, (unsigned long long)gathered_pieces, (unsigned long long)gathered_multi,
              (unsigned long long)gathered_groups, groups.size());
    fprintf(stderr, "\n");
  }
  for (int s2 = 0; s2 < 2; s2++)
    if (ctx->bulk[s2]) vpz_batch_reset(ctx->bulk[s2]);
  return rc ? rc : total;
}

extern "C" {

int64_t vpz_decode_excerpts(vpz_ctx* ctx, uint32_t n_files, const uint8_t* const* datas, const size_t* lens, uint32_t n,
                            const uint32_t* file_of, const int64_t* start, const int32_t* count, int clip, float* dst,
                            size_t dst_floats, int64_t* dst_offsets, int32_t* got) {
  if (!ctx || !datas || !lens || (n && (!file_of || !start || !count))) return VPZ_E_ARGUMENT;
  VPZ_USE(ctx);
  return decode_excerpts_impl(ctx, n_files, datas, lens, n, file_of, start, count, clip, dst, dst_floats, dst_offsets,
                              got, nullptr);
}

int64_t vpz_decode_excerpts_device(vpz_ctx* ctx, uint32_t n_files, const uint8_t* const* datas, const size_t* lens,
                                   uint32_t n, const uint32_t* file_of, const int64_t* start, const int32_t* count,
                                   int clip, int format, void* dst_dev, size_t dst_elems, int64_t* dst_offsets,
                                   int32_t* got, void* stream) {
  if (!ctx || !datas || !lens || (n && (!file_of || !start || !count))) return VPZ_E_ARGUMENT;
  VPZ_USE(ctx);
  DevOut o;
  o.p = dst_dev;
  o.format = format;
  o.stream = stream;
  dev::Event* ev = nullptr;
  int rc = device_output_begin(ctx, o, &ev);
  if (rc) return device_output_end(ctx, ev, rc);
  return device_output_end(ctx, ev, decode_excerpts_impl(ctx, n_files, datas, lens, n, file_of, start, count, clip,
                                                         static_cast<float*>(dst_dev), dst_elems, dst_offsets, got, &o));
}

int64_t vpz_decode_excerpts_device_conv(vpz_ctx* ctx, uint32_t n_files, const uint8_t* const* datas, const size_t* lens,
                                        uint32_t n, const uint32_t* file_of, const int64_t* start, const int32_t* count,
                                        int clip, const vpz_out_conv* conv, void* dst_dev, size_t dst_elems,
                                        int64_t* dst_offsets, int32_t* got, void* stream) {
  if (!ctx || !datas || !lens || (n && (!file_of || !start || !count))) return VPZ_E_ARGUMENT;
  VPZ_USE(ctx);
  int rc = conv_check(ctx, conv);
  if (rc) return rc;
  DevOut o;
  o.p = dst_dev;
  o.format = conv->format;
  o.stream = stream;
  o.conv = conv;
  dev::Event* ev = nullptr;
  rc = device_output_begin(ctx, o, &ev);
  if (rc) return device_output_end(ctx, ev, rc);
  return device_output_end(ctx, ev, decode_excerpts_impl(ctx, n_files, datas, lens, n, file_of, start, count, clip,
                                                         static_cast<float*>(dst_dev), dst_elems, dst_offsets, got, &o));
}

}  // extern "C"

extern "C" {

int vpz_corpus_open(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens, int copy,
                    vpz_corpus** out) {
  if (!ctx || !out || (n && (!datas || !lens))) return VPZ_E_ARGUMENT;
  *out = nullptr;
  VPZ_USE(ctx);
  if (!ctx->pool) {
    unsigned t = ctx->host_threads > 0 ? (unsigned)ctx->host_threads
                                       : std::max(1u, std::min(std::thread::hardware_concurrency(), 32u));
    ctx->pool = new (std::nothrow) ThreadPool(t);
    if (!ctx->pool) return VPZ_E_NOMEM;
  }
  std::unique_ptr<vpz_corpus> c(new (std::nothrow) vpz_corpus);
  if (!c) return VPZ_E_NOMEM;
  c->ctx = ctx;
  std::vector<const uint8_t*> ptrs(datas, datas + n);
  if (copy) {
    c->copies.resize(n);
    for (uint32_t i = 0; i < n; i++) {
      c->copies[i].assign(datas[i], datas[i] + lens[i]);
      ptrs[i] = c->copies[i].data();
    }
  }
  // the device images: 16-byte aligned, at least 16 zero bytes behind each (K7 reads whole aligned words)
  c->dev_off.resize(n);
  for (uint32_t i = 0; i < n; i++) {
    c->dev_off[i] = c->d_bytes;
    c->d_bytes += ((uint64_t)lens[i] + 16 + 15) & ~(uint64_t)15;
  }
  int rc = VPZ_OK;
  if (c->d_bytes) {
    c->d_img = static_cast<uint8_t*>(dev::alloc(c->d_bytes, ctx->last_error));
    if (!c->d_img) return VPZ_E_CUDA;
    if ((rc = dev::fill(c->d_img, 0, c->d_bytes, ctx->stream, ctx->last_error))) return rc;
  }
  // slices of at most "bulk_group_mib" of images: the scan's pinned staging never holds the whole corpus; each
  // slice's images go from the scan's device copy (or, after a host scan, from the host images) into the corpus buffer
  const uint64_t cap = ctx->bulk_group_bytes > 0 ? (uint64_t)ctx->bulk_group_bytes : (uint64_t)ctx->bulk_group_mib << 20;
  c->files.resize(n);
  for (uint32_t i0 = 0; i0 < n;) {
    uint32_t i1 = i0;
    uint64_t bytes = 0;
    while (i1 < n && (i1 == i0 || bytes + lens[i1] <= cap)) bytes += lens[i1++];
    std::vector<std::unique_ptr<ExcerptFile>> part(i1 - i0);
    ScanResult sr;
    if ((rc = open_excerpt_files(ctx, i1 - i0, ptrs.data() + i0, lens + i0, part, nullptr, &sr))) break;
    for (uint32_t k = i0; k < i1; k++) {   // from the scan's staged images when the device scanned them
      c->files[k] = std::move(part[k - i0]);
      rc = sr.images ? dev::d2d(c->d_img + c->dev_off[k], sr.images + sr.files[k - i0].data_off, lens[k], ctx->stream,
                                ctx->last_error)
                     : dev::h2d(c->d_img + c->dev_off[k], ptrs[k], lens[k], ctx->stream, ctx->last_error);
      if (rc) break;
    }
    // the copies read the scan's staged images, which the next slice's scan (on the scan stream) overwrites
    if (rc || (rc = dev::stream_sync(ctx->stream, ctx->last_error))) break;
    i0 = i1;
  }
  const std::string err = ctx->last_error;
  const int src = dev::stream_sync(ctx->stream, ctx->last_error);   // the caller's bytes may go once open returns
  if (rc) {
    ctx->last_error = err;
    return rc;
  }
  if (src) return src;
  c->samples.resize(n);
  for (uint32_t i = 0; i < n; i++) {
    int err = 0;
    c->samples[i] = c->files[i]->master.ls->total_granules(&err);   // cached by the open
    if (err) return err;
  }
  *out = c.release();
  return VPZ_OK;
}

void vpz_corpus_close(vpz_corpus* c) { delete c; }

uint64_t vpz_corpus_device_bytes(const vpz_corpus* c) { return c ? c->d_bytes : 0; }

int64_t vpz_corpus_info(const vpz_corpus* c, int32_t* channels, int32_t* sample_rate, int64_t* samples) {
  if (!c) return VPZ_E_ARGUMENT;
  for (size_t i = 0; i < c->files.size(); i++) {
    const StreamDec& m = c->files[i]->master;
    if (channels) channels[i] = m.channels();
    if (sample_rate) sample_rate[i] = m.setup->host.id.sample_rate;
    if (samples) samples[i] = c->samples[i];
  }
  return (int64_t)c->files.size();
}

int64_t vpz_corpus_excerpts_device(vpz_corpus* c, uint32_t n, const uint32_t* file_of, const int64_t* start,
                                   const int32_t* count, int clip, const vpz_out_conv* conv, void* dst_dev,
                                   size_t dst_elems, int64_t* dst_offsets, int32_t* got, void* stream) {
  if (!c || (n && (!file_of || !start || !count))) return VPZ_E_ARGUMENT;
  vpz_ctx* ctx = c->ctx;
  VPZ_USE(ctx);
  int rc = conv_check(ctx, conv);
  if (rc) return rc;
  DevOut o;
  o.p = dst_dev;
  o.format = conv->format;
  o.stream = stream;
  o.conv = conv;
  dev::Event* ev = nullptr;
  rc = device_output_begin(ctx, o, &ev);
  if (rc) return device_output_end(ctx, ev, rc);
  return device_output_end(ctx, ev, decode_excerpts_impl(ctx, (uint32_t)c->files.size(), nullptr, nullptr, n, file_of,
                                                         start, count, clip, static_cast<float*>(dst_dev), dst_elems,
                                                         dst_offsets, got, &o, c));
}

// Debug / tests: the page-end granule index of one container image (first logical stream), built on the device
// (K0 + K0g; VPZ_E_UNSUPPORTED when the file does not qualify) or by the host's packet walk.  Returns the number
// of pages, writes min(pages, cap) entries.
int64_t vpz_debug_page_end_granules(vpz_ctx* ctx, const uint8_t* data, size_t len, int on_device, int64_t* out, size_t cap) {
  if (!ctx || !data) return VPZ_E_ARGUMENT;
  VPZ_USE(ctx);
  if (!ctx->pool) {
    ctx->pool = new (std::nothrow) ThreadPool(ctx->host_threads > 0 ? (unsigned)ctx->host_threads
                                                                    : std::max(1u, std::min(std::thread::hardware_concurrency(), 32u)));
    if (!ctx->pool) return VPZ_E_NOMEM;
  }
  std::vector<std::unique_ptr<ExcerptFile>> files(1);
  const int saved = ctx->gpu_scan;
  ctx->gpu_scan = on_device ? 1 : 0;
  uint32_t on_dev = 0;
  int rc = open_excerpt_files(ctx, 1, &data, &len, files, &on_dev);
  ctx->gpu_scan = saved;
  if (rc) return rc;
  if (on_device && !on_dev) {
    ctx->last_error = "file does not qualify for the device seek index";
    return VPZ_E_UNSUPPORTED;
  }
  const std::vector<int64_t>& v = files[0]->master.ls->page_end_granules;
  for (size_t i = 0; i < v.size() && i < cap; i++) out[i] = v[i];
  return (int64_t)v.size();
}

}  // extern "C"

#ifdef VPZ_EMU
// The emulated CPU test build (tests/emu, never linked into libvpz.so) takes the K5, K6 and K7 launchers and the
// caller-memory hooks of the device-output and corpus calls above from here.
#include "../../tests/emu/dev_emu_place.h"
#include "../../tests/emu/dev_emu_convert.h"
#include "../../tests/emu/dev_emu_corpus.h"
#endif
