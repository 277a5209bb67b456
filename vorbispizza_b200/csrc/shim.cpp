// shim.cpp -- extern "C" entry points of include/vpz.h for the context, setup, batch, debug and
// synthetic-spectrum layers.  (The reader layer lives in reader.cpp.)
#include <string.h>

#include <algorithm>
#include <new>

#include "../../include/vpz.h"
#include "engine.h"

using namespace vpz;

extern "C" {

const char* vpz_strerror(int code) {
  switch (code) {
    case VPZ_OK: return "ok";
    case VPZ_E_INVALID_DATA: return "invalid data";
    case VPZ_E_ARGUMENT: return "bad argument";
    case VPZ_E_SEEK_RANGE: return "seek out of range";
    case VPZ_E_PREROLL: return "could not read pre-roll packet";
    case VPZ_E_UNSUPPORTED: return "stream feature not supported by the GPU path";
    case VPZ_E_CUDA: return "CUDA error";
    case VPZ_E_NOMEM: return "out of memory";
    case VPZ_E_DISPOSED: return "object disposed";
    case VPZ_E_INVALID_OP: return "invalid operation";
    case VPZ_E_NO_DEVICE: return "no sm_100 device (no CPU fallback)";
    case VPZ_E_REF_FAULT: return "the reference decoder faults on this input";
    default: return "unknown error";
  }
}

const char* vpz_last_error(const vpz_ctx* ctx) { return ctx ? ctx->last_error.c_str() : ""; }

const char* vpz_version(void) {
#ifdef VPZ_EMU
  return "vpz 0.1 EMULATED (tests only)";
#else
  return "vpz 0.1 sm_100a";
#endif
}

int vpz_device_count(void) { return dev::device_count(); }

int vpz_ctx_create(int device, vpz_ctx** out) {
  if (!out) return VPZ_E_ARGUMENT;
  *out = nullptr;
  std::string err;
  int resolved = device;
  int rc = dev::init(device, &resolved, err);
  if (rc) return rc;
  vpz_ctx* c = new (std::nothrow) vpz_ctx;
  if (!c) return VPZ_E_NOMEM;
  c->device = resolved;
  c->stream = dev::stream_create();
  c->copy_stream = dev::stream_create();
  for (int i = 0; i < 4; i++) c->ev[i] = dev::event_create();
  c->d_counter = static_cast<uint32_t*>(dev::alloc(64, c->last_error));
  if (!c->stream || !c->copy_stream || !c->ev[0] || !c->ev[1] || !c->ev[2] || !c->ev[3] || !c->d_counter) {
    vpz_ctx_destroy(c);
    return VPZ_E_CUDA;
  }
  *out = c;
  return VPZ_OK;
}

void vpz_ctx_destroy(vpz_ctx* c) {
  if (!c) return;
  VPZ_USE(c);
  for (int i = 0; i < 3; i++) {
    if (c->bulk[i]) vpz_batch_destroy(c->bulk[i]);
    c->bulk[i] = nullptr;
    dev::event_destroy(c->bulk_done[i]);
    dev::event_destroy(c->bulk_ready[i]);
  }
  delete c->xb;
  delete c->place;
  delete c->pool;
  c->pool = nullptr;
  scan_bufs_destroy(c->scan);
  c->scan = nullptr;
  for (int i = 0; i < 8; i++) dev::event_destroy(c->marks[i]);
  while (!c->setups.empty()) {
    vpz_setup* s = c->setups.begin()->second;
    s->refs = 1;
    setup_release(s);
  }
  dev::free(c->d_counter);
  for (int i = 0; i < 4; i++) dev::event_destroy(c->ev[i]);
  dev::stream_destroy(c->stream);
  dev::stream_destroy(c->copy_stream);
  delete c;
}

int vpz_ctx_mark(vpz_ctx* c, int slot) {
  if (!c || slot < 0 || slot >= 8) return VPZ_E_ARGUMENT;
  VPZ_USE(c);
  if (!c->marks[slot]) c->marks[slot] = dev::event_create();
  if (!c->marks[slot]) return VPZ_E_CUDA;
  dev::event_record(c->marks[slot], c->stream);
  return VPZ_OK;
}

float vpz_ctx_elapsed_ms(vpz_ctx* c, int a, int b) {
  if (!c || a < 0 || a >= 8 || b < 0 || b >= 8 || !c->marks[a] || !c->marks[b]) return -1.f;
  VPZ_USE(c);
  if (dev::event_sync(c->marks[b], c->last_error)) return -1.f;
  return dev::event_elapsed_ms(c->marks[a], c->marks[b]);
}

int64_t vpz_ctx_kernel_launches(const vpz_ctx* c) { return c ? c->kernel_launches : VPZ_E_ARGUMENT; }

int vpz_ctx_set(vpz_ctx* c, const char* key, int value) {
  if (!c || !key) return VPZ_E_ARGUMENT;
  if (!strcmp(key, "l1_bits")) {
    if (value < 1 || value > 12) return VPZ_E_ARGUMENT;
    c->l1_bits = value;
  } else if (!strcmp(key, "ola_chunk")) {
    if (value < 1 || value > 65536) return VPZ_E_ARGUMENT;
    c->ola_chunk = value;
    c->ola_chunk_set = true;
  } else if (!strcmp(key, "k1a_smem")) {
    if (value < 0 || value > 1) return VPZ_E_ARGUMENT;
    c->k1a_smem = value;
  } else if (!strcmp(key, "k1_warps")) {
    if (value < 1 || value > 8) return VPZ_E_ARGUMENT;
    c->k1_warps = value;
  } else if (!strcmp(key, "bulk_group")) {
    if (value < 1 || value > (1 << 20)) return VPZ_E_ARGUMENT;
    c->bulk_group = value;
  } else if (!strcmp(key, "bulk_group_mib")) {
    // a batch addresses its entry-index area (~8x the compressed bytes) and its spectra (~11 floats per compressed
    // byte) with 32 bits: 384 MiB of images is the most one group can hold
    if (value < 1 || value > 384) return VPZ_E_ARGUMENT;
    c->bulk_group_mib = value;
  } else if (!strcmp(key, "bulk_group_bytes")) {
    if (value < 0) return VPZ_E_ARGUMENT;
    c->bulk_group_bytes = value;
  } else if (!strcmp(key, "force_general")) {
    // test knob: 1 routes every packet through the general spectrum kernel and the generic IMDCT kernel,
    // 2 also through the full symbol kernel (floor 0 / multi-submap walk); 0 = per-setup choice
    if (value < 0 || value > 2) return VPZ_E_ARGUMENT;
    c->force_general = value;
  } else if (!strcmp(key, "gpu_scan")) {
    if (value < 0 || value > 2) return VPZ_E_ARGUMENT;   // 2: single readers too (tests)
    c->gpu_scan = value;
  } else if (!strcmp(key, "bulk_threads")) {
    if (value < 0 || value > 256) return VPZ_E_ARGUMENT;
    c->bulk_threads = value;
  } else if (!strcmp(key, "bulk_threads_device")) {
    if (value < 0 || value > 256) return VPZ_E_ARGUMENT;
    c->bulk_threads_device = value;
  } else if (!strcmp(key, "host_threads")) {
    if (value < 0 || value > 256 || c->pool) return VPZ_E_ARGUMENT;  // before the first bulk call
    c->host_threads = value;
  } else {
    return VPZ_E_ARGUMENT;
  }
  return VPZ_OK;
}

int vpz_setup_create(vpz_ctx* ctx, const uint8_t* id_pkt, size_t id_len, const uint8_t* setup_pkt, size_t setup_len,
                     vpz_setup** out) {
  if (!ctx || !id_pkt || !setup_pkt || !out) return VPZ_E_ARGUMENT;
  VPZ_USE(ctx);
  return setup_create(ctx, id_pkt, id_len, setup_pkt, setup_len, out);
}
void vpz_setup_release(vpz_setup* s) {
  if (!s) return;
  VPZ_USE(s->ctx);
  setup_release(s);
}

int vpz_setup_get_info(const vpz_setup* s, vpz_setup_info* info) {
  if (!s || !info) return VPZ_E_ARGUMENT;
  const VpzSetupHdr* h = s->host.hdr();
  memset(info, 0, sizeof(*info));
  info->channels = s->host.id.channels;
  info->sample_rate = s->host.id.sample_rate;
  info->bitrate_upper = s->host.id.br_upper;
  info->bitrate_nominal = s->host.id.br_nominal;
  info->bitrate_lower = s->host.id.br_lower;
  info->block_size0 = s->host.id.size0;
  info->block_size1 = s->host.id.size1;
  info->n_books = (int32_t)h->nbooks;
  info->n_floors = h->nfloors;
  info->n_residues = s->host.n_residues_hdr;
  info->n_mappings = h->nmappings;
  info->n_modes = h->nmodes;
  info->max_codeword_bits = s->host.max_codeword_bits;
  info->table_bytes = (uint64_t)s->host.blob.size() * 4;
  return VPZ_OK;
}

int vpz_packet_info(const vpz_setup* s, const uint8_t* pkt, size_t len, int32_t info[6]) {
  if (!s || !info || (!pkt && len)) return VPZ_E_ARGUMENT;
  PacketGeom g = s->host.packet_geometry(pkt, len);
  if (g.bad_mode) return VPZ_E_INVALID_DATA;
  if (!g.valid) {
    memset(info, 0, 6 * sizeof(int32_t));
    return 0;
  }
  info[0] = g.length;
  info[1] = g.left_use_size1 ? 1 : 0;
  info[2] = g.left_start;
  info[3] = g.left_end;
  info[4] = g.right_start;
  info[5] = g.right_end;
  return 1;
}

// ---- batch ----------------------------------------------------------------------------------
int vpz_batch_create(vpz_ctx* ctx, vpz_batch** out) {
  if (!ctx || !out) return VPZ_E_ARGUMENT;
  vpz_batch* b = new (std::nothrow) vpz_batch;
  if (!b) return VPZ_E_NOMEM;
  b->ctx = ctx;
  *out = b;
  return VPZ_OK;
}
void vpz_batch_destroy(vpz_batch* b) {
  if (!b) return;
  VPZ_USE(b->ctx);
  batch_drop_slots(b);
  if (b->owned_setup) setup_release(b->owned_setup);
  delete b;
}

int vpz_batch_reset(vpz_batch* b) {
  if (!b) return VPZ_E_ARGUMENT;
  if (b->synthetic) return VPZ_E_INVALID_OP;
  b->bytes.clear();
  b->pkts_in.clear();
  b->pkts_ola.clear();
  b->items.clear();
  b->runs.clear();
  VPZ_USE(b->ctx);
  batch_drop_slots(b);
  b->total_floats = b->spec_floats = b->payload_bytes = 0;
  b->rec_words = b->ent_total = 0;
  b->max_channels = 1;
  b->uploaded = b->decoded = false;
  b->gather_images = nullptr;
  b->gather_bytes = 0;
  b->gather_fill = nullptr;
  b->pieces.clear();
  return VPZ_OK;
}

int vpz_batch_add_run(vpz_batch* b, vpz_setup* s, const uint8_t* bytes, const uint32_t* offsets, uint32_t n_pkts,
                      const int32_t* trim) {
  if (!b || !s || !offsets || (!bytes && n_pkts && offsets[n_pkts] != offsets[0])) return VPZ_E_ARGUMENT;
  return batch_add_run(b, s, bytes, offsets, n_pkts, trim);
}

int64_t vpz_batch_run_samples(const vpz_batch* b, int run) {
  if (!b || run < 0 || (size_t)run >= b->runs.size()) return VPZ_E_ARGUMENT;
  return b->runs[run].samples;
}
int vpz_batch_run_channels(const vpz_batch* b, int run) {
  if (!b || run < 0 || (size_t)run >= b->runs.size()) return VPZ_E_ARGUMENT;
  return b->runs[run].setup->host.id.channels;
}
int vpz_batch_run_status(const vpz_batch* b, int run, int32_t* stop_packet) {
  if (!b || run < 0 || (size_t)run >= b->runs.size()) return VPZ_E_ARGUMENT;
  if (stop_packet) *stop_packet = b->runs[run].stop_packet;
  return b->runs[run].status;
}
int vpz_batch_run_packet_samples(const vpz_batch* b, int run, int32_t* counts) {
  if (!b || !counts || run < 0 || (size_t)run >= b->runs.size()) return VPZ_E_ARGUMENT;
  const Run& r = b->runs[run];
  memcpy(counts, r.counts.data(), r.counts.size() * sizeof(int32_t));
  return (int)r.counts.size();
}
int64_t vpz_batch_total_floats(const vpz_batch* b) { return b ? (int64_t)b->total_floats : VPZ_E_ARGUMENT; }
int64_t vpz_batch_total_packets(const vpz_batch* b) { return b ? (int64_t)b->pkts_ola.n : VPZ_E_ARGUMENT; }
int64_t vpz_batch_total_bytes(const vpz_batch* b) { return b ? (int64_t)b->payload_bytes : VPZ_E_ARGUMENT; }

int vpz_batch_upload(vpz_batch* b) {
  if (!b) return VPZ_E_ARGUMENT;
  VPZ_USE(b->ctx);
  return batch_upload(b);
}
int vpz_batch_decode(vpz_batch* b, int clip) {
  if (!b) return VPZ_E_ARGUMENT;
  VPZ_USE(b->ctx);
  return batch_decode(b, clip);
}
int vpz_batch_sync(vpz_batch* b) {
  if (!b) return VPZ_E_ARGUMENT;
  VPZ_USE(b->ctx);
  int rc = dev::stream_sync(b->ctx->stream, b->ctx->last_error);
  if (rc) return rc;
  if (b->decoded) {
    b->ms_k1a = dev::event_elapsed_ms(b->ctx->ev[0], b->ctx->ev[1]);
    b->ms_k1b = dev::event_elapsed_ms(b->ctx->ev[1], b->ctx->ev[2]);
    b->ms_k1 = dev::event_elapsed_ms(b->ctx->ev[0], b->ctx->ev[2]);
    b->ms_k3 = dev::event_elapsed_ms(b->ctx->ev[2], b->ctx->ev[3]);
    b->ms_total = dev::event_elapsed_ms(b->ctx->ev[0], b->ctx->ev[3]);
  }
  return VPZ_OK;
}

int vpz_batch_has_clipped(vpz_batch* b) {
  if (!b || !b->decoded) return VPZ_E_INVALID_OP;
  VPZ_USE(b->ctx);
  int rc = batch_fetch_clip(b);
  if (rc) return rc;
  for (size_t i = 0; i < b->h_clip.n; i++)
    if (b->h_clip.p[i] != 0xffffffffu) return 1;
  return 0;
}

int64_t vpz_batch_run_offset(const vpz_batch* b, int run) {
  if (!b || run < 0 || (size_t)run >= b->runs.size()) return VPZ_E_ARGUMENT;
  return (int64_t)b->runs[run].out_base;
}
const float* vpz_batch_device_pcm(const vpz_batch* b) { return b ? static_cast<const float*>(b->d_pcm.p) : nullptr; }

int vpz_batch_read_run(vpz_batch* b, int run, float* dst) {
  if (!b || !dst || run < 0 || (size_t)run >= b->runs.size()) return VPZ_E_ARGUMENT;
  if (!b->decoded) return VPZ_E_INVALID_OP;
  VPZ_USE(b->ctx);
  const Run& r = b->runs[run];
  size_t n = (size_t)r.samples * r.setup->host.id.channels;
  int rc = dev::d2h(dst, static_cast<const float*>(b->d_pcm.p) + r.out_base, n * 4, b->ctx->stream, b->ctx->last_error);
  if (rc) return rc;
  return dev::stream_sync(b->ctx->stream, b->ctx->last_error);
}

int vpz_batch_read_all(vpz_batch* b, float* dst) {
  if (!b || !dst) return VPZ_E_ARGUMENT;
  if (!b->decoded) return VPZ_E_INVALID_OP;
  VPZ_USE(b->ctx);
  int rc = dev::d2h(dst, b->d_pcm.p, b->total_floats * 4, b->ctx->stream, b->ctx->last_error);
  if (rc) return rc;
  return dev::stream_sync(b->ctx->stream, b->ctx->last_error);
}

float vpz_batch_last_ms(vpz_batch* b, int which, int* launches) {
  if (!b) return -1.f;
  if (launches) *launches = b->launches;
  return which == 1 ? b->ms_k1 : which == 3 ? b->ms_k3 : which == 11 ? b->ms_k1a : which == 12 ? b->ms_k1b : b->ms_total;
}

uint64_t vpz_transfer_bytes(int which) { return dev::transfer_bytes(which); }

void* vpz_host_alloc(size_t bytes) { return dev::host_alloc(bytes); }
void vpz_host_free(void* p) { dev::host_free(p); }

// ---- single packet with stage dumps ---------------------------------------------------------
int vpz_debug_decode_packet(vpz_ctx* ctx, vpz_setup* s, const uint8_t* pkt, size_t len, vpz_packet_dump* dump,
                            int32_t* scalars, int32_t scalars_cap, int32_t* classes, int32_t classes_cap,
                            float* residue, float* spectrum, float* imdct) {
  if (!ctx || !s || !dump || (!pkt && len)) return VPZ_E_ARGUMENT;
  VPZ_USE(ctx);
  memset(dump, 0, sizeof(*dump));
  dump->status = 1;
  PacketGeom g = s->host.packet_geometry(pkt, len);
  if (g.bad_mode) return VPZ_E_INVALID_DATA;
  if (!g.valid) return VPZ_OK;
  const int C = s->host.id.channels, N = g.block_size, M = N / 2;
  std::string& err = ctx->last_error;
  vpz_batch* b = nullptr;
  int rc = vpz_batch_create(ctx, &b);
  if (rc) return rc;
  uint32_t offs[2] = {0, (uint32_t)len};
  rc = batch_add_run(b, s, pkt, offs, 1, nullptr);
  if (rc < 0) {
    vpz_batch_destroy(b);
    return rc;
  }
  // one K3 item so the raw transform output can be dumped (no previous packet: nothing is emitted)
  VpzOlaItem it;
  memset(&it, 0, sizeof(it));
  it.first_pkt = 0;
  it.n_pkts = 1;
  it.has_pre = 0;
  it.setup_slot = 0;
  b->items.push(it);
  DevBuf d_hdr, d_scal, d_cls, d_res, d_imdct;
  const size_t hdr_words = sizeof(vpz_packet_dump) / 4;
  scalars_cap = scalars ? std::max(scalars_cap, 0) : 0;
  classes_cap = classes ? std::max(classes_cap, 0) : 0;
  if (!d_hdr.reserve(hdr_words * 4, err) || !d_scal.reserve((size_t)scalars_cap * 4 + 4, err) ||
      !d_cls.reserve((size_t)classes_cap * 4 + 4, err) || !d_res.reserve((size_t)C * M * 4, err) ||
      !d_imdct.reserve((size_t)C * N * 4, err)) {
    vpz_batch_destroy(b);
    return VPZ_E_CUDA;
  }
  dev::fill(d_hdr.p, 0, hdr_words * 4, ctx->stream, err);
  dev::fill(d_imdct.p, 0, (size_t)C * N * 4, ctx->stream, err);
  b->dbg.hdr = static_cast<int32_t*>(d_hdr.p);
  b->dbg.scalars = scalars_cap ? static_cast<int32_t*>(d_scal.p) : nullptr;
  b->dbg.scalars_cap = scalars_cap;
  b->dbg.classes = classes_cap ? static_cast<int32_t*>(d_cls.p) : nullptr;
  b->dbg.classes_cap = classes_cap;
  b->dbg.residue = static_cast<float*>(d_res.p);
  b->dbg_imdct = static_cast<float*>(d_imdct.p);
  rc = batch_decode(b, 0);
  if (!rc) rc = dev::stream_sync(ctx->stream, err);
  if (!rc) rc = dev::d2h(dump, d_hdr.p, sizeof(*dump), ctx->stream, err);
  if (!rc && scalars_cap) rc = dev::d2h(scalars, d_scal.p, (size_t)scalars_cap * 4, ctx->stream, err);
  if (!rc && classes_cap) rc = dev::d2h(classes, d_cls.p, (size_t)classes_cap * 4, ctx->stream, err);
  if (!rc && residue) rc = dev::d2h(residue, d_res.p, (size_t)C * M * 4, ctx->stream, err);
  if (!rc && imdct) rc = dev::d2h(imdct, d_imdct.p, (size_t)C * N * 4, ctx->stream, err);
  std::vector<float> spec_host;
  std::vector<VpzPktRes> res_host(1);
  if (!rc) rc = dev::d2h(res_host.data(), b->d_res.p, sizeof(VpzPktRes), ctx->stream, err);
  if (!rc && spectrum) {
    spec_host.resize((size_t)C * M);
    rc = dev::d2h(spec_host.data(), b->d_spec.p, (size_t)C * M * 4, ctx->stream, err);
  }
  if (!rc) rc = dev::stream_sync(ctx->stream, err);
  if (!rc) {
    dump->info[0] = g.length;
    dump->info[1] = g.left_use_size1 ? 1 : 0;
    dump->info[2] = g.left_start;
    dump->info[3] = g.left_end;
    dump->info[4] = g.right_start;
    dump->info[5] = g.right_end;
    if (spectrum) {
      // channels without floor energy never get a spectrum written (K3 treats them as zero)
      for (int c = 0; c < C; c++) {
        bool on = (res_host[0].exec_mask >> c) & 1;
        for (int i = 0; i < M; i++) spectrum[(size_t)c * M + i] = on ? spec_host[(size_t)c * M + i] : 0.f;
      }
    }
  }
  vpz_batch_destroy(b);
  return rc;
}

// ---- kernel-only IMDCT + window + OLA on caller spectra (BASELINE config 3) ----------------------
int vpz_synth_create(vpz_ctx* ctx, int channels, int log2_size0, int log2_size1, uint32_t n_streams,
                     uint32_t n_blocks, const uint8_t* flags, const float* spectra, vpz_batch** out) {
  if (!ctx || !flags || !spectra || !out || n_blocks < 2 || n_streams < 1) return VPZ_E_ARGUMENT;
  VPZ_USE(ctx);
  vpz_setup* s = nullptr;
  int rc = setup_create_synthetic(ctx, channels, log2_size0, log2_size1, &s);
  if (rc) return rc;
  vpz_batch* b = nullptr;
  rc = vpz_batch_create(ctx, &b);
  if (rc) {
    setup_release(s);
    return rc;
  }
  b->synthetic = true;
  b->owned_setup = s;  // released by vpz_batch_destroy
  b->slots.push_back(s);
  b->max_channels = channels;
  const int size0 = 1 << log2_size0, size1 = 1 << log2_size1;
  const uint32_t chunk = pick_ola_chunk(ctx, (uint64_t)n_streams * n_blocks);
  for (uint32_t st = 0; st < n_streams; st++) {
    Run run;
    run.setup = s;
    run.slot = 0;
    run.first_valid = (uint32_t)b->pkts_ola.n;
    run.out_base = b->total_floats;
    run.counts.assign(n_blocks, 0);
    int64_t pos = 0;
    int prev_rs = 0, prev_re = 0;
    for (uint32_t i = 0; i < n_blocks; i++) {
      const uint8_t* f = flags + (size_t)st * n_blocks;
      bool lb = f[i] & 1;
      bool prev = i == 0 ? true : (f[i - 1] & 1);
      bool next = i + 1 == n_blocks ? true : (f[i + 1] & 1);
      PacketGeom g;
      compute_geometry(size0, size1, lb, prev, next, &g);
      int count = 0;
      if (i > 0) {
        if (prev_re - prev_rs != g.length) {
          ctx->last_error = "inconsistent window flags";
          vpz_batch_destroy(b);
          return VPZ_E_ARGUMENT;
        }
        count = g.right_start - g.left_start;
      }
      VpzPktOla ola;
      memset(&ola, 0, sizeof(ola));
      if (b->spec_floats + (uint64_t)channels * g.block_size / 2 > 0xffffff00ull) {
        ctx->last_error = "synthetic batch exceeds 2^32 spectrum floats";
        vpz_batch_destroy(b);
        return VPZ_E_ARGUMENT;
      }
      ola.spec_off = (uint32_t)b->spec_floats;
      ola.out_off = (uint32_t)pos;
      ola.left_start = (uint16_t)g.left_start;
      ola.right_start = (uint16_t)g.right_start;
      ola.right_end = (uint16_t)g.right_end;
      ola.flags = (uint8_t)((lb ? VPZ_OLA_LONG : 0) | (g.left_use_size1 ? VPZ_OLA_LEFT1 : 0) | (i ? 0 : VPZ_OLA_NOOUT));
      b->pkts_ola.push(ola);
      b->spec_floats += (uint64_t)channels * g.block_size / 2;
      run.counts[i] = count;
      pos += count;
      prev_rs = g.right_start;
      prev_re = g.right_end;
    }
    run.n_valid = n_blocks;
    run.samples = pos;
    b->total_floats += (uint64_t)pos * channels;
    for (uint32_t k = 1; k < n_blocks; k += chunk) {
      VpzOlaItem it;
      it.first_pkt = run.first_valid + k;
      it.n_pkts = std::min(chunk, n_blocks - k);
      it.has_pre = 1;
      it.setup_slot = 0;
      it.out_base = run.out_base;
      b->items.push(it);
    }
    b->runs.push_back(std::move(run));
  }
  std::string& err = ctx->last_error;
  if (!b->d_spec.reserve(b->spec_floats * 4, err)) rc = VPZ_E_CUDA;
  if (!rc) rc = dev::h2d(b->d_spec.p, spectra, b->spec_floats * 4, ctx->stream, err);
  if (!rc) rc = batch_upload(b);
  if (rc) {
    vpz_batch_destroy(b);
    return rc;
  }
  *out = b;
  return VPZ_OK;
}

}  // extern "C"
