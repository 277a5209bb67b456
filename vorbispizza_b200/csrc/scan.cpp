// scan.cpp -- host side of K0 (k0_pages.cuh): stages container images, runs the page scan on the device and
// brings the page records back.  The physical Ogg layer (capture-pattern search, header parse, lacing sums,
// page CRC -- Ogg/PageReaderBase.cs:41-84,286-361, Ogg/Crc.cs:20-63) is the data-parallel part of container
// parsing; the per-serial bookkeeping stays on the host (ogg.cpp, OggContainer::scan_from_records).
#include <string.h>

#include <algorithm>
#include <new>

#include "../../include/vpz.h"
#include "engine.h"

namespace vpz {

struct ScanSlot {
  HostBuf<uint8_t> h_img;
  HostBuf<VpzScanFile> h_files;
  // The kernel writes its records STRAIGHT into these pinned (mapped) host arrays: a page record is two
  // 16-byte posted writes over the link.  No device->host copy is queued, so a scan never waits behind the
  // bulk pipeline's PCM copies on the copy engine (measured: 8 ms per group when it did).
  HostBuf<VpzPageRec> h_pages;
  HostBuf<VpzScanOut> h_out;
  DevBuf d_img, d_files, d_jobs, d_irregular;   // + CRC jobs and per-file flags of the fast path (k0_walk / k0_crc)
  // K0g (granule_index): per-file parameters in, the page-end granule index out (pinned + mapped like h_pages)
  HostBuf<VpzGranFile> h_gfiles;
  DevBuf d_gfiles;
  HostBuf<long long> h_page_end;
  dev::Event* done = nullptr;
  uint32_t* d_counter = nullptr;
  uint32_t n = 0;
  bool in_flight = false;
};

struct ScanBufs {
  ScanSlot slot[2];                  // two scans may be in flight: the bulk path scans group g+1 while it plans g
  dev::Stream* stream = nullptr;
  ~ScanBufs() {
    for (ScanSlot& s : slot) {
      if (s.in_flight && s.done) {
        std::string e;
        dev::event_sync(s.done, e);
      }
      dev::event_destroy(s.done);
      dev::free(s.d_counter);
    }
    dev::stream_destroy(stream);
  }
};

void scan_bufs_destroy(ScanBufs* s) { delete s; }

// Pages a file of `len` bytes may produce before the device gives up on it (the host then scans that file
// itself): a page is at least 27 bytes; audio pages carry kilobytes.
static uint32_t page_cap(size_t len) { return (uint32_t)std::min<size_t>(len / 64 + 16, 1u << 24); }

// Starts the scan of n images in slot `which` (0 / 1): stages the images in pinned memory (on `pool`), uploads
// them and launches K0 on the scan stream.  Returns without waiting; scan_end collects.
int scan_begin(vpz_ctx* ctx, int which, uint32_t n, const uint8_t* const* datas, const size_t* lens, ThreadPool* pool) {
  std::string& err = ctx->last_error;
  if (!ctx->scan) {
    ctx->scan = new (std::nothrow) ScanBufs;
    if (!ctx->scan) return VPZ_E_NOMEM;
    ctx->scan->stream = dev::stream_create();
    if (!ctx->scan->stream) return VPZ_E_CUDA;
  }
  ScanSlot& b = ctx->scan->slot[which & 1];
  dev::Stream* stream = ctx->scan->stream;
  if (b.in_flight) {   // a scan nobody collected (an error path): its buffers must be quiet before they are reused
    dev::event_sync(b.done, err);
    b.in_flight = false;
  }
  if (!b.done) {
    b.done = dev::event_create();
    b.d_counter = static_cast<uint32_t*>(dev::alloc(64, err));
    if (!b.done || !b.d_counter) return VPZ_E_CUDA;
  }
  b.n = n;
  if (n == 0) return VPZ_OK;
  if (!b.h_files.reserve(n) || !b.h_out.reserve(n)) return VPZ_E_NOMEM;
  uint64_t bytes = 0, pages = 0;
  for (uint32_t i = 0; i < n; i++) {
    if (lens[i] > 0xfffffff0ull) {
      err = "container image larger than 4 GiB";
      return VPZ_E_ARGUMENT;
    }
    VpzScanFile f;
    f.data_off = bytes;
    f.len = (uint32_t)lens[i];
    f.page_base = (uint32_t)pages;
    f.page_cap = page_cap(lens[i]);
    f.pad = 0;
    b.h_files.p[i] = f;
    bytes += (lens[i] + 8 + 15) & ~(uint64_t)15;   // 16-byte aligned images, >= 8 readable bytes behind each
    pages += f.page_cap;
    if (pages > 0xfffffff0ull) {
      err = "too many pages in one scan; split the call";
      return VPZ_E_ARGUMENT;
    }
  }
  b.h_files.n = b.h_out.n = n;
  if (!b.h_img.reserve(bytes) || !b.h_pages.reserve(pages)) return VPZ_E_NOMEM;
  auto stage = [&](size_t i) {
    const VpzScanFile& f = b.h_files.p[i];
    uint8_t* dst = b.h_img.p + f.data_off;
    if (f.len) memcpy(dst, datas[i], f.len);
    const uint64_t end = i + 1 < n ? b.h_files.p[i + 1].data_off : bytes;
    memset(dst + f.len, 0, (size_t)(end - f.data_off - f.len));
  };
  if (pool)
    pool->parallel_for(n, stage);
  else
    for (uint32_t i = 0; i < n; i++) stage(i);
  if (!b.d_img.reserve(bytes, err) || !b.d_files.reserve(n * sizeof(VpzScanFile), err) ||
      !b.d_jobs.reserve(pages * sizeof(VpzCrcJob), err) || !b.d_irregular.reserve((size_t)n * 4, err))
    return VPZ_E_CUDA;
  int rc;
  if ((rc = dev::h2d(b.d_img.p, b.h_img.p, bytes, stream, err))) return rc;
  if ((rc = dev::h2d(b.d_files.p, b.h_files.p, n * sizeof(VpzScanFile), stream, err))) return rc;
  if ((rc = dev::fill(b.d_counter, 0, 16, stream, err))) return rc;
  if ((rc = dev::fill(b.d_irregular.p, 0, (size_t)n * 4, stream, err))) return rc;
  K0Params p;
  p.images = static_cast<const uint8_t*>(b.d_img.p);
  p.files = static_cast<const VpzScanFile*>(b.d_files.p);
  p.pages = b.h_pages.p;   // pinned + mapped: device address == host address (unified addressing)
  p.out = b.h_out.p;
  p.n_files = n;
  p.counter = b.d_counter;
  p.jobs = static_cast<VpzCrcJob*>(b.d_jobs.p);
  p.irregular = static_cast<uint32_t*>(b.d_irregular.p);
  p.only_irregular = 0;
  if ((rc = dev::launch_k0(p, stream, err))) return rc;
  ctx->kernel_launches += 3;
  dev::event_record(b.done, stream);
  b.in_flight = true;
  return VPZ_OK;
}

// Waits for slot `which`.  On return res->files[i] / res->pages hold file i's records (res->out[i].overflow
// set when the file has more pages than page_cap); they stay valid until the slot's next scan_begin.
int scan_end(vpz_ctx* ctx, int which, ScanResult* res) {
  ScanSlot& b = ctx->scan->slot[which & 1];
  res->n = b.n;
  res->files = nullptr;
  res->pages = nullptr;
  res->out = nullptr;
  if (b.in_flight) {
    b.in_flight = false;
    int rc = dev::event_sync(b.done, ctx->last_error);
    if (rc) return rc;
  }
  if (b.n == 0) return VPZ_OK;
  res->files = b.h_files.p;
  res->pages = b.h_pages.p;
  res->out = b.h_out.p;
  res->images = static_cast<const uint8_t*>(b.d_img.p);
  return VPZ_OK;
}

// K0g on the images slot `which` still holds from its last scan: the page-end granule index of the n files described
// by gf (page_base / data_off as in the scan's VpzScanFile records).  *out is indexed like the slot's page records and
// stays valid until the slot's next scan_begin.  Waits for the kernel.
int granule_index(vpz_ctx* ctx, int which, const VpzGranFile* gf, uint32_t n, const long long** out) {
  std::string& err = ctx->last_error;
  if (!ctx->scan) return VPZ_E_INVALID_OP;
  ScanSlot& b = ctx->scan->slot[which & 1];
  dev::Stream* stream = ctx->scan->stream;
  *out = nullptr;
  if (n == 0) return VPZ_OK;
  if (b.in_flight || !b.h_pages.p) return VPZ_E_INVALID_OP;
  if (!b.h_gfiles.reserve(n) || !b.h_page_end.reserve(b.h_pages.cap)) return VPZ_E_NOMEM;
  memcpy(b.h_gfiles.p, gf, n * sizeof(VpzGranFile));
  if (!b.d_gfiles.reserve(n * sizeof(VpzGranFile), err)) return VPZ_E_CUDA;
  int rc;
  if ((rc = dev::h2d(b.d_gfiles.p, b.h_gfiles.p, n * sizeof(VpzGranFile), stream, err))) return rc;
  K0gParams p;
  p.images = static_cast<const uint8_t*>(b.d_img.p);
  p.files = static_cast<const VpzGranFile*>(b.d_gfiles.p);
  p.pages = b.h_pages.p;          // pinned + mapped (the scan wrote them there)
  p.page_end = b.h_page_end.p;
  p.n_files = n;
  if ((rc = dev::launch_k0g(p, stream, err))) return rc;
  ctx->kernel_launches++;
  if ((rc = dev::stream_sync(stream, err))) return rc;
  *out = b.h_page_end.p;
  return VPZ_OK;
}

int scan_pages(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens, ThreadPool* pool,
               ScanResult* res) {
  int rc = scan_begin(ctx, 0, n, datas, lens, pool);
  return rc ? rc : scan_end(ctx, 0, res);
}

}  // namespace vpz

using namespace vpz;

extern "C" int64_t vpz_scan_pages(vpz_ctx* ctx, uint32_t n, const uint8_t* const* datas, const size_t* lens,
                                  vpz_page_info* pages, size_t pages_cap, uint32_t* first, uint32_t* count,
                                  uint64_t* waste_bits, uint32_t* crc_failures) {
  if (!ctx || (n && (!datas || !lens))) return VPZ_E_ARGUMENT;
  VPZ_USE(ctx);
  static_assert(sizeof(vpz_page_info) == sizeof(VpzPageRec), "vpz_page_info mirrors VpzPageRec");
  if (!ctx->pool && n > 16) {   // staging many images is a parallel memcpy
    unsigned t = ctx->host_threads > 0 ? (unsigned)ctx->host_threads
                                       : std::max(1u, std::min(std::thread::hardware_concurrency(), 32u));
    ctx->pool = new (std::nothrow) ThreadPool(t);
  }
  ScanResult r;
  int rc = scan_pages(ctx, n, datas, lens, n > 16 ? ctx->pool : nullptr, &r);
  if (rc) return rc;
  int64_t total = 0;
  for (uint32_t i = 0; i < n; i++) {
    const VpzScanOut& o = r.out[i];
    if (o.overflow) {
      ctx->last_error = "file has more pages than the device scan sized for";
      return VPZ_E_UNSUPPORTED;
    }
    if (first) first[i] = (uint32_t)total;
    if (count) count[i] = o.n_pages;
    if (waste_bits) waste_bits[i] = 8 * (((uint64_t)o.waste_hi << 32) | o.waste_lo);
    if (crc_failures) crc_failures[i] = o.crc_failures;
    if (pages) {
      if ((size_t)total + o.n_pages > pages_cap) {
        ctx->last_error = "page array too small";
        return VPZ_E_ARGUMENT;
      }
      memcpy(pages + total, r.pages + r.files[i].page_base, (size_t)o.n_pages * sizeof(VpzPageRec));
    }
    total += o.n_pages;
  }
  return total;
}
