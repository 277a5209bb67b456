// ogg.cpp -- host-side Ogg layer (see ogg.h).  Reference behaviour followed, by function:
//   physical: PageReaderBase.ReadNextPage / VerifyHeader / VerifyPage (Ogg/PageReaderBase.cs:41-84,176-212,286-361),
//             PageReader.AddPage (Ogg/PageReader.cs:58-102), Crc (Ogg/Crc.cs:20-63, Ogg/Crc.Table.cs:14),
//             PageHeader.GetPacketCount (Ogg/PageHeader.cs:35-59), PageData.GetPacket (Ogg/PageData.cs:53-83)
//   logical:  StreamPageReader.AddPage / FindPage / GetPage (Ogg/StreamPageReader.cs:44-110,152-305,335-424),
//             PacketProvider.* (Ogg/PacketProvider.cs:35-560)
#include "ogg.h"

#include <limits.h>
#include <string.h>

#include <map>

#include "../../include/vpz.h"

namespace vpz {

// Ogg CRC-32 (poly 0x04c11db7, init 0, MSB first, no final xor), slice-by-8: the same check as the
// reference's byte-swapped slice-by-8 table (Ogg/Crc.cs:20-63, Ogg/Crc.Table.cs:14-40).
static uint32_t g_crc_table[8][256];
static bool crc_init() {
  for (uint32_t i = 0; i < 256; i++) {
    uint32_t r = i << 24;
    for (int j = 0; j < 8; j++) r = (r << 1) ^ ((r & 0x80000000u) ? 0x04c11db7u : 0u);
    g_crc_table[0][i] = r;
  }
  for (uint32_t i = 0; i < 256; i++)
    for (int k = 1; k < 8; k++) {
      uint32_t r = g_crc_table[k - 1][i];
      g_crc_table[k][i] = (r << 8) ^ g_crc_table[0][r >> 24];
    }
  return true;
}
static const bool g_crc_ready = crc_init();

static uint32_t crc_table(const uint8_t* data, size_t len, uint32_t crc) {
  (void)g_crc_ready;
  size_t i = 0;
  for (; i + 8 <= len; i += 8) {
    const uint8_t* p = data + i;
    uint32_t hi = crc ^ (((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3]);
    crc = g_crc_table[7][hi >> 24] ^ g_crc_table[6][(hi >> 16) & 0xff] ^ g_crc_table[5][(hi >> 8) & 0xff] ^
          g_crc_table[4][hi & 0xff] ^ g_crc_table[3][p[4]] ^ g_crc_table[2][p[5]] ^ g_crc_table[1][p[6]] ^
          g_crc_table[0][p[7]];
  }
  for (; i < len; i++) crc = (crc << 8) ^ g_crc_table[0][((crc >> 24) ^ data[i]) & 0xff];
  return crc;
}

#if defined(__x86_64__) && defined(__GNUC__)
}  // namespace vpz
#include <immintrin.h>
namespace vpz {
// The same CRC by carry-less multiplication (page bodies are ~4 KB; the page scan is the largest host cost
// of the bulk path).  The message is a polynomial with its first byte on top.  A 16-byte accumulator
// A = Ah x^64 + Al followed by d more bytes is congruent to Ah (x^(8d+64) mod P) + Al (x^(8d) mod P) plus
// those bytes: 64 x 32-bit products, so the sum stays below 128 bits.  Four accumulators run 64 bytes
// apart; what is left (the folded 16 bytes and the tail) goes through the table.  An initial crc is the
// same as XOR-ing it into the first four message bytes.
static uint32_t xpow_mod(unsigned n) {   // x^n mod P
  uint32_t r = 1;
  for (unsigned i = 0; i < n; i++) r = (r << 1) ^ ((r & 0x80000000u) ? 0x04c11db7u : 0u);
  return r;
}
static uint64_t g_k64_hi, g_k64_lo, g_k16_hi, g_k16_lo;
static bool g_crc_clmul = false;

#define VPZ_CRC_LOAD(p) _mm_shuffle_epi8(_mm_loadu_si128(reinterpret_cast<const __m128i*>(p)), bswap)
#define VPZ_CRC_FOLD(a, k, next) \
  _mm_xor_si128(_mm_xor_si128(_mm_clmulepi64_si128(a, k, 0x11), _mm_clmulepi64_si128(a, k, 0x00)), next)
__attribute__((target("pclmul,ssse3"))) static uint32_t crc_clmul(const uint8_t* data, size_t len, uint32_t crc) {
  const __m128i bswap = _mm_set_epi8(0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15);
  const __m128i k64 = _mm_set_epi64x((long long)g_k64_hi, (long long)g_k64_lo);
  const __m128i k16 = _mm_set_epi64x((long long)g_k16_hi, (long long)g_k16_lo);
  __m128i a0 = _mm_xor_si128(VPZ_CRC_LOAD(data), _mm_set_epi32((int)crc, 0, 0, 0));
  size_t i = 16;
  if (len >= 128) {
    __m128i a1 = VPZ_CRC_LOAD(data + 16), a2 = VPZ_CRC_LOAD(data + 32), a3 = VPZ_CRC_LOAD(data + 48);
    i = 64;
    for (; i + 64 <= len; i += 64) {
      a0 = VPZ_CRC_FOLD(a0, k64, VPZ_CRC_LOAD(data + i));
      a1 = VPZ_CRC_FOLD(a1, k64, VPZ_CRC_LOAD(data + i + 16));
      a2 = VPZ_CRC_FOLD(a2, k64, VPZ_CRC_LOAD(data + i + 32));
      a3 = VPZ_CRC_FOLD(a3, k64, VPZ_CRC_LOAD(data + i + 48));
    }
    a0 = VPZ_CRC_FOLD(a0, k16, a1);
    a0 = VPZ_CRC_FOLD(a0, k16, a2);
    a0 = VPZ_CRC_FOLD(a0, k16, a3);
  }
  for (; i + 16 <= len; i += 16) a0 = VPZ_CRC_FOLD(a0, k16, VPZ_CRC_LOAD(data + i));
  uint8_t tmp[16];
  _mm_storeu_si128(reinterpret_cast<__m128i*>(tmp), _mm_shuffle_epi8(a0, bswap));
  return crc_table(data + i, len - i, crc_table(tmp, 16, 0));
}
#undef VPZ_CRC_LOAD
#undef VPZ_CRC_FOLD

static bool crc_clmul_init() {
  __builtin_cpu_init();   // this runs from a static initialiser
  if (!__builtin_cpu_supports("pclmul") || !__builtin_cpu_supports("ssse3")) return false;
  g_k64_hi = xpow_mod(512 + 64);
  g_k64_lo = xpow_mod(512);
  g_k16_hi = xpow_mod(128 + 64);
  g_k16_lo = xpow_mod(128);
  // self-check against the table on every length class before the fast path is trusted
  uint8_t buf[400];
  uint32_t x = 0x12345678u;
  for (size_t i = 0; i < sizeof(buf); i++) {
    x = x * 1664525u + 1013904223u;
    buf[i] = (uint8_t)(x >> 24);
  }
  for (size_t n = 16; n <= sizeof(buf); n += 7)
    if (crc_clmul(buf, n, 0x9e3779b9u * (uint32_t)n) != crc_table(buf, n, 0x9e3779b9u * (uint32_t)n)) return false;
  return true;
}
static const bool g_crc_clmul_ready = (g_crc_clmul = crc_clmul_init());
#endif

uint32_t ogg_crc(const uint8_t* data, size_t len, uint32_t crc) {
#if defined(__x86_64__) && defined(__GNUC__)
  if (len >= 64 && g_crc_clmul) return crc_clmul(data, len, crc);
#endif
  return crc_table(data, len, crc);
}

// page length when a valid page starts at `pos`, else 0
static size_t try_page(const uint8_t* f, size_t len, size_t pos, int* crc_fail) {
  if (pos + 27 > len) return 0;
  if (memcmp(f + pos, "OggS", 4) != 0) return 0;
  int nseg = f[pos + 26];
  if (pos + 27 + (size_t)nseg > len) return 0;
  size_t body = 0;
  for (int i = 0; i < nseg; i++) body += f[pos + 27 + i];
  size_t total = 27 + (size_t)nseg + body;
  if (pos + total > len) return 0;
  uint32_t want;
  memcpy(&want, f + pos + 22, 4);
  static const uint8_t zero4[4] = {0, 0, 0, 0};
  uint32_t crc = ogg_crc(f + pos, 22, 0);
  crc = ogg_crc(zero4, 4, crc);
  crc = ogg_crc(f + pos + 26, total - 26, crc);
  if (crc != want) {
    ++*crc_fail;
    return 0;
  }
  return total;
}

OggContainer::~OggContainer() {
  for (LogicalStream* s : streams) delete s;
}

// PageReader.AddPage (Ogg/PageReader.cs:58-102): hands a verified page to the logical stream of its serial
// number.  `open` / `ignored` live for one scan.
namespace {
struct Demux {
  std::map<uint32_t, LogicalStream*> open;   // serial -> stream still receiving pages
  std::map<uint32_t, bool> ignored;
};
}  // namespace

static void demux_page(OggContainer* c, Demux& dm, const OggPage& p, uint32_t serial, size_t plen) {
  if (dm.ignored.count(serial) || p.packet_count == 0) {
    // PageReader.AddPage refuses a page without packets; the serial is ignored from then on
    if (p.packet_count == 0 && !dm.open.count(serial)) dm.ignored[serial] = true;
    if (p.packet_count == 0 && dm.open.count(serial)) {
      dm.open.erase(serial);
      dm.ignored[serial] = true;
    }
    c->waste_bits += (int64_t)plen * 8;
    return;
  }
  LogicalStream* ls;
  auto it = dm.open.find(serial);
  if (it == dm.open.end()) {
    ls = new LogicalStream;
    ls->serial = serial;
    c->streams.push_back(ls);
    dm.open[serial] = ls;
  } else {
    ls = it->second;
  }
  ls->pages.push_back(p);
  if (p.flags & 4) dm.open.erase(serial);  // PageReader.cs:76-84: a later page with this serial starts a new stream
}

int OggContainer::scan(const uint8_t* d, size_t n) {
  data = d;
  len = n;
  Demux dm;
  size_t pos = 0;
  bool resync = false;
  while (pos + 4 <= len) {
    size_t plen = try_page(d, len, pos, &crc_failures);
    if (!plen) {
      pos++;
      waste_bits += 8;
      resync = true;
      continue;
    }
    const uint8_t* h = d + pos;
    OggPage p;
    p.offset = (int64_t)pos;
    p.flags = h[5];
    memcpy(&p.granule, h + 6, 8);
    uint32_t serial;
    memcpy(&serial, h + 14, 4);
    memcpy(&p.seq, h + 18, 4);
    p.nseg = h[26];
    p.seg = h + 27;
    p.body = h + 27 + p.nseg;
    p.body_len = (int)(plen - 27 - (size_t)p.nseg);
    p.is_resync = resync;
    int cnt = 0;
    for (int i = 0; i < p.nseg; i++)
      if (p.seg[i] < 255) cnt++;
    p.is_continued = p.nseg > 0 && p.seg[p.nseg - 1] == 255;
    if (p.is_continued) cnt++;
    p.packet_count = cnt;
    resync = false;
    pos += plen;
    demux_page(this, dm, p, serial, plen);
  }
  if (pos < len) waste_bits += 8 * (int64_t)(len - pos);
  return streams.empty() ? VPZ_E_INVALID_DATA : VPZ_OK;
}

// The same container state from the page records of the GPU scan (k0_pages.cuh): the device found the pages,
// verified their CRCs and counted their packets; the host only files them under their serial numbers.
int OggContainer::scan_from_records(const uint8_t* d, size_t n, const VpzPageRec* recs, uint32_t count,
                                    uint64_t waste_bytes, uint32_t crc_fail) {
  data = d;
  len = n;
  waste_bits = 8 * (int64_t)waste_bytes;
  crc_failures = (int)crc_fail;
  Demux dm;
  for (uint32_t i = 0; i < count; i++) {
    const VpzPageRec& r = recs[i];
    const size_t plen = 27 + (size_t)r.nseg + r.body_len;
    if ((size_t)r.offset + plen > n) return VPZ_E_INVALID_DATA;   // a record that does not fit its own file
    const uint8_t* h = d + r.offset;
    OggPage p;
    p.offset = (int64_t)r.offset;
    p.flags = r.flags;
    p.granule = (int64_t)(((uint64_t)r.granule_hi << 32) | r.granule_lo);
    p.seq = r.seq;
    p.nseg = r.nseg;
    p.seg = h + 27;
    p.body = h + 27 + p.nseg;
    p.body_len = (int)r.body_len;
    p.is_resync = r.is_resync != 0;
    p.is_continued = r.is_continued != 0;
    p.packet_count = r.packet_count;
    demux_page(this, dm, p, r.serial, plen);
  }
  return streams.empty() ? VPZ_E_INVALID_DATA : VPZ_OK;
}

// StreamPageReader.AddPage (Ogg/StreamPageReader.cs:44-110), applied when a page is first touched
int LogicalStream::load_pages_upto(int64_t idx) {
  while (pages_loaded <= idx && !has_all_pages) {
    if (pages_loaded >= (int64_t)pages.size()) {
      has_all_pages = true;  // SetEndOfStreams at the physical end
      break;
    }
    const OggPage& p = pages[(size_t)pages_loaded];
    if (p.granule != -1) {
      if (first_data_page < 0 && p.granule > 0) {
        first_data_page = pages_loaded;
      } else if (max_granule > p.granule) {
        return VPZ_E_INVALID_DATA;  // "Granule Position regressed?!"
      }
      max_granule = p.granule;
    } else if (first_data_page >= 0 && (!p.is_continued || p.packet_count != 1)) {
      return VPZ_E_INVALID_DATA;
    }
    if (p.flags & 4) has_all_pages = true;
    if (pages_loaded > 0) {
      uint32_t last = pages[(size_t)pages_loaded - 1].seq;
      if (last != 0 && last + 1 != p.seq) pages.mut((size_t)pages_loaded).is_resync = true;
    }
    container_bits += 8 * (27 + p.nseg);
    pages_loaded++;
  }
  return VPZ_OK;
}

const OggPage* LogicalStream::get_page(int64_t idx) {
  if (idx < 0) return nullptr;
  if (load_pages_upto(idx) != VPZ_OK) return nullptr;
  if (idx < pages_loaded) return &pages[(size_t)idx];
  return nullptr;
}

// PageData.GetPacket (Ogg/PageData.cs:53-83)
static void page_packet_slice(const OggPage* p, int packet_index, const uint8_t** data, int* len) {
  int pk = 0, ofs = 0, size = 0;
  for (int i = 0; i < p->nseg; i++) {
    size += p->seg[i];
    if (p->seg[i] < 255) {
      if (pk == packet_index) {
        *data = p->body + ofs;
        *len = size;
        return;
      }
      pk++;
      ofs += size;
      size = 0;
    }
  }
  if (pk == packet_index) {
    *data = p->body + ofs;
    *len = size;
    return;
  }
  *data = p->body;
  *len = 0;
}

// PacketProvider.CreatePacket (Ogg/PacketProvider.cs:427-560)
void LogicalStream::create_packet(int64_t* pg, int* pk, bool advance, int64_t granule_pos, bool is_resync,
                                  bool is_continued, int packet_count, OggPacket* out) {
  *out = OggPacket();
  const OggPage* first = get_page(*pg);
  if (!first) return;
  const uint8_t* d;
  int n;
  out->page_index = *pg;
  out->packet_index = *pk;
  page_packet_slice(first, *pk, &d, &n);
  out->ptr = d;
  out->len = (uint32_t)n;
  bool is_last;
  int64_t final_page = *pg;
  if (is_continued && *pk == packet_count - 1) {
    int64_t cont = *pg;
    while (is_continued) {
      const OggPage* np = get_page(++cont);
      if (!np) {
        *out = OggPacket();  // default(VorbisPacket)
        return;
      }
      granule_pos = np->granule;
      is_resync = np->is_resync;
      is_continued = np->is_continued;
      packet_count = np->packet_count;
      if (!(np->flags & 1) || is_resync) break;
      if (is_continued && packet_count > 1) is_continued = false;
      page_packet_slice(np, 0, &d, &n);
      if (out->spans.empty()) out->spans.push_back(OggSpan{out->ptr, out->len});
      out->spans.push_back(OggSpan{d, (uint32_t)n});
      if (out->owned.empty() && out->len) out->owned.assign(out->ptr, out->ptr + out->len);
      out->owned.insert(out->owned.end(), d, d + n);
      out->len = (uint32_t)out->owned.size();
      out->ptr = out->owned.data();
    }
    is_last = packet_count == 1;
    final_page = cont;
  } else {
    is_last = *pk == packet_count - 1;
  }
  out->valid = true;
  out->is_resync = is_resync;
  if (is_last) {
    out->granule = granule_pos;
    if (has_all_pages && final_page == page_count() - 1) out->is_eos = true;
  } else {
    out->granule = -1;
  }
  if (advance) {
    if (final_page != *pg) {
      *pg = final_page;
      *pk = 0;
    }
    if (*pk == packet_count - 1) {
      ++*pg;
      *pk = 0;
    } else {
      ++*pk;
    }
  }
}

void LogicalStream::next_packet(OggPacket* out) {
  const OggPage* p = get_page(page_index);
  if (!p) {
    *out = OggPacket();
    return;
  }
  create_packet(&page_index, &packet_index, true, p->granule, p->is_resync, p->is_continued, p->packet_count, out);
}

// PacketProvider.CreateValidPacket (Ogg/PacketProvider.cs:413-425)
int LogicalStream::create_valid_packet(int64_t* pg, int* pk, bool is_resync, bool is_continued, int packet_count,
                                       OggPacket* out) {
  create_packet(pg, pk, false, 0, *pk == 0 && is_resync, is_continued, packet_count, out);
  return out->valid ? VPZ_OK : VPZ_E_INVALID_DATA;
}

// StreamPageReader.FindFirstDataPage (Ogg/StreamPageReader.cs:191-208)
int64_t LogicalStream::first_data_page_index() {
  int64_t idx = pages_loaded - 1;
  if (idx < 0) idx = 0;
  while (first_data_page < 0) {
    if (!get_page(idx)) return -1;
    idx++;
  }
  return first_data_page;
}

// PacketProvider.FillPageEndGranuleCache (Ogg/PacketProvider.cs:203-307)
int LogicalStream::fill_page_end_cache(int64_t target) {
  int64_t p_index = (int64_t)page_end_granules.size();
  int64_t first_data = first_data_page_index();
  if (first_data < 0) first_data = 0;
  while (p_index < first_data) {
    page_end_granules.push_back(0);
    p_index++;
  }
  while (p_index <= target) {
    if (has_all_pages && p_index >= page_count()) break;
    int64_t page_length = 0;
    int first_real = 0;
    int64_t prev = p_index - 1;
    if (prev >= 0) {
      const OggPage* pp = get_page(prev);
      if (!pp) return VPZ_E_INVALID_DATA;
      if (pp->is_continued) {
        int last_idx = pp->packet_count - 1;
        OggPacket pk;
        int64_t pi = prev;
        create_packet(&pi, &last_idx, false, 0, false, pp->is_continued, pp->packet_count, &pk);
        if (!pk.valid) {
          if (!has_all_pages) return VPZ_E_INVALID_DATA;
          break;
        }
        page_length += granule_count ? granule_count(pk) : 0;
        first_real = 1;
      }
    }
    const OggPage* p = get_page(p_index);
    if (!p) {
      if (!has_all_pages) return VPZ_E_INVALID_DATA;
      break;
    }
    int packet_idx = first_real;
    if (p_index == first_data) packet_idx = 1;
    int p_count = p->packet_count;
    if (p->is_continued) p_count--;
    for (; packet_idx < p_count; packet_idx++) {
      OggPacket pk;
      int64_t pi = p_index;
      int rc = create_valid_packet(&pi, &packet_idx, p->is_resync, p->is_continued, p->packet_count, &pk);
      if (rc != VPZ_OK) return rc;
      page_length += granule_count ? granule_count(pk) : 0;
    }
    int64_t g = page_length;
    if (p_index > 0) g += page_end_granules[(size_t)p_index - 1];
    page_end_granules.push_back(g);
    p_index++;
  }
  return VPZ_OK;
}

// PacketProvider.GetPageRange (Ogg/PacketProvider.cs:171-201)
bool LogicalStream::get_page_range(int64_t pg, int64_t* start, int64_t* end, int* err) {
  const uint64_t n = page_end_granules.size();
  if ((uint64_t)pg >= n) {
    int rc = fill_page_end_cache(pg);
    if (rc != VPZ_OK) {
      *err = rc;
      *start = *end = 0;
      return false;
    }
    if ((uint64_t)pg > page_end_granules.size()) pg = (int64_t)page_end_granules.size();
  }
  const uint64_t m = page_end_granules.size();
  *start = (uint64_t)(pg - 1) < m ? page_end_granules[(size_t)(pg - 1)] : 0;
  if ((uint64_t)pg < m) {
    *end = page_end_granules[(size_t)pg];
    return true;
  }
  *end = *start;
  return false;
}

// PacketProvider.GetGranuleCount (Ogg/PacketProvider.cs:35-49)
int64_t LogicalStream::total_granules(int* err) {
  int64_t start, end;
  int e = 0;
  get_page_range(INT64_MAX, &start, &end, &e);
  if (e) {
    *err = e;
    return 0;
  }
  if (has_all_pages && start > max_granule) start = max_granule;
  return start;
}

// StreamPageReader.FindPage (Ogg/StreamPageReader.cs:152-305): all three search strategies land on
// the first page whose header granule exceeds the target (index + 1 on a direct hit).
int64_t LogicalStream::find_page(int64_t granule_pos, int* err) {
  if (granule_pos == 0) {
    int64_t fd = first_data_page_index();
    if (fd < 0) *err = VPZ_E_SEEK_RANGE;
    return fd;
  }
  int64_t last = pages_loaded - 1;
  if (last < 0) {
    if (!get_page(0)) {
      *err = VPZ_E_SEEK_RANGE;
      return -1;
    }
    last = pages_loaded - 1;
  }
  int64_t last_gp = pages[(size_t)last].granule;
  if (granule_pos < last_gp) {
    int64_t low = first_data_page_index(), high = last, high_gp = last_gp, low_gp = 0, dist;
    if (low < 0) {
      *err = VPZ_E_SEEK_RANGE;
      return -1;
    }
    while ((dist = high - low) > 0) {
      int64_t index = low + (int64_t)((double)dist * ((double)(granule_pos - low_gp) / (double)(high_gp - low_gp)));
      int64_t gp = pages[(size_t)index].granule;
      if (gp > granule_pos) {
        high = index;
        high_gp = gp;
      } else if (gp < granule_pos) {
        low = index + 1;
        low_gp = gp + 1;
      } else {
        return index + 1;
      }
    }
    return low;
  } else if (granule_pos > last_gp) {
    int64_t idx = last, gp = last_gp;
    while (gp <= granule_pos) {
      ++idx;
      const OggPage* p = get_page(idx);
      if (!p) {
        if (max_granule < granule_pos) {
          *err = VPZ_E_SEEK_RANGE;
          return -1;
        }
        break;
      }
      gp = p->granule;
    }
    return idx;
  }
  return last + 1;
}

// PacketProvider.NormalizePacketIndex (Ogg/PacketProvider.cs:312-348)
bool LogicalStream::normalize_packet_index(int64_t* page_idx, int* packet_idx) {
  const OggPage* p = get_page(*page_idx);
  if (!p) return false;
  bool is_resync = p->is_resync, is_continuation = (p->flags & 1) != 0;
  int64_t pg = *page_idx;
  int pk = *packet_idx;
  while (pk < (is_continuation ? 1 : 0)) {
    if (is_continuation && is_resync) return false;
    bool was_continuation = is_continuation;
    const OggPage* q = get_page(--pg);
    if (!q) return false;
    is_resync = q->is_resync;
    is_continuation = (q->flags & 1) != 0;
    if (was_continuation && !q->is_continued) return false;
    pk += q->packet_count - (was_continuation ? 1 : 0);
  }
  *page_idx = pg;
  *packet_idx = pk;
  return true;
}

// PacketProvider.SeekTo + GetTargetPageInfo (Ogg/PacketProvider.cs:56-169)
int64_t LogicalStream::seek_to(int64_t granule_pos, int pre_roll, int* err) {
  if (granule_pos < 0) {
    *err = VPZ_E_ARGUMENT;
    return 0;
  }
  int64_t pg = find_page(granule_pos, err);
  if (*err) return 0;
  int64_t page_start = 0, page_end = 0;
  for (;;) {
    if (!get_page_range(pg, &page_start, &page_end, err)) return page_start;  // "we're at the last page"
    if (granule_pos >= page_start && granule_pos <= page_end) break;
    if (granule_pos - page_end > 0) pg++; else pg--;
  }
  const OggPage* p = get_page(pg);
  if (!p) {
    *err = VPZ_E_INVALID_DATA;
    return 0;
  }
  bool is_continuation = (p->flags & 1) != 0;
  int first_real = is_continuation ? 1 : 0;
  int64_t cur = page_end;
  int pk_idx = p->packet_count - 1;
  if (p->is_continued) pk_idx--;
  for (; pk_idx >= first_real; pk_idx--) {
    OggPacket pk;
    int64_t pi = pg;
    int rc = create_valid_packet(&pi, &pk_idx, pk_idx == 0 && p->is_resync, p->is_continued, p->packet_count, &pk);
    if (rc != VPZ_OK) {
      *err = rc;
      return 0;
    }
    cur -= granule_count ? granule_count(pk) : 0;
    if (granule_pos >= cur) break;
  }
  if (pk_idx == 0 && first_real == 1) {
    int64_t prev = pg - 1;
    const OggPage* pp = get_page(prev);
    if (!pp) {
      *err = VPZ_E_INVALID_DATA;
      return 0;
    }
    int last_idx = pp->packet_count - 1;
    OggPacket pk;
    int64_t pi = prev;
    int rc = create_valid_packet(&pi, &last_idx, pk_idx == 0 && p->is_resync, p->is_continued, p->packet_count, &pk);
    if (rc != VPZ_OK) {
      *err = rc;
      return 0;
    }
    cur -= granule_count ? granule_count(pk) : 0;
    pg = prev;
    pk_idx = last_idx;
  }
  if (pg > first_data_page_index() || pk_idx > 0) pk_idx -= pre_roll;
  if (!normalize_packet_index(&pg, &pk_idx)) {
    *err = VPZ_E_SEEK_RANGE;
    return 0;
  }
  page_index = pg;
  packet_index = (uint8_t)pk_idx;
  return cur;
}

}  // namespace vpz
