// ogg.h -- host-side Ogg layer over an in-memory container image: physical page scan with CRC
// and resync accounting, per-serial logical streams, packet assembly across pages, granule
// bookkeeping and seeking.  Behaviour follows the reference's Ogg/ classes (cited per function in
// ogg.cpp); this layer feeds the GPU batcher and never touches the device.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <functional>
#include <memory>
#include <vector>

#include "vpz_dev.h"

namespace vpz {

struct OggPage {
  int64_t offset = 0;
  int64_t granule = 0;
  uint32_t seq = 0;
  uint8_t flags = 0;  // 1 continuation, 2 BOS, 4 EOS
  int nseg = 0;
  const uint8_t* seg = nullptr;
  const uint8_t* body = nullptr;
  int body_len = 0;
  bool is_resync = false;
  int packet_count = 0;
  bool is_continued = false;
};

struct OggSpan {   // bytes of the container image
  const uint8_t* p = nullptr;
  uint32_t len = 0;
};

struct OggPacket {
  // A packet that lies inside one page is a VIEW into the container image (no copy); only packets
  // continued across pages are assembled into `owned`.
  const uint8_t* ptr = nullptr;
  uint32_t len = 0;
  std::vector<uint8_t> owned;
  std::vector<OggSpan> spans;   // a packet continued across pages: its bytes on each page, in order (views)
  const uint8_t* data() const { return ptr; }
  size_t size() const { return len; }
  bool valid = false;
  bool is_resync = false, is_eos = false;
  int64_t granule = -1;
  int64_t page_index = 0;
  int packet_index = 0;
};

uint32_t ogg_crc(const uint8_t* data, size_t len, uint32_t crc = 0);

// A vector that copies of its owner share until one of them writes (copy on write): a copy of a LogicalStream is a
// new packet cursor over the same page list and page-end index, whatever the length of the file.  Writers copy first,
// so a shared vector is never written; concurrent copies of one unchanged master are safe.
template <class T>
class SharedVec {
 public:
  size_t size() const { return v_->size(); }
  bool empty() const { return v_->empty(); }
  const T& operator[](size_t i) const { return (*v_)[i]; }
  T& mut(size_t i) { return own()[i]; }
  void push_back(const T& x) { own().push_back(x); }
  template <class It>
  void assign(It first, It last) { own().assign(first, last); }
  operator const std::vector<T>&() const { return *v_; }

 private:
  std::shared_ptr<std::vector<T>> v_ = std::make_shared<std::vector<T>>();
  std::vector<T>& own() {
    if (v_.use_count() > 1) v_ = std::make_shared<std::vector<T>>(*v_);
    return *v_;
  }
};

// One logical bitstream (one serial number, BOS..EOS) = StreamPageReader + PacketProvider.
class LogicalStream {
 public:
  uint32_t serial = 0;
  SharedVec<OggPage> pages;         // every page the physical reader would hand to this stream
  // lazily "read" prefix: HasAllPages / IsEndOfStream in the reference depend on how far the
  // reader has got (StreamPageReader.cs:82-85,249,442-446)
  int64_t pages_loaded = 0;
  bool has_all_pages = false;
  int64_t first_data_page = -1;
  int64_t max_granule = 0;
  int64_t container_bits = 0;
  // packet cursor (PacketProvider._pageIndex/_packetIndex)
  int64_t page_index = 0;
  int packet_index = 0;
  SharedVec<int64_t> page_end_granules;
  // IPacketGranuleCountProvider.GetPacketGranuleCount (set by the decoder)
  std::function<int(const OggPacket&)> granule_count;

  int load_pages_upto(int64_t idx);                  // StreamPageReader.AddPage; <0: InvalidData
  const OggPage* get_page(int64_t idx);              // IStreamPageReader.GetPage
  int64_t page_count() const { return pages_loaded; }
  void next_packet(OggPacket* out);                  // PacketProvider.GetNextPacket
  int64_t total_granules(int* err);                  // PacketProvider.GetGranuleCount
  int64_t seek_to(int64_t granule, int pre_roll, int* err);  // PacketProvider.SeekTo
  bool can_seek() const { return true; }

 private:
  void create_packet(int64_t* page_index, int* packet_index, bool advance, int64_t granule_pos, bool is_resync,
                     bool is_continued, int packet_count, OggPacket* out);
  int create_valid_packet(int64_t* page_index, int* packet_index, bool is_resync, bool is_continued, int packet_count,
                          OggPacket* out);
  int64_t first_data_page_index();
  int fill_page_end_cache(int64_t target);
  bool get_page_range(int64_t page_index, int64_t* start, int64_t* end, int* err);
  int64_t find_page(int64_t granule_pos, int* err);
  bool normalize_packet_index(int64_t* page_index, int* packet_index);
};

// Physical layer: scans the whole image once and demultiplexes by serial number.
class OggContainer {
 public:
  const uint8_t* data = nullptr;
  size_t len = 0;
  int64_t waste_bits = 0;
  int crc_failures = 0;
  std::vector<LogicalStream*> streams;  // in order of first page
  ~OggContainer();
  int scan(const uint8_t* d, size_t n);  // 0, or <0 when no page was found
  // the same from the page records of the GPU scan (vpz_dev.h VpzPageRec, k0_pages.cuh)
  int scan_from_records(const uint8_t* d, size_t n, const VpzPageRec* recs, uint32_t count, uint64_t waste_bytes,
                        uint32_t crc_fail);
};

}  // namespace vpz
