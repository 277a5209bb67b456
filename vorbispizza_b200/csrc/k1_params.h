// k1_params.h -- kernel parameter blocks (plain structs, shared by host engine and kernels).
#pragma once
#include <stdint.h>

#include "vpz_dev.h"

struct K1Debug {                 // all device pointers; used by vpz_debug_decode_packet only
  int32_t* hdr;                  // vpz_packet_dump as int32 words
  int32_t* scalars;
  int32_t scalars_cap;
  int32_t* classes;
  int32_t classes_cap;
  float* residue;                // [ch][n/2] before coupling
};

struct K1Params {
  const uint32_t* bytes;         // batch byte buffer (4-byte aligned packets, zero padded)
  const VpzPktIn* pkts;
  VpzPktRes* res;
  const uint32_t* const* setups; // per setup slot: device pointer of the blob
  float* spec;
  uint32_t n_pkts;
  uint32_t* counter;             // work-stealing cursor (zeroed before each launch)
  uint32_t smem_words_per_warp;  // K1b
  uint32_t seg_stride;           // K1b gather: words of the floor segment table per channel
  uint32_t* rec;                 // symbol records (K1a -> K1b), VpzPktIn.rec_off
  uint16_t* ent;                 // VQ entry indices (K1a -> K1b), VpzPktIn.ent_off
  const uint32_t* order;         // K1a: packet indices sorted by byte length (neighbouring lanes get like work)
  int gather_ok;                 // K1b: every setup of the batch can take the gather path
  int k1a_smem;                  // K1a: first-level Huffman tables in shared memory (simple, non-debug variant)
  K1Debug dbg;
};

struct K3Params {
  const float* spec;
  const VpzPktOla* pkts;
  const VpzPktRes* res;            // exec masks from K1 (NULL: every channel executes)
  const VpzOlaItem* items;
  const uint32_t* const* setups;
  float* pcm;                      // interleaved output; holds int16 elements at the same element offsets when out16 is set
  int out16;                       // 1: 16-bit PCM by the reference tests' rule (AssetTest.cs:131-132); fast kernel only
  uint32_t* clip_first;            // per packet: smallest clipped sample index (init 0xffffffff), may be NULL
  uint32_t n_items;
  uint32_t* counter;               // work-stealing cursor over items (zeroed before each launch)
  int clip;
  float* dbg_imdct;                // debug: raw y[0..N) of every packet, [ch][N] at 2*spec_off, may be NULL
};

struct K0Params {
  const uint8_t* images;           // staged container images
  const VpzScanFile* files;
  VpzPageRec* pages;
  VpzScanOut* out;                 // one per file
  uint32_t n_files;
  uint32_t* counter;               // four zeroed words: file cursor of the walk, number of CRC jobs, job cursor, file
                                   // cursor of the serial pass
  // fast path (k0_walk / k0_crc): a file that is one gapless chain of pages is walked header by header, its page
  // CRCs are checked by all warps in parallel; anything else is flagged and left to the serial pass
  VpzCrcJob* jobs;                 // one CRC job per page the walk accepted
  uint32_t* irregular;             // per file, zeroed: 1 = the serial pass scans this file
  int only_irregular;              // serial pass: skip the files whose flag is 0
};

struct K4Params {
  const float* pcm;                // batch PCM (K3 output, unclipped)
  float* out;                      // dense output of the group, zero-filled before the launch
  const VpzCopySeg* segs;
  uint32_t n_segs;
  int clip;
};

struct K5Params {
  const float* pcm;                // batch PCM (K3 output)
  void* out;                       // the caller's device buffer: fp32 or int16 elements
  const VpzPlaceTile* tiles;
  uint32_t n_tiles;
  int planar;                      // 1: channel-major items, 0: interleaved
  int out16;                       // 1: int16 elements by K3's rule (k3_s16)
  int clip;                        // clip before the conversion (the excerpt path decodes unclipped)
};

struct K6Params {
  const float* src;                // interleaved fp32 source items: the batch PCM (files) or the slot's scratch (excerpts)
  void* out;                       // the caller's device buffer: fp32 or int16 elements
  const VpzConvTile* tiles;
  uint32_t n_tiles;
  uint32_t smem_floats;            // shared memory of the largest tile (staged frames x staged channels)
  int planar;                      // 1: channel-major items, 0: interleaved
  int out16;                       // 1: int16 elements by K3's rule (k3_s16)
};

struct K7Params {
  const uint8_t* images;           // the corpus's images: 16-byte aligned, zeros behind each
  uint8_t* bytes;                  // the batch's packet-byte area (K1a's input)
  const VpzGatherPiece* pieces;
  uint32_t n_pieces;
};

struct K0gParams {
  const uint8_t* images;           // the staged images of the K0 scan
  const VpzGranFile* files;
  const VpzPageRec* pages;         // K0's records
  long long* page_end;             // out: per page, granules up to and including it (same indexing as pages)
  uint32_t n_files;
};
