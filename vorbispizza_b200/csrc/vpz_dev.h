// vpz_dev.h -- structures shared by the host table builder and the sm_100a kernels.
//
// One "setup blob" per distinct Vorbis setup (id + setup header pair) is built on the host
// (setup.cpp) and uploaded once; every kernel argument that refers to codebooks, floors,
// residues, mappings or modes is an offset into that blob.  The blob is position independent:
// all references are 32-bit offsets counted in 4-byte words from the start of the blob.
#pragma once
#include <stdint.h>

#define VPZ_MAX_CH 8          // channels handled by the GPU path (reference has no limit; SURVEY 8f-3)
#define VPZ_MAX_POSTS 64      // Floor1.cs:17 (Posts capacity, quirk Q2)
#define VPZ_MAX_BOOKS 256
#define VPZ_MAX_MODES 64
#define VPZ_L1_BITS_DEFAULT 9 // first-level Huffman table width (reference: 10, Huffman.cs:12)
#define VPZ_L2_BITS_MAX 8      // second-level table width

// ---- codebook (Codebook.cs, Huffman.cs) ------------------------------------------------
// L1 table entry: (value << 8) | length for codes with length <= l1_bits, replicated over the
// don't-care bits exactly like Huffman.GenerateTable.  Codes longer than l1_bits:
// 0x80000000 | (L2 word offset from l1_off) << 5 | l2_bits: a second table over the next l2_bits
// stream bits with the same entry format; codes longer than l1_bits + VPZ_L2_BITS_MAX leave
// 0x80000000 | range_id there, where range_id indexes `ranges` = {lo, hi} into the long-code arrays
// (sorted by MSB-first left-aligned code).  0 = no code with this prefix (DecodeScalar -> -1).
struct VpzBook {
  uint32_t l1_off;      // word offset of the L1 table, 1 << l1_bits entries
  uint32_t range_off;   // word offset of {lo,hi} pairs
  uint32_t lcode_off;   // word offset of left-aligned long codes (ascending)
  uint32_t linfo_off;   // word offset of (value << 8) | length per long code
  uint32_t vq_off;      // word offset of the float lookup [entries * dims], 0 when map_type == 0
  uint32_t entries;
  uint16_t dims;
  uint8_t l1_bits;
  uint8_t max_bits;     // Codebook._maxBits (quirk Q7 kept for the record; decode does not need it)
  uint8_t map_type;
  uint8_t pad[3];
  uint32_t long_n;
};

// ---- floor 1 (Floor1.cs:39-155) ---------------------------------------------------------
struct VpzFloor1 {
  uint8_t partitions;
  uint8_t multiplier;   // 1..4
  uint8_t ybits;
  uint8_t xcount;       // posts incl. the two end posts, <= 64
  uint16_t range;
  uint16_t floor_type;  // 1 = floor 1 (this struct), 0 = floor 0 (the f0 part below; Floor0.cs)
  uint8_t part_class[32];
  uint8_t class_dim[16];
  uint8_t class_sub[16];
  uint8_t class_master[16];
  int16_t sub_books[16][8];  // -1: no book, value 0
  uint16_t xlist[VPZ_MAX_POSTS + 1];
  uint8_t lneigh[VPZ_MAX_POSTS + 1];
  uint8_t hneigh[VPZ_MAX_POSTS + 1];
  uint8_t sortidx[VPZ_MAX_POSTS + 1];
  uint8_t pad1[3];
  // K1a: [16 classes][9] x {first-level table word offset, l1_bits | book << 8}; entry 0 of a class is its master
  // book, entries 1..8 the sub books; the second word is 0 for "no book" (the post is 0, nothing is read).  One
  // 8-byte load per codeword instead of sub_books -> VpzBook.l1_off -> VpzBook.l1_bits.
  uint32_t fbook_tab_off;
  // ---- floor 0 (Floor0.cs:39-113), valid when floor_type == 0 ----
  struct {
    uint8_t order;          // 1..255 LSP coefficients
    uint8_t amp_bits;       // 1..32 on the GPU path
    uint8_t amp_ofs;
    uint8_t nbooks;         // 1..16
    uint8_t book_bits;      // ilog(nbooks)
    uint8_t pad[3];
    uint16_t rate, bark_map_size;
    uint8_t books[16];
    uint32_t bark_off[2];   // per block size: uint16 bark index per bin, n entries (entry n-1 is 0: Floor0.cs:88-94)
    uint32_t wmap_off[2];   // per block size: 2 cos(pi / bark_map_size * k), n floats, indexed by BARK index
  } f0;
};

// ---- residue 0/1/2 (Residue0.cs:25-115) -------------------------------------------------
struct VpzResidue {
  uint8_t type;
  uint8_t classifications;
  uint8_t class_book;
  uint8_t max_stages;
  uint32_t begin, end, part_size;
  uint32_t decode_map_off;   // word offset; one byte per (classword, dim) packed 4 per word
  uint32_t decode_map_len;   // partvals * classbook.dims (quirk Q8 bound)
  uint8_t cascade[64];
  uint8_t has_books[64];
  uint8_t books[64][8];
  // K1a walk tables (built by setup.cpp; the lanes of K1a never loop over classes or cascades):
  //   unit_tab [classifications][8] x {l1 table word offset, l1_bits | book << 8 | entries per unit << 16};
  //            the second word is 0 when (class, stage) carries no codewords
  //   cw_tab   [nvec][partvals][max_stages] x uint32: for classword value `sym` of vector v, bit k * nvec + v
  //            is set when partition k of the group has codewords in that stage
  uint32_t unit_tab_off;
  uint32_t unit_tabb_off;    // K1b: [classifications][8] x {dims | log2 dims << 8 | entries per unit << 16, VQ table word offset}
  uint32_t cw_tab_off;
  uint32_t partvals;         // classifications ^ classbook.dims
  uint16_t cdim;             // classbook.dims (partitions per classword)
  uint16_t nvec;             // vectors the residue decodes: 1 for type 2, else nch
  uint16_t nch;              // channels of the submap this INSTANCE serves (Mapping.cs:136-146)
  uint16_t pad2;
};
// The device image holds residue INSTANCES: one per distinct (residue, channels of the submap) pair that a
// mapping uses, because the walk tables (cw_tab) depend on the number of vectors.  A stream whose mappings
// have a single submap has exactly one instance per residue, in header order.

// ---- mapping (Mapping.cs:19-95) ---------------------------------------------------------
struct VpzMapping {
  uint8_t submaps;
  uint8_t coupling_steps;
  uint8_t pad[2];
  uint8_t mag[32], ang[32];       // GPU path: at most 32 coupling steps
  uint8_t mux[VPZ_MAX_CH];
  uint8_t submap_floor[16], submap_residue[16];   // submap_residue: residue INSTANCE index (see VpzResidue)
};

struct VpzMode {
  uint8_t block_flag;
  uint8_t mapping;
};

// Header at word 0 of the blob.
struct VpzSetupHdr {
  uint32_t magic;           // 'VPZ1'
  uint32_t total_words;
  uint8_t channels;
  uint8_t log2_size0, log2_size1;
  uint8_t mode_bits;
  uint8_t nmodes, nmappings, nfloors, nresidues;
  uint32_t nbooks;
  uint32_t books_off, floors_off, residues_off, mappings_off, modes_off;
  uint32_t slope_off[2];    // window slopes, size0/2 and size1/2 floats (BlocksizeDerivedCache.cs)
  uint32_t tw_off[2];       // IMDCT pre/post twiddle exp(-i*pi*(n+1/8)/M), interleaved re,im, N/4 pairs
  uint32_t fft_off[2];      // FFT roots exp(-2*pi*i*k/H), interleaved re,im, H = N/4 pairs
  uint32_t db_off;          // 256 floats, Floor1.cs:407-473
  // K1a shared-memory tables, per block flag (0 short, 1 long): the first-level Huffman tables of the books the
  // packets of that block size decode with (residue books first, then classbooks, then floor books, up to
  // K1A_SM_WORDS words).  stage_off: {n, total words, n x {l1 table word offset, words, shared-memory word
  // offset}}; soff_off: 256 x uint16 shared-memory word offset per book, 0xffff = not staged.
  uint32_t k1a_stage_off[2];
  uint32_t k1a_soff_off[2];
  // ceil(2^32 / d) for d = 2 .. VPZ_RCP_MAX (d < 2: 0): floor(n / d) = umulhi(n, rcp[d]) exactly while n * d < 2^32 --
  // the floor-1 line arithmetic (RenderPoint, RenderLineMulti) divides by post distances only
  uint32_t rcp_off;
};
#define VPZ_RCP_MAX 4096
#define K1A_SM_WORDS 16384    // 64 KB of tables per CTA
#define K1A_SM_NONE 0xffffu

// ---- per-packet descriptors ------------------------------------------------------------
// K1 input: where the packet bytes are and where its spectrum goes.
struct alignas(16) VpzPktIn {
  uint32_t byte_off;        // into the batch byte buffer; packet is followed by >= 12 zero bytes
  uint32_t byte_len;
  uint32_t spec_off;        // float offset of [channels][n/2] in the spectrum buffer
  uint32_t setup_slot;      // index into the batch's setup pointer table
  uint32_t rec_off;         // word offset of the packet's symbol record (K1a -> K1b)
  uint32_t ent_off;         // uint16 offset of the packet's VQ entry indices; room for 8 * byte_len + 8
  uint32_t pad[2];
};

// K1 output / K3 input.
struct VpzPktRes {
  uint8_t exec_mask;        // bit ch set: channel has its own floor energy -> IMDCT runs (Mapping.cs:185)
  uint8_t status;           // 0 ok, 1 residue decode hit end of packet (kept what was decoded)
  // Spectrum bins >= 16 * end16[ch] of channel ch (ch < 2) are an exact +0 and were NOT written: the packet
  // codes nothing above its last active residue partition (typically 65 % of the bins of the TestFiles).
  // The 256 / 2048 IMDCT kernel reads only below it; 255 = everything was written (general K1b).
  uint8_t end16[2];
};

// K3 per-packet descriptor (host built from Mode.GetPacketInfo, Mode.cs:30-66)
struct alignas(16) VpzPktOla {
  uint32_t spec_off;        // as VpzPktIn
  uint32_t out_off;         // sample offset (per channel) inside the stream's output region
  uint16_t left_start, right_start;   // right_start already EOS-trimmed (StreamDecoder.cs:658-666)
  uint16_t right_end;
  uint8_t flags;            // bit0 long block, bit1 left slope uses size1 (LeftUseSize1), bit2 no output (first after reset)
  uint8_t pad;
};
#define VPZ_OLA_LONG 1
#define VPZ_OLA_LEFT1 2
#define VPZ_OLA_NOOUT 4

// K3 work item: a run of consecutive packets of one stream.
struct VpzOlaItem {
  uint32_t first_pkt;       // index into the batch packet arrays
  uint32_t n_pkts;          // packets that emit output
  uint32_t has_pre;         // 1: packet first_pkt-1 belongs to the same stream and seeds the carry
  uint32_t setup_slot;
  uint64_t out_base;        // float offset of the stream's output region in the batch PCM buffer
};
// No overlap state lives on the device between batches: the host re-submits the last valid
// packet of a stream as the "pre" packet of its next batch (it is decoded again and only seeds
// the carry), which is also exactly how SeekTo pre-roll works (StreamDecoder.cs:817-880).

// ---- K0: physical Ogg page scan on the device (k0_pages.cuh) -----------------------------------------------
struct VpzScanFile {
  uint64_t data_off;        // of the container image in the staged byte buffer (>= 4 readable bytes follow it)
  uint32_t len;
  uint32_t page_base;       // first record of this file in the page array
  uint32_t page_cap;        // records the file may use
  uint32_t pad;
};
struct alignas(16) VpzPageRec {   // one valid page (PageReaderBase.VerifyPage passed), 32 bytes
  uint32_t offset;          // of the page in its file image
  uint32_t body_len;
  uint32_t granule_lo, granule_hi;
  uint32_t serial, seq;
  uint8_t flags;            // 1 continuation, 2 BOS, 4 EOS
  uint8_t nseg;
  uint8_t is_resync;        // bytes were skipped in front of this page
  uint8_t is_continued;     // the last lacing value is 255
  uint16_t packet_count;    // PageHeader.GetPacketCount (Ogg/PageHeader.cs:35-59)
  uint16_t pad;
};
struct alignas(16) VpzCrcJob {    // fast path of K0: one page whose CRC is still to be checked
  uint32_t file, offset, length, pad;
};
struct alignas(16) VpzScanOut {
  uint32_t n_pages, crc_failures;
  uint32_t waste_lo, waste_hi;   // bytes that belong to no valid page
  uint32_t overflow;             // 1: page_cap was too small, the records are incomplete
  uint32_t pad[3];
};

// ---- K0g: page-end granule index on the device (k0_pages.cuh) -------------------------------------------------
struct VpzGranFile {        // one container image holding one clean logical stream
  uint64_t data_off;        // of the image in the staged byte buffer (the K0 scan's)
  uint32_t page_base;       // first page record / first index entry of the file
  uint32_t n_pages;
  uint32_t mode_flags_lo, mode_flags_hi;   // bit m: mode m is a long block (Mode.cs:30-37)
  uint8_t mode_bits, log2_size0, log2_size1, nmodes;
  uint32_t pad;
};

// ---- K4: delivery of random-access excerpts (k4_deliver.cuh) -------------------------------------------------
struct VpzCopySeg {
  uint64_t src;             // float offset in the batch PCM buffer
  uint64_t dst;             // float offset in the group's output buffer (the caller's layout)
  uint32_t n;               // floats
  uint32_t pad;
};

// ---- K5: placement into the caller's device buffer (k5_place.cuh) -------------------------------------------
#define VPZ_TILE_SAMPLES 2048                  // samples per tile at most
#define VPZ_TILE_ZERO 0xffffffffffffffffull    // VpzPlaceTile.src of a tile of zeros
struct VpzPlaceTile {
  uint64_t src;             // float offset of the tile's first sample frame in the batch PCM, or VPZ_TILE_ZERO
  uint64_t base;            // element offset of the item in the destination
  uint64_t len;             // samples per channel of the item (channel stride of the planar layout)
  uint64_t first;           // first sample of the tile in the item
  uint32_t n;               // samples
  uint32_t ch;              // channels
};

// ---- K7: packet bytes of a corpus call gathered from the corpus's device-resident images (k7_gather.cuh) ------
#define VPZ_PIECE_MORE 0x80000000u             // VpzGatherPiece.len: the packet continues in the next piece
struct VpzGatherPiece {
  uint64_t src;             // byte offset of the piece in the corpus's images
  uint32_t dst;             // byte offset in the batch's packet-byte area (a packet's first piece: 16-byte aligned)
  uint32_t len;             // bytes | VPZ_PIECE_MORE when the packet's next piece follows (a packet over pages)
};

// ---- K6: rate and channel conversion into the caller's device buffer (k6_convert.cuh) ------------------------
// Output j of an item at source rate fi and output rate fo (fi / fo = o / n in lowest terms) reads the 2 width + 2
// source frames from floor(j o / n) - width on, weighted by phase j mod n of the rate pair's coefficient table.
enum { VPZ_MIX_KEEP = 0, VPZ_MIX_MEAN = 1, VPZ_MIX_DUP = 2 };
#define K6_SMEM_BUDGET 32768           // bytes of staged source a tile aims for (several CTAs per SM)
#define K6_MAX_OUTS 4096               // output samples per tile at most
#define K6_MAX_TAB_FLOATS (1u << 22)   // coefficient table of one rate pair at most
struct VpzConvTile {
  uint64_t src;             // float offset of the item's source frame 0 in the source buffer (interleaved fp32)
  int64_t s_first;          // first staged frame, relative to the item's frame 0 (frames outside [0, src_len): zeros)
  uint64_t base;            // element offset of the item in the destination
  uint64_t len;             // output samples per channel of the item (channel stride of the planar layout)
  uint64_t first;           // first output sample of the tile in the item
  const float* taps;        // coefficient table, [2 width + 2][n] (tap-major); NULL: equal rates, no filter
  uint32_t src_len;         // source frames of the item
  uint32_t span;            // frames staged
  uint32_t n;               // output samples of the tile
  uint32_t valid;           // of them computed from the source; the rest are zero (an excerpt's got)
  uint32_t ro, rn;          // o, n: fi / fo in lowest terms
  uint32_t width;
  uint32_t p0, r0;          // first output j0 of the tile: j0 mod n, (j0 * o) mod n
  uint8_t ch_src, ch_out;   // channels of the source and of the output
  uint8_t mix;              // VPZ_MIX_*
  uint8_t pad[5];
};
