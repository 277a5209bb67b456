// k7_gather.cuh -- K7: the packet bytes of a corpus call (vpz_corpus_excerpts_device), gathered on the device from the
// corpus's resident container images instead of being copied into pinned staging on the host and sent over PCIe.
//
// The host describes every committed packet by PIECES: one {image offset, batch offset, length} per page the packet
// lies on (one for almost every packet; a packet continued across pages has one per page, in order, all but the last
// flagged VPZ_PIECE_MORE).  One warp writes one packet's whole staged slot [dst, dst + ((len + 12 + 15) & ~15)) --
// the payload, then zeros -- which is byte for byte what batch_commit stages on the host (plan_run's layout: 16-byte
// aligned slots, at least 12 zero bytes behind each packet), so K1a reads the same bytes either way.  A lane builds
// 16 bytes of the slot and stores them with one 16-byte store.  Single-piece packets load the 5 aligned words that
// cover the lane's 16 source bytes and shift them into place (funnel shifts); words that start behind the packet's
// last byte are not loaded, so no read leaves the packet's own aligned words.
#pragma once
#include "k1_params.h"
#include "k3_imdct.cuh"   // VPZ_DEV, VPZ_LDG

#define K7_THREADS 256

// bytes [q, q + 4) of a packet as one little-endian word, bytes at or past `len` zero
VPZ_DEV uint32_t k7_mask(uint32_t w, int64_t left) {
  return left >= 4 ? w : left <= 0 ? 0u : (w & ((1u << (8 * (uint32_t)left)) - 1u));
}

// byte q of a packet of several pieces (piece i0 onward); 0 past its end
VPZ_DEV uint32_t k7_byte(const K7Params& P, uint32_t i0, uint32_t q) {
  for (uint32_t i = i0;; i++) {
    const VpzGatherPiece pc = P.pieces[i];
    const uint32_t n = pc.len & ~VPZ_PIECE_MORE;
    if (q < n) return P.images[pc.src + q];
    q -= n;
    if (!(pc.len & VPZ_PIECE_MORE)) return 0u;
  }
}

VPZ_DEV void k7_packet(const K7Params& P, uint32_t i0, uint32_t lane) {
  const VpzGatherPiece first = P.pieces[i0];
  uint32_t len = first.len & ~VPZ_PIECE_MORE;
  const bool multi = (first.len & VPZ_PIECE_MORE) != 0;
  if (multi)
    for (uint32_t i = i0 + 1;; i++) {
      const uint32_t l = P.pieces[i].len;
      len += l & ~VPZ_PIECE_MORE;
      if (!(l & VPZ_PIECE_MORE)) break;
    }
  const uint32_t chunks = (len + 12u + 15u) >> 4;
  uint4* __restrict__ out = reinterpret_cast<uint4*>(P.bytes + first.dst);
  const uint64_t end = first.src + len;   // one past the payload in the images
  for (uint32_t c = lane; c < chunks; c += 32u) {
    uint32_t w[4];
    if (!multi) {
      const uint64_t s = first.src + 16ull * c;
      const uint64_t a = s & ~3ull;
      const uint32_t sh = 8u * (uint32_t)(s & 3u);
      uint32_t v[5];
#pragma unroll
      for (int k = 0; k < 5; k++)
        v[k] = a + 4u * k < end ? VPZ_LDG(reinterpret_cast<const uint32_t*>(P.images + a + 4u * k)) : 0u;
#pragma unroll
      for (int k = 0; k < 4; k++) w[k] = k7_mask(__funnelshift_r(v[k], v[k + 1], sh), (int64_t)len - (16ll * c + 4 * k));
    } else {   // a packet over pages: byte by byte (a few packets per file)
#pragma unroll
      for (int k = 0; k < 4; k++) {
        uint32_t x = 0;
        for (uint32_t j = 0; j < 4; j++) {
          const uint32_t q = 16u * c + 4u * k + j;
          if (q < len) x |= k7_byte(P, i0, q) << (8 * j);
        }
        w[k] = x;
      }
    }
    out[c] = uint4{w[0], w[1], w[2], w[3]};
  }
}

// one warp per packet, grid-stride over the pieces: the warp of a packet's first piece writes the packet's slot
VPZ_DEV void k7_cta(const K7Params& P) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warps_per_cta = blockDim.x >> 5;
  const uint32_t nwarps = gridDim.x * warps_per_cta;
  for (uint32_t i = blockIdx.x * warps_per_cta + (threadIdx.x >> 5); i < P.n_pieces; i += nwarps) {
    if (i > 0 && (P.pieces[i - 1].len & VPZ_PIECE_MORE)) continue;   // a later piece of a packet another warp writes
    k7_packet(P, i, lane);
  }
}
