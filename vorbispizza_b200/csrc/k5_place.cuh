// k5_place.cuh -- K5: places decoded PCM into the caller's device buffer (vpz_decode_files_device,
// vpz_decode_excerpts_device).
//
// The batch PCM is interleaved fp32, run after run (K3's output).  The host cuts every item of the caller's
// layout (a file, an excerpt) into TILES of at most VPZ_TILE_SAMPLES samples: for a file, consecutive pieces of
// its run; for an excerpt, the copy segments of the reader replay (the same segments K4 moves) plus zero tiles
// for the samples the reader does not deliver.  One warp places one tile: aligned 16-byte loads of the
// interleaved source, then per element the destination in the caller's layout -- interleaved (the host calls'
// layout) or planar, channel c of item k at base_k + c * samples_k -- as fp32 or as 16-bit by K3's rule
// (k3_s16).  Between them the tiles of a call write every element of the destination range exactly once.
#pragma once
#include "k1_params.h"
#include "k3_imdct.cuh"   // k3_s16, VPZ_DEV, VPZ_LDG

#define K5_THREADS 256
#define K5_UNROLL 4       // 16-byte loads a lane has in flight

template <bool OUT16>
struct K5Elem {
  typedef float T;
  static VPZ_DEV float conv(float v) { return v; }
};
template <>
struct K5Elem<true> {
  typedef int16_t T;
  static VPZ_DEV int16_t conv(float v) { return (int16_t)k3_s16(v); }
};

VPZ_DEV float k5_clip(float v, int clip) {   // Utils.ClipValue: NaN passes, like the reference's two comparisons
  if (clip) {
    if (v > 0.99999994f) v = 0.99999994f;
    if (v < -0.99999994f) v = -0.99999994f;
  }
  return v;
}

// destination element of element e (sample e / C, channel e % C) of a tile
template <bool PLANAR>
VPZ_DEV uint64_t k5_dst(const VpzPlaceTile& t, uint32_t e) {
  if (!PLANAR) return t.base + t.first * t.ch + e;
  const uint32_t s = t.ch == 2 ? e >> 1 : e / t.ch, c = t.ch == 2 ? e & 1u : e - s * t.ch;
  return t.base + (uint64_t)c * t.len + t.first + s;
}

// two adjacent elements at d, d + 1: one 8-byte (fp32) or 4-byte (s16) store when d is aligned for it
template <bool OUT16>
VPZ_DEV void k5_put2(typename K5Elem<OUT16>::T* out, uint64_t d, float a, float b) {
  typedef typename K5Elem<OUT16>::T T;
  T* p = out + d;
  if ((reinterpret_cast<uintptr_t>(p) & (2 * sizeof(T) - 1)) == 0) {
    if (OUT16)
      *reinterpret_cast<uint32_t*>(p) = ((uint32_t)k3_s16(a) & 0xffffu) | ((uint32_t)k3_s16(b) << 16);
    else
      *reinterpret_cast<float2*>(p) = float2{a, b};
  } else {
    p[0] = K5Elem<OUT16>::conv(a);
    p[1] = K5Elem<OUT16>::conv(b);
  }
}

template <bool OUT16, bool PLANAR>
VPZ_DEV void k5_tile(const K5Params& P, const VpzPlaceTile& t, uint32_t lane) {
  typedef typename K5Elem<OUT16>::T T;
  T* __restrict__ out = static_cast<T*>(P.out);
  const uint32_t nel = t.n * t.ch;
  if (t.src == VPZ_TILE_ZERO) {   // samples the reader does not deliver
    for (uint32_t e = lane; e < nel; e += 32u) out[k5_dst<PLANAR>(t, e)] = K5Elem<OUT16>::conv(0.f);
    return;
  }
  // 16-byte chunks over [src, src + nel): the first may start up to 3 floats before the tile and the last end up
  // to 3 floats behind it, inside the same aligned 16 bytes of the batch PCM buffer; those floats are not stored
  const float* src = P.pcm + t.src;
  const uint32_t head = (uint32_t)(reinterpret_cast<uintptr_t>(src) >> 2) & 3u;
  const float4* __restrict__ q = reinterpret_cast<const float4*>(src - head);
  const uint32_t nq = (head + nel + 3u) >> 2;
  // a stereo frame lies in one chunk when the tile starts on an even float: then a chunk is two samples of both
  // channels and splits into two row stores
  const bool pairs = PLANAR && t.ch == 2 && (head & 1u) == 0;
  const bool contiguous = !PLANAR || t.ch == 1;
  for (uint32_t k0 = lane; k0 < nq; k0 += 32u * K5_UNROLL) {
    float4 v[K5_UNROLL];
#pragma unroll
    for (int u = 0; u < K5_UNROLL; u++)
      if (k0 + 32u * u < nq) v[u] = VPZ_LDG(q + k0 + 32u * u);
#pragma unroll
    for (int u = 0; u < K5_UNROLL; u++) {
      const uint32_t k = k0 + 32u * u;
      if (k >= nq) break;
      const float x = k5_clip(v[u].x, P.clip), y = k5_clip(v[u].y, P.clip), z = k5_clip(v[u].z, P.clip),
                  w = k5_clip(v[u].w, P.clip);
      const int e0 = (int)(4u * k) - (int)head;   // tile element of v.x
      if (e0 >= 0 && (uint32_t)e0 + 4u <= nel && (contiguous || pairs)) {
        if (contiguous) {
          const uint64_t d = k5_dst<PLANAR>(t, (uint32_t)e0);
          k5_put2<OUT16>(out, d, x, y);
          k5_put2<OUT16>(out, d + 2, z, w);
        } else {
          const uint64_t d = k5_dst<PLANAR>(t, (uint32_t)e0);   // channel 0 of sample e0 / 2
          k5_put2<OUT16>(out, d, x, z);
          k5_put2<OUT16>(out, d + t.len, y, w);
        }
      } else {
        const float f[4] = {x, y, z, w};
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int e = e0 + i;
          if (e >= 0 && (uint32_t)e < nel) out[k5_dst<PLANAR>(t, (uint32_t)e)] = K5Elem<OUT16>::conv(f[i]);
        }
      }
    }
  }
}

// one warp per tile, grid-stride over the tiles
template <bool OUT16, bool PLANAR>
VPZ_DEV void k5_cta(const K5Params& P) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warps_per_cta = blockDim.x >> 5;
  const uint32_t nwarps = gridDim.x * warps_per_cta;
  for (uint32_t s = blockIdx.x * warps_per_cta + (threadIdx.x >> 5); s < P.n_tiles; s += nwarps) {
    const VpzPlaceTile t = P.tiles[s];
    k5_tile<OUT16, PLANAR>(P, t, lane);
  }
}
