// k6_convert.cuh -- K6: converts decoded PCM to one sample rate and channel layout on its way into the caller's
// device buffer (vpz_decode_files_device_conv, vpz_decode_excerpts_device_conv).
//
// The source of an item is contiguous interleaved fp32: its run in the batch PCM (files, clipped by K3) or its
// source window in the slot's scratch (excerpts, placed and clipped there by K5).  The host cuts every converted
// item into TILES of consecutive output samples whose staged source span fits a fixed shared-memory budget.  One
// CTA converts one tile:
//   1. stage the span channel-major in shared memory with aligned 16-byte loads (K5's chunking), zeros outside the
//      item's source frames; for a mono mix, add the channels in channel order and divide by C;
//   2. each lane computes K6_OUTS outputs of one channel, 32 apart, so that a warp covers consecutive outputs: at
//      equal rates the staged sample itself, otherwise the 2 width + 2 taps of the output's table row against the
//      staged frames, fp32 FMA; the table is tap-major, so the lanes' loads of one tap are adjacent;
//   3. store through K5's k5_dst / k5_put2 (interleaved or planar, fp32 or int16 by k3_s16).
// Outputs from `valid` on are zero.  Between them the tiles of a call write every element of the range once.
#pragma once
#include "k5_place.cuh"

#define K6_THREADS 256
#define K6_OUTS 4                   // outputs of one channel per lane (32 apart)

#ifdef VPZ_EMU
inline float k6_div(float a, float b) { return a / b; }
#else
__device__ __forceinline__ float k6_div(float a, float b) { return __fdiv_rn(a, b); }
#endif

// 1. the tile's span, channel-major: sm[c * span + f] = channel c of item frame s_first + f
VPZ_DEV void k6_stage(const float* __restrict__ src_all, const VpzConvTile& t, float* sm) {
  const uint32_t C = t.ch_src, span = t.span;
  const int64_t end = t.s_first + (int64_t)span;
  const int64_t lo = t.s_first > 0 ? t.s_first : 0;
  const int64_t hi = end < (int64_t)t.src_len ? end : (int64_t)t.src_len;
  const uint32_t f_lo = lo < hi ? (uint32_t)(lo - t.s_first) : span, f_hi = lo < hi ? (uint32_t)(hi - t.s_first) : span;
  for (uint32_t f = threadIdx.x; f < span; f += blockDim.x)
    if (f < f_lo || f >= f_hi)
      for (uint32_t c = 0; c < C; c++) sm[c * span + f] = 0.f;
  if (f_lo >= f_hi) return;
  const float* src = src_all + t.src + (uint64_t)lo * C;
  const uint32_t nel = (f_hi - f_lo) * C;
  const uint32_t head = (uint32_t)(reinterpret_cast<uintptr_t>(src) >> 2) & 3u;
  const float4* __restrict__ q = reinterpret_cast<const float4*>(src - head);
  const uint32_t nq = (head + nel + 3u) >> 2;
  for (uint32_t k0 = threadIdx.x; k0 < nq; k0 += blockDim.x * K5_UNROLL) {
    float4 v[K5_UNROLL];
#pragma unroll
    for (int u = 0; u < K5_UNROLL; u++)
      if (k0 + blockDim.x * u < nq) v[u] = VPZ_LDG(q + k0 + blockDim.x * u);
#pragma unroll
    for (int u = 0; u < K5_UNROLL; u++) {
      const uint32_t k = k0 + blockDim.x * u;
      if (k >= nq) break;
      const float f4[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const int e = (int)(4u * k) + i - (int)head;
        if (e < 0 || (uint32_t)e >= nel) continue;
        const uint32_t fr = C == 1 ? (uint32_t)e : C == 2 ? (uint32_t)e >> 1 : (uint32_t)e / C;
        sm[((uint32_t)e - fr * C) * span + f_lo + fr] = f4[i];
      }
    }
  }
}

template <bool OUT16, bool PLANAR>
VPZ_DEV void k6_tile(const K6Params& P, const VpzConvTile& t, float* sm) {
  typedef typename K5Elem<OUT16>::T T;
  T* __restrict__ out = static_cast<T*>(P.out);
  const uint32_t C = t.ch_src, span = t.span;
  if (t.valid) {
    k6_stage(P.src, t, sm);
    __syncthreads();
    if (t.mix == VPZ_MIX_MEAN) {   // mono: the channels in channel order, then / C
      for (uint32_t f = threadIdx.x; f < span; f += blockDim.x) {
        float s = sm[f];
        for (uint32_t c = 1; c < C; c++) s = __fadd_rn(s, sm[c * span + f]);
        sm[C * span + f] = k6_div(s, (float)C);
      }
      __syncthreads();
    }
  }
  // 2. + 3.: a warp takes 32 x K6_OUTS consecutive outputs of one computed channel, lane l outputs l + 32 r: the lanes
  // read consecutive rows of the tap-major table (coalesced) and store consecutive samples
  const uint32_t nch = t.mix == VPZ_MIX_KEEP ? C : 1u;
  const uint32_t chunk = 32u * K6_OUTS;
  const uint32_t chunks = (t.n + chunk - 1) / chunk;
  const uint32_t ntaps = 2u * t.width + 2u;
  const uint32_t lane = threadIdx.x & 31u, nwarps = blockDim.x >> 5;
  VpzPlaceTile pt;
  pt.src = 0;
  pt.base = t.base;
  pt.len = t.len;
  pt.first = t.first;
  pt.n = t.n;
  pt.ch = t.ch_out;
  for (uint32_t w = threadIdx.x >> 5; w < nch * chunks; w += nwarps) {
    const uint32_t c = w / chunks, s0 = (w - c * chunks) * chunk + lane;
    const float* x = t.mix == VPZ_MIX_MEAN ? sm + C * span : sm + c * span;
    float y[K6_OUTS];
    if (!t.taps) {
#pragma unroll
      for (int r = 0; r < K6_OUTS; r++) {
        const uint32_t s = s0 + 32u * r;
        y[r] = s < t.valid ? x[s] : 0.f;
      }
    } else {
      // taps of output j0 + s start at staged frame floor((r0 + s o) / n); its table row is (p0 + s) mod n
      const float* xs[K6_OUTS];
      const float* tp[K6_OUTS];
#pragma unroll
      for (int r = 0; r < K6_OUTS; r++) {
        const uint32_t s = s0 + 32u * r;
        const bool ok = s < t.valid;
        xs[r] = ok ? x + (t.r0 + s * t.ro) / t.rn : x;
        tp[r] = t.taps + (ok ? (t.p0 + s) % t.rn : 0u);
        y[r] = 0.f;
      }
#pragma unroll 2
      for (uint32_t i = 0; i < ntaps; i++) {
#pragma unroll
        for (int r = 0; r < K6_OUTS; r++) y[r] = fmaf(VPZ_LDG(tp[r] + (size_t)i * t.rn), xs[r][i], y[r]);
      }
#pragma unroll
      for (int r = 0; r < K6_OUTS; r++)
        if (s0 + 32u * r >= t.valid) y[r] = 0.f;
    }
#pragma unroll
    for (int r = 0; r < K6_OUTS; r++) {
      const uint32_t s = s0 + 32u * r;
      if (s >= t.n) break;
      if (t.mix == VPZ_MIX_DUP) {   // the mono value in both output channels
        const uint64_t d = k5_dst<PLANAR>(pt, 2u * s);
        if (PLANAR) {
          out[d] = K5Elem<OUT16>::conv(y[r]);
          out[d + t.len] = K5Elem<OUT16>::conv(y[r]);
        } else {
          k5_put2<OUT16>(out, d, y[r], y[r]);
        }
      } else {
        out[k5_dst<PLANAR>(pt, s * t.ch_out + c)] = K5Elem<OUT16>::conv(y[r]);
      }
    }
  }
}

// one CTA per tile, grid-stride over the tiles; sm: P.smem_floats floats of shared memory
template <bool OUT16, bool PLANAR>
VPZ_DEV void k6_cta(const K6Params& P, float* sm) {
  for (uint32_t i = blockIdx.x; i < P.n_tiles; i += gridDim.x) {
    const VpzConvTile t = P.tiles[i];
    k6_tile<OUT16, PLANAR>(P, t, sm);
    __syncthreads();   // the next tile restages sm
  }
}
