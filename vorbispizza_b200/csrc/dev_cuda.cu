// dev_cuda.cu -- CUDA implementation of devapi.h: the sm_100a kernels and their launchers.
// This is the only device backend linked into libvpz.so; there is no CPU path.
#include <cuda_runtime.h>
#include <stdio.h>

#include <algorithm>

#include "../../include/vpz.h"
#include "devapi.h"
#include "k0_pages.cuh"
#include "k1_symbols.cuh"
#include "k3_streams.cuh"
#include "k4_deliver.cuh"
#include "k5_place.cuh"
#include "k6_convert.cuh"
#include "k7_gather.cuh"

// ---- kernels ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(K0_THREADS) vpz_k0_pages(K0Params P) {
  __shared__ uint32_t k0_smem[K0_SMEM_WORDS];
  k0_cta(P, k0_smem);
}
__global__ void __launch_bounds__(K0_THREADS) vpz_k0_walk(K0Params P) { k0_walk_cta(P); }
__global__ void __launch_bounds__(K0_THREADS) vpz_k0_crc(K0Params P) {
  __shared__ uint32_t k0_smem[K0_SMEM_WORDS];
  k0_crc_cta(P, k0_smem);
}

__global__ void __launch_bounds__(K0_THREADS) vpz_k0g_granules(K0gParams P) { k0g_cta(P); }

__global__ void __launch_bounds__(K4_THREADS) vpz_k4_deliver(K4Params P) { k4_cta(P); }

template <bool OUT16, bool PLANAR>
__global__ void __launch_bounds__(K5_THREADS) vpz_k5_place(K5Params P) { k5_cta<OUT16, PLANAR>(P); }

__global__ void __launch_bounds__(K7_THREADS) vpz_k7_gather(K7Params P) { k7_cta(P); }

template <bool OUT16, bool PLANAR>
__global__ void __launch_bounds__(K6_THREADS) vpz_k6_convert(K6Params P) {
  extern __shared__ float k6_smem[];
  k6_cta<OUT16, PLANAR>(P, k6_smem);
}

#ifndef K1A_MIN_CTAS
#define K1A_MIN_CTAS 8
#endif
template <bool DEBUG, bool FULL>
__global__ void __launch_bounds__(128, K1A_MIN_CTAS) vpz_k1a_symbols(K1Params P) {
  const int lane = threadIdx.x & 31;
  for (;;) {
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(P.counter, 32u);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (base >= P.n_pkts) break;
    const uint32_t i = base + lane;
    if (i < P.n_pkts) k1a_decode_packet<DEBUG, FULL>(P, P.order ? P.order[i] : i, reinterpret_cast<uint4*>(k1a_sm) + 2 * threadIdx.x,
                                                     k1a_sm + K1A_RING_BYTES(128) / 4 + threadIdx.x);
    __syncwarp();
  }
}

// the same walk with the first-level Huffman tables of the CTA's current (setup, block size) in shared memory
__global__ void __launch_bounds__(K1A_SM_THREADS, 2) vpz_k1a_symbols_sm(K1Params P) {
  __shared__ uint32_t s_ctl[2];
  k1a_sm_loop(P, s_ctl);
}

// gather path: one warp per packet
#ifndef K1B_MIN_CTAS
#define K1B_MIN_CTAS 9
#endif
template <bool DEBUG>
__global__ void __launch_bounds__(K1B_THREADS, K1B_MIN_CTAS) vpz_k1b_spectrum(K1Params P) {
  extern __shared__ uint32_t k1_smem[];
  k1b_gather_loop<DEBUG>(P, k1_smem);
}
// general path: one CTA per packet
template <bool DEBUG>
__global__ void __launch_bounds__(K1B_THREADS, 4) vpz_k1b_general(K1Params P) {
  extern __shared__ uint32_t k1_smem[];
  __shared__ uint32_t s_idx;
  k1b_general_loop<DEBUG>(P, k1_smem, &s_idx);
}

// generic block sizes / channel counts
template <bool OUT16>
__global__ void __launch_bounds__(128, 1) vpz_k3_imdct_ola(K3Params P, int ncb) {
  extern __shared__ float k3_smem[];
  k3_cta_loop<OUT16>(P, k3_smem, ncb);
}

// block sizes 256 / 2048, mono / stereo: one CTA per SM, up to 12 independent 64-thread workers
// ENDS: the spectra come from K1b (exec masks and written ends in P.res); false for caller-provided spectra
template <bool OUT16, bool ENDS>
__global__ void __launch_bounds__(K3_THREADS_PER_CH * K3S_MAX_GROUPS, 1) vpz_k3_streams(K3Params P) {
  extern __shared__ float k3_smem[];
  k3s_cta<OUT16, ENDS>(P, k3_smem);
}

namespace vpz {
namespace dev {

struct Stream {
  cudaStream_t s;
};
struct Event {
  cudaEvent_t e;
};

// per device (a process may hold contexts on several GPUs); the calling thread's current device is
// tracked here so that make_current costs nothing when it does not change
#define VPZ_MAX_DEVICES 64
static int g_sm_count[VPZ_MAX_DEVICES] = {0};
static size_t g_max_smem[VPZ_MAX_DEVICES] = {0};
static thread_local int t_device = -1;

// lets a kernel use all of the opt-in shared memory: the dynamic part may be what its static part leaves
template <typename F>
static void allow_max_smem(F func, int optin) {
  cudaFuncAttributes a;
  if (cudaFuncGetAttributes(&a, func) != cudaSuccess) return;
  cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)a.sharedSizeBytes);
}

static int fail(cudaError_t e, const char* what, std::string& err) {
  err = std::string(what) + ": " + cudaGetErrorString(e);
  return VPZ_E_CUDA;
}

int device_count() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

void make_current(int device) {
  if (device == t_device || device < 0) return;
  if (cudaSetDevice(device) == cudaSuccess) t_device = device; else cudaGetLastError();
}

int init(int device, int* resolved, std::string& err) {
  int n = device_count();
  if (n <= 0) {
    err = "no CUDA device visible (libvpz has no CPU path)";
    return VPZ_E_NO_DEVICE;
  }
  if (device < 0) {
    if (cudaGetDevice(&device) != cudaSuccess) device = 0;
  }
  if (device >= n || device >= VPZ_MAX_DEVICES) {
    err = "device index out of range";
    return VPZ_E_NO_DEVICE;
  }
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(e, "cudaSetDevice", err);
  t_device = device;
  if (resolved) *resolved = device;
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return fail(e, "cudaGetDeviceProperties", err);
  if (prop.major != 10) {
    err = std::string("device is sm_") + std::to_string(prop.major) + std::to_string(prop.minor) +
          "; libvpz is built for sm_100a only";
    return VPZ_E_NO_DEVICE;
  }
  g_sm_count[device] = prop.multiProcessorCount;
  g_max_smem[device] = prop.sharedMemPerBlockOptin;
  const int optin = (int)prop.sharedMemPerBlockOptin;   // function attributes are per device
  allow_max_smem(vpz_k1a_symbols_sm, optin);
  allow_max_smem(vpz_k1b_spectrum<false>, optin);
  allow_max_smem(vpz_k1b_spectrum<true>, optin);
  allow_max_smem(vpz_k1b_general<false>, optin);
  allow_max_smem(vpz_k1b_general<true>, optin);
  allow_max_smem(vpz_k3_imdct_ola<false>, optin);
  allow_max_smem(vpz_k3_imdct_ola<true>, optin);
  allow_max_smem(vpz_k3_streams<false, false>, optin);
  allow_max_smem(vpz_k3_streams<true, false>, optin);
  allow_max_smem(vpz_k3_streams<false, true>, optin);
  allow_max_smem(vpz_k3_streams<true, true>, optin);
  allow_max_smem(vpz_k6_convert<false, false>, optin);
  allow_max_smem(vpz_k6_convert<false, true>, optin);
  allow_max_smem(vpz_k6_convert<true, false>, optin);
  allow_max_smem(vpz_k6_convert<true, true>, optin);
  e = cudaGetLastError();
  if (e != cudaSuccess) return fail(e, "cudaFuncSetAttribute", err);
  return VPZ_OK;
}

int sm_count() { return t_device >= 0 ? g_sm_count[t_device] : 0; }
size_t max_smem_per_block() { return t_device >= 0 ? g_max_smem[t_device] : 0; }

void* alloc(size_t bytes, std::string& err) {
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes ? bytes : 1);
  if (e != cudaSuccess) {
    fail(e, "cudaMalloc", err);
    return nullptr;
  }
  return p;
}
void free(void* p) {
  if (p) cudaFree(p);
}
void* host_alloc(size_t bytes) {
  void* p = nullptr;
  // portable: pinned for every device, whichever context's thread allocated it; mapped: kernels may write
  // into it under the same address (K0's page records)
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
void host_free(void* p) {
  if (p) cudaFreeHost(p);
}

Stream* stream_create() {
  Stream* s = new Stream;
  if (cudaStreamCreateWithFlags(&s->s, cudaStreamNonBlocking) != cudaSuccess) {
    delete s;
    return nullptr;
  }
  return s;
}
void stream_destroy(Stream* s) {
  if (!s) return;
  cudaStreamDestroy(s->s);
  delete s;
}
int stream_sync(Stream* s, std::string& err) {
  cudaError_t e = cudaStreamSynchronize(s->s);
  if (e != cudaSuccess) return fail(e, "cudaStreamSynchronize", err);
  return VPZ_OK;
}

Event* event_create() {
  Event* e = new Event;
  if (cudaEventCreate(&e->e) != cudaSuccess) {
    delete e;
    return nullptr;
  }
  return e;
}
void event_destroy(Event* e) {
  if (!e) return;
  cudaEventDestroy(e->e);
  delete e;
}
void event_record(Event* e, Stream* s) { cudaEventRecord(e->e, s->s); }
void stream_wait_event(Stream* s, Event* e) { cudaStreamWaitEvent(s->s, e->e, 0); }
int event_sync(Event* e, std::string& err) {
  cudaError_t r = cudaEventSynchronize(e->e);
  return r == cudaSuccess ? VPZ_OK : fail(r, "cudaEventSynchronize", err);
}
float event_elapsed_ms(Event* a, Event* b) {
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, a->e, b->e) != cudaSuccess) {
    cudaGetLastError();
    return -1.f;
  }
  return ms;
}

static unsigned long long g_h2d_bytes = 0, g_d2h_bytes = 0;
unsigned long long transfer_bytes(int which) { return which ? g_d2h_bytes : g_h2d_bytes; }

int h2d(void* dst, const void* src, size_t bytes, Stream* s, std::string& err) {
  if (!bytes) return VPZ_OK;
  g_h2d_bytes += bytes;
  cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s->s);
  return e == cudaSuccess ? VPZ_OK : fail(e, "cudaMemcpyAsync H2D", err);
}
int d2h(void* dst, const void* src, size_t bytes, Stream* s, std::string& err) {
  if (!bytes) return VPZ_OK;
  g_d2h_bytes += bytes;
  cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s->s);
  return e == cudaSuccess ? VPZ_OK : fail(e, "cudaMemcpyAsync D2H", err);
}
int d2d(void* dst, const void* src, size_t bytes, Stream* s, std::string& err) {
  if (!bytes) return VPZ_OK;
  cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s->s);
  return e == cudaSuccess ? VPZ_OK : fail(e, "cudaMemcpyAsync D2D", err);
}
int fill(void* dst, int byte_value, size_t bytes, Stream* s, std::string& err) {
  if (!bytes) return VPZ_OK;
  cudaError_t e = cudaMemsetAsync(dst, byte_value, bytes, s->s);
  return e == cudaSuccess ? VPZ_OK : fail(e, "cudaMemsetAsync", err);
}

int launch_k0(const K0Params& p, Stream* s, std::string& err) {
  if (p.n_files == 0) return VPZ_OK;
  const unsigned warps = K0_THREADS / 32;
  unsigned grid = (unsigned)std::min<size_t>(((size_t)p.n_files + warps - 1) / warps, (size_t)8 * sm_count());
  vpz_k0_walk<<<grid, K0_THREADS, 0, s->s>>>(p);
  vpz_k0_crc<<<8 * sm_count(), K0_THREADS, 0, s->s>>>(p);   // as many warps as fit: the jobs are pages, not files
  K0Params q = p;
  q.only_irregular = 1;
  vpz_k0_pages<<<grid, K0_THREADS, 0, s->s>>>(q);           // a no-op pass over the flags when every file was regular
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? VPZ_OK : fail(e, "launch vpz_k0_walk / crc / pages", err);
}

int launch_k0g(const K0gParams& p, Stream* s, std::string& err) {
  if (p.n_files == 0) return VPZ_OK;
  const unsigned warps = K0_THREADS / 32;
  unsigned grid = (unsigned)std::min<size_t>(((size_t)p.n_files + warps - 1) / warps, (size_t)8 * sm_count());
  vpz_k0g_granules<<<grid, K0_THREADS, 0, s->s>>>(p);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? VPZ_OK : fail(e, "launch vpz_k0g_granules", err);
}

int launch_k4(const K4Params& p, Stream* s, std::string& err) {
  if (p.n_segs == 0) return VPZ_OK;
  const unsigned warps = K4_THREADS / 32;
  unsigned grid = (unsigned)std::min<size_t>(((size_t)p.n_segs + warps - 1) / warps, (size_t)8 * sm_count());
  vpz_k4_deliver<<<grid, K4_THREADS, 0, s->s>>>(p);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? VPZ_OK : fail(e, "launch vpz_k4_deliver", err);
}

int launch_k5(const K5Params& p, Stream* s, std::string& err) {
  if (p.n_tiles == 0) return VPZ_OK;
  const unsigned warps = K5_THREADS / 32;
  unsigned grid = (unsigned)std::min<size_t>(((size_t)p.n_tiles + warps - 1) / warps, (size_t)8 * sm_count());
  if (p.out16) {
    if (p.planar) vpz_k5_place<true, true><<<grid, K5_THREADS, 0, s->s>>>(p); else vpz_k5_place<true, false><<<grid, K5_THREADS, 0, s->s>>>(p);
  } else {
    if (p.planar) vpz_k5_place<false, true><<<grid, K5_THREADS, 0, s->s>>>(p); else vpz_k5_place<false, false><<<grid, K5_THREADS, 0, s->s>>>(p);
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? VPZ_OK : fail(e, "launch vpz_k5_place", err);
}

int launch_k7(const K7Params& p, Stream* s, std::string& err) {
  if (p.n_pieces == 0) return VPZ_OK;
  const unsigned warps = K7_THREADS / 32;
  unsigned grid = (unsigned)std::min<size_t>(((size_t)p.n_pieces + warps - 1) / warps, (size_t)8 * sm_count());
  vpz_k7_gather<<<grid, K7_THREADS, 0, s->s>>>(p);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? VPZ_OK : fail(e, "launch vpz_k7_gather", err);
}

int launch_k6(const K6Params& p, Stream* s, std::string& err) {
  if (p.n_tiles == 0) return VPZ_OK;
  const size_t smem = (size_t)p.smem_floats * 4;
  if (smem > max_smem_per_block()) {
    err = "vpz_k6_convert: a tile needs " + std::to_string(smem) + " bytes of shared memory";
    return VPZ_E_UNSUPPORTED;
  }
  const unsigned grid = (unsigned)std::min<size_t>(p.n_tiles, (size_t)8 * sm_count());
  if (p.out16) {
    if (p.planar) vpz_k6_convert<true, true><<<grid, K6_THREADS, smem, s->s>>>(p); else vpz_k6_convert<true, false><<<grid, K6_THREADS, smem, s->s>>>(p);
  } else {
    if (p.planar) vpz_k6_convert<false, true><<<grid, K6_THREADS, smem, s->s>>>(p); else vpz_k6_convert<false, false><<<grid, K6_THREADS, smem, s->s>>>(p);
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? VPZ_OK : fail(e, "launch vpz_k6_convert", err);
}

int check_device_ptr(const void* p, int device, std::string& err) {
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    err = std::string("destination: cudaPointerGetAttributes: ") + cudaGetErrorString(e);
    return VPZ_E_ARGUMENT;
  }
  if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) {
    err = a.type == cudaMemoryTypeHost ? "destination is pinned host memory, not device memory"
                                       : "destination is not CUDA device memory";
    return VPZ_E_ARGUMENT;
  }
  if (a.type == cudaMemoryTypeDevice && a.device != device) {
    err = "destination is memory of device " + std::to_string(a.device) + ", the context's device is " + std::to_string(device);
    return VPZ_E_ARGUMENT;
  }
  return VPZ_OK;
}

void event_record_external(Event* e, void* cuda_stream) { cudaEventRecord(e->e, static_cast<cudaStream_t>(cuda_stream)); }

int launch_k1a(const K1Params& p, bool debug, bool full, int blocks, Stream* s, std::string& err) {
  if (p.n_pkts == 0) return VPZ_OK;
  if (!debug && !full && p.k1a_smem) {
    const size_t smem = ((size_t)K1A_SM_WORDS + 128) * 4 + K1A_RING_BYTES(K1A_SM_THREADS);
    const unsigned grid = (unsigned)std::min<size_t>(((size_t)p.n_pkts + K1A_SM_THREADS - 1) / K1A_SM_THREADS, (size_t)2 * sm_count());
    vpz_k1a_symbols_sm<<<grid, K1A_SM_THREADS, smem, s->s>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      cudaFuncAttributes a;
      cudaFuncGetAttributes(&a, vpz_k1a_symbols_sm);
      char buf[256];
      snprintf(buf, sizeof(buf), "launch vpz_k1a_symbols_sm (grid %u, smem %zu, max dynamic %d, static %zu, regs %d, max threads %d)",
               grid, smem, a.maxDynamicSharedSizeBytes, a.sharedSizeBytes, a.numRegs, a.maxThreadsPerBlock);
      return fail(e, buf, err);
    }
    return VPZ_OK;
  }
  if (debug) {
    if (full) vpz_k1a_symbols<true, true><<<blocks, 128, K1A_RING_BYTES(128) + K1A_CLS_BYTES(128), s->s>>>(p); else vpz_k1a_symbols<true, false><<<blocks, 128, K1A_RING_BYTES(128) + K1A_CLS_BYTES(128), s->s>>>(p);
  } else {
    if (full) vpz_k1a_symbols<false, true><<<blocks, 128, K1A_RING_BYTES(128) + K1A_CLS_BYTES(128), s->s>>>(p); else vpz_k1a_symbols<false, false><<<blocks, 128, K1A_RING_BYTES(128) + K1A_CLS_BYTES(128), s->s>>>(p);
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? VPZ_OK : fail(e, "launch vpz_k1a_symbols", err);
}

int launch_k1b(const K1Params& p, bool debug, int blocks, int warps, Stream* s, std::string& err) {
  if (p.n_pkts == 0) return VPZ_OK;
  // gather path: smem_words_per_warp per warp; general path: per CTA
  size_t smem = (size_t)p.smem_words_per_warp * 4 * (p.gather_ok ? warps : 1) + (p.gather_ok ? 1024 : 0);  // + the dB table
  if (smem > max_smem_per_block()) {
    err = "K1b shared memory request exceeds the device limit";
    return VPZ_E_UNSUPPORTED;
  }
  if (p.gather_ok) {
    if (debug) vpz_k1b_spectrum<true><<<blocks, K1B_THREADS, smem, s->s>>>(p); else vpz_k1b_spectrum<false><<<blocks, K1B_THREADS, smem, s->s>>>(p);
  } else {
    if (debug) vpz_k1b_general<true><<<blocks, K1B_THREADS, smem, s->s>>>(p); else vpz_k1b_general<false><<<blocks, K1B_THREADS, smem, s->s>>>(p);
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? VPZ_OK : fail(e, "launch vpz_k1b_spectrum", err);
}

int launch_k3(const K3Params& p, int ncb, size_t smem_bytes, Stream* s, std::string& err) {
  if (p.n_items == 0) return VPZ_OK;
  if (smem_bytes > max_smem_per_block()) {
    err = "K3 shared memory request exceeds the device limit";
    return VPZ_E_UNSUPPORTED;
  }
  int threads = ncb * K3_THREADS_PER_CH;
  // persistent CTAs: enough to fill every SM, items are handed out by the counter
  unsigned grid = (unsigned)std::min<size_t>(p.n_items, (size_t)8 * sm_count());
  if (p.out16)
    vpz_k3_imdct_ola<true><<<grid, threads, smem_bytes, s->s>>>(p, ncb);
  else
    vpz_k3_imdct_ola<false><<<grid, threads, smem_bytes, s->s>>>(p, ncb);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? VPZ_OK : fail(e, "launch vpz_k3_imdct_ola", err);
}

int k3_streams_groups(size_t n_items) {
  // workers per CTA: as many as shared memory holds; small batches are spread over all SMs instead
  size_t fit = (max_smem_per_block() / 4 - K3S_TAB_FLOATS) / K3S_GROUP_FLOATS;
  size_t g = std::min<size_t>(K3S_MAX_GROUPS, fit);
  size_t per_sm = (n_items + (size_t)sm_count() - 1) / (size_t)std::max(sm_count(), 1);
  return (int)std::max<size_t>(1, std::min(g, per_sm));
}

int launch_k3_streams(const K3Params& p, Stream* s, std::string& err) {
  if (p.n_items == 0) return VPZ_OK;
  const int groups = k3_streams_groups(p.n_items);
  const size_t smem_bytes = ((size_t)K3S_TAB_FLOATS + (size_t)groups * K3S_GROUP_FLOATS) * 4;
  if (smem_bytes > max_smem_per_block()) {
    err = "K3 shared memory request exceeds the device limit";
    return VPZ_E_UNSUPPORTED;
  }
  unsigned grid = (unsigned)std::min<size_t>((p.n_items + groups - 1) / groups, (size_t)sm_count());
  const int threads = groups * K3_THREADS_PER_CH;
  if (p.res) {
    if (p.out16) vpz_k3_streams<true, true><<<grid, threads, smem_bytes, s->s>>>(p); else vpz_k3_streams<false, true><<<grid, threads, smem_bytes, s->s>>>(p);
  } else {
    if (p.out16) vpz_k3_streams<true, false><<<grid, threads, smem_bytes, s->s>>>(p); else vpz_k3_streams<false, false><<<grid, threads, smem_bytes, s->s>>>(p);
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? VPZ_OK : fail(e, "launch vpz_k3_streams", err);
}

}  // namespace dev
}  // namespace vpz
