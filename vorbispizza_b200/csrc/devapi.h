// devapi.h -- the only place the host engine touches the device.  The product implements it with
// the CUDA runtime + the sm_100a kernels (dev_cuda.cu, no CPU fallback).  tests/emu/ implements
// the same interface with a thread-per-CUDA-thread emulator so that `pytest -m "not gpu"` can run
// the unmodified kernel source and the whole host engine on a box without a GPU; that emulator is
// test infrastructure and is never linked into libvpz.so.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <string>

#include "k1_params.h"

namespace vpz {
namespace dev {

struct Stream;  // opaque
struct Event;

// Selects the device (< 0: the calling thread's current one), checks that it is an sm_100 part and
// caches its properties; *resolved receives the device index.  0 or VPZ_E_NO_DEVICE / VPZ_E_CUDA
int init(int device, int* resolved, std::string& err);
// Makes `device` the calling thread's current CUDA device.  Every extern "C" entry point that touches
// the device calls this first: the current device is per host thread, and one process may hold
// contexts on several GPUs (include/vpz.h: "one context per GPU").
void make_current(int device);
int device_count();
int sm_count();                          // of the calling thread's current device (make_current)

void* alloc(size_t bytes, std::string& err);
void free(void* p);
void* host_alloc(size_t bytes);
void host_free(void* p);

Stream* stream_create();
void stream_destroy(Stream* s);
int stream_sync(Stream* s, std::string& err);

Event* event_create();
void event_destroy(Event* e);
void event_record(Event* e, Stream* s);
int event_sync(Event* e, std::string& err);
void stream_wait_event(Stream* s, Event* e);   // later work on s waits for e
float event_elapsed_ms(Event* a, Event* b);

int h2d(void* dst, const void* src, size_t bytes, Stream* s, std::string& err);
int d2h(void* dst, const void* src, size_t bytes, Stream* s, std::string& err);
int d2d(void* dst, const void* src, size_t bytes, Stream* s, std::string& err);
int fill(void* dst, int byte_value, size_t bytes, Stream* s, std::string& err);
unsigned long long transfer_bytes(int which);  // process-wide bytes copied so far: 0 host->device, 1 device->host

// Every launcher works on the slice of the batch its parameter block describes (p.order / p.n_pkts for
// K1, p.items / p.n_items for K3) and hands the work out through *p.counter, which the caller has
// zeroed on the same stream (one word per launch of a decode pass).
// K1a: one lane per packet, `blocks` CTAs of 128 threads; full = the variant that also walks floor 0
// and mappings with several submaps.  K1b: p.gather_ok ? one warp per packet, `blocks` CTAs of `warps`
// warps, dynamic shared memory = warps * smem_words_per_warp * 4 : one CTA per packet.
int launch_k1a(const K1Params& p, bool debug, bool full, int blocks, Stream* s, std::string& err);
int launch_k1b(const K1Params& p, bool debug, int blocks, int warps, Stream* s, std::string& err);
// K3, generic block sizes / channel counts: one CTA per work item, ncb channels side by side (64 threads each)
int launch_k3(const K3Params& p, int ncb, size_t smem_bytes, Stream* s, std::string& err);
// K3, block sizes 256 / 2048 and at most 2 channels: one CTA per SM of independent 64-thread workers
int launch_k3_streams(const K3Params& p, Stream* s, std::string& err);
// K0: physical Ogg page scan.  Three launches on s: the header-chain walk (one warp per image), the page CRCs of
// the files the walk accepted (one warp per page), the serial scan of the files either of them flagged.
int launch_k0(const K0Params& p, Stream* s, std::string& err);
// K0g: page-end granule index of scanned images, one warp per file
int launch_k0g(const K0gParams& p, Stream* s, std::string& err);
// K4: copy segments of decoded excerpts into the caller's layout, one warp per segment
int launch_k4(const K4Params& p, Stream* s, std::string& err);
// K5: tiles of the batch PCM into the caller's device buffer, one warp per tile
int launch_k5(const K5Params& p, Stream* s, std::string& err);
// K6: rate / channel conversion of tiles into the caller's device buffer, one CTA per tile, p.smem_floats * 4 bytes of
// dynamic shared memory (VPZ_E_UNSUPPORTED when that exceeds the device's limit)
int launch_k6(const K6Params& p, Stream* s, std::string& err);
// K7: packet bytes of a corpus call from the corpus's device images into the batch's packet-byte area, one warp per
// packet
int launch_k7(const K7Params& p, Stream* s, std::string& err);

// Caller-owned device memory (the *_device bulk calls): 0 when p is device or managed memory of `device`,
// VPZ_E_ARGUMENT (with the reason in err) for host, pinned or another device's memory
int check_device_ptr(const void* p, int device, std::string& err);
// Records e on the caller's cudaStream_t (NULL: the legacy default stream)
void event_record_external(Event* e, void* cuda_stream);
size_t max_smem_per_block();             // of the calling thread's current device

}  // namespace dev
}  // namespace vpz
