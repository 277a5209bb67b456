// dev_emu_place.h -- TEST INFRASTRUCTURE ONLY: the parts of devapi.h that the device-output bulk calls add
// (vpz_decode_files_device / vpz_decode_excerpts_device), on top of cuda_emu.h.  The emulated build compiles this
// into the translation unit of csrc/reader.cpp, their only caller; the product build never sees it.
#pragma once
#include "cuda_emu.h"

#include "../../vorbispizza_b200/csrc/devapi.h"
#include "../../vorbispizza_b200/csrc/k5_place.cuh"

namespace vpz {
namespace dev {

// K5: the unmodified kernel body, two emulated CTAs of two warps grid-striding over the tiles
int launch_k5(const K5Params& p, Stream*, std::string&) {
  if (p.n_tiles == 0) return VPZ_OK;
  emu::launch(2, 64, 0, [&] {
    if (p.out16) {
      if (p.planar) k5_cta<true, true>(p); else k5_cta<true, false>(p);
    } else {
      if (p.planar) k5_cta<false, true>(p); else k5_cta<false, false>(p);
    }
  });
  return VPZ_OK;
}

// the emulator's device memory is host memory: any pointer passes, and there is no other stream to wait for
int check_device_ptr(const void*, int, std::string&) { return VPZ_OK; }
void event_record_external(Event* e, void*) { event_record(e, nullptr); }

}  // namespace dev
}  // namespace vpz
