// dev_emu_convert.h -- TEST INFRASTRUCTURE ONLY: the part of devapi.h that the converting device-output bulk calls
// add (vpz_decode_files_device_conv / vpz_decode_excerpts_device_conv), on top of cuda_emu.h.  The emulated build
// compiles this into the translation unit of csrc/reader.cpp, their only caller; the product build never sees it.
#pragma once
#include "cuda_emu.h"

#include "../../vorbispizza_b200/csrc/devapi.h"
#include "../../vorbispizza_b200/csrc/k6_convert.cuh"

namespace vpz {
namespace dev {

// K6: the unmodified kernel body, two emulated CTAs of 64 threads grid-striding over the tiles
int launch_k6(const K6Params& p, Stream*, std::string&) {
  if (p.n_tiles == 0) return VPZ_OK;
  emu::launch(2, 64, (size_t)p.smem_floats * 4, [&] {
    float* sm = static_cast<float*>(emu::t_block->smem);
    if (p.out16) {
      if (p.planar) k6_cta<true, true>(p, sm); else k6_cta<true, false>(p, sm);
    } else {
      if (p.planar) k6_cta<false, true>(p, sm); else k6_cta<false, false>(p, sm);
    }
  });
  return VPZ_OK;
}

}  // namespace dev
}  // namespace vpz
