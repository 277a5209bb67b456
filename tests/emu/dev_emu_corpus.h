// dev_emu_corpus.h -- TEST INFRASTRUCTURE ONLY: the part of devapi.h that the corpus calls add (vpz_corpus_*: K7, the
// gather of packet bytes from the corpus's device images), on top of cuda_emu.h.  The emulated build compiles this
// into the translation unit of csrc/reader.cpp, where the corpus lives; the product build never sees it.
#pragma once
#include "cuda_emu.h"

#include "../../vorbispizza_b200/csrc/devapi.h"
#include "../../vorbispizza_b200/csrc/k7_gather.cuh"

namespace vpz {
namespace dev {

// K7: the unmodified kernel body, two emulated CTAs of two warps grid-striding over the pieces
int launch_k7(const K7Params& p, Stream*, std::string&) {
  if (p.n_pieces == 0) return VPZ_OK;
  emu::launch(2, 64, 0, [&] { k7_cta(p); });
  return VPZ_OK;
}

}  // namespace dev
}  // namespace vpz
