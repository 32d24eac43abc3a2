// The order-preserving key of an fp32 score, shared by TAR@FAR and the ROC curve (verify.cu) and 1:N identification
// (identify.cu), so that the 1:1 and 1:N protocols order scores, fold -0.0 onto +0.0 and set NaN apart the same way.
// Kernel sources include it as "../../fedfr_b200/csrc/score_key.cuh", like dot_chain.cuh.
#pragma once

namespace pfc {

// Order-preserving key of an fp32 score given as its bits: larger score -> larger key; -0.0 and +0.0 -> one key.
// NaN -> 0, which no number maps to (0 is the key of the bit pattern 0xffffffff, itself a NaN).
__device__ __forceinline__ unsigned int tar_key(unsigned int u) {
  if ((u & 0x7fffffffu) > 0x7f800000u) return 0u;
  if ((u & 0x7fffffffu) == 0u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

}  // namespace pfc
