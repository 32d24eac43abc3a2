// The exact pair-score chain shared by the ROC histogram (roc.cu) and 1:1 template verification (verify.cu):
//     tmp = tmp + (double)fl32(a[k] * b[k])      k ascending: fp32 products, fp64 adds, no FMA
// Kernel sources include it as "../../fedfr_b200/csrc/dot_chain.cuh": that path resolves from csrc/ for nvcc and from
// tests/emu/ for the CPU emulation of the kernels, which compiles the .cu files outside this directory.
#pragma once

namespace pfc {

__device__ __forceinline__ double dot_chain(double tmp, const float* __restrict__ a, const float* __restrict__ b, int n) {
  for (int k = 0; k < n; ++k) tmp = __dadd_rn(tmp, (double)__fmul_rn(a[k], b[k]));
  return tmp;
}

}  // namespace pfc
