// 64-bit additions to the execution-model emulator (cuda_emu.h) for the 1:N identification kernels of
// fedfr_b200/csrc/identify.cu: the xor shuffle of an unsigned long long and the 64-bit atomicMax.  Included right after
// cuda_emu.h by tests/test_identify.py's emulated build.  TEST INFRASTRUCTURE ONLY -- never shipped.
#pragma once

static inline unsigned long long __shfl_xor_sync(unsigned, unsigned long long v, int o) { return emu_shfl_exchange(v, o, -1); }
static inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v) {
  const unsigned long long o = *p;
  if (v > o) *p = v;
  return o;
}
