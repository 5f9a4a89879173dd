// tests/emu/cuda_emu_at.h -- TEST INFRASTRUCTURE: the few CUDA intrinsics the autotune_v1 kernels use beyond
// cuda_emu.h (warp votes, find-first-set, float division rounded to nearest, the float bits of the envelope maximum).
// Included after cuda_emu.h and before the kernel headers by tests/emu/emu_at_ragged.cpp.
#pragma once
#include "cuda_emu.h"

// full warps only (every kernel that votes runs whole warps)
static inline unsigned __ballot_sync(unsigned, int pred) {
    unsigned r = 0;
    for (int l = 0; l < 32; ++l) r |= (unsigned)(qd_emu::shfl_idx(pred ? 1 : 0, l) != 0) << l;
    return r;
}
static inline int __all_sync(unsigned m, int pred) { return __ballot_sync(m, pred) == 0xffffffffu; }
static inline int __ffs(unsigned v) { return __builtin_ffs((int)v); }
static inline float __fdiv_rn(float a, float b) { volatile float r = a / b; return r; }
static inline int atomicMax(int *p, int v) {
    int old = __atomic_load_n(p, __ATOMIC_SEQ_CST);
    while (old < v && !__atomic_compare_exchange_n(p, &old, v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST)) {}
    return old;
}
static inline int __float_as_int(float f) { int u; std::memcpy(&u, &f, 4); return u; }
