// naf_load.cuh -- unaligned 16-byte loads shared by the kernels that move decoded bytes (naf_text.cu, naf_export.cuh).
#pragma once
#include "cuda_compat.h"
#include <stdint.h>

namespace nk {

// 16 bytes from an arbitrarily aligned address: two aligned loads + funnel shifts (reads up to 31 bytes past p & ~15;
// every blob in the arena is followed by 32 bytes of slack).
__device__ __forceinline__ uint4 load16u(const uint8_t* p) {
    const uint32_t s = (uint32_t)((uintptr_t)p & 15);
    const uint4* q = (const uint4*)(p - s);
    const uint4 lo = q[0];
    if (s == 0) return lo;
    const uint4 hi = q[1];
    // barrel shifter over the 8 words: by two words, by one word, then by bytes
    const bool s2 = s & 8, s1 = s & 4;
    const uint32_t a0 = s2 ? lo.z : lo.x, a1 = s2 ? lo.w : lo.y, a2 = s2 ? hi.x : lo.z, a3 = s2 ? hi.y : lo.w, a4 = s2 ? hi.z : hi.x, a5 = s2 ? hi.w : hi.y;
    const uint32_t b0 = s1 ? a1 : a0, b1 = s1 ? a2 : a1, b2 = s1 ? a3 : a2, b3 = s1 ? a4 : a3, b4 = s1 ? a5 : a4;
    const uint32_t bs = (s & 3) * 8;
    const uint32_t o[4] = {__funnelshift_r(b0, b1, bs), __funnelshift_r(b1, b2, bs), __funnelshift_r(b2, b3, bs), __funnelshift_r(b3, b4, bs)};
    return make_uint4(o[0], o[1], o[2], o[3]);
}

}  // namespace nk
