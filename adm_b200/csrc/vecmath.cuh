// Device helpers for the memory-side kernels (GroupNorm family):
//   * packed fp32 arithmetic (sm_100 FFMA2 / FADD2 / FMUL2: two IEEE fp32 lanes per instruction, bit-identical to the
//     scalar ops, half the issue slots),
//   * bf16-pair <-> fp32-pair conversions,
//   * the counter-based dropout mask (role of torch.nn.functional.dropout in UNetBlock.forward,
//     /root/reference/unet/uncond_unet.py:200; the reference's Philox stream cannot be reproduced, so parity tests export
//     these masks to the oracle instead — engine.export_dropout_masks).
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace adm {

typedef unsigned long long f32x2;  // two fp32 lanes in one 64-bit register pair (lo = element 0)

__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 splat2(float x) { return pack2(x, x); }
__device__ __forceinline__ f32x2 ffma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ f32x2 fadd2(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 fmul2(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
// one 32-bit word holding two bf16 (element 0 in the low half) -> fp32 pair, and back (round to nearest even)
__device__ __forceinline__ f32x2 bf2_to_f2(uint32_t w) {
    return pack2(__uint_as_float(w << 16), __uint_as_float(w & 0xFFFF0000u));
}
__device__ __forceinline__ uint32_t f2_to_bf2(f32x2 v) {
    float lo, hi;
    unpack2(v, lo, hi);
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ f32x2 tanh2_fast(f32x2 h) {  // two SFU ops
    float lo, hi;
    unpack2(h, lo, hi);
    asm("tanh.approx.f32 %0, %0;" : "+f"(lo));
    asm("tanh.approx.f32 %0, %0;" : "+f"(hi));
    return pack2(lo, hi);
}

// ------------------------------------------------------------------------------------------------ dropout mask
// Stateless: keep(element) = hash(seed, vector index, lane) >= p * 2^32, where a "vector" is 8 consecutive channels of one
// pixel, vector index = (sample * HW + pixel) * (C / 8) + channel / 8 (32-bit, wraps).  Forward and backward regenerate the
// same mask from the same (seed, index).  The 64-bit seed is avalanche-mixed once per thread (DropCtx); per vector a
// two-round multiply-xorshift of the index gives `base`, and the 8 lanes are 8 multiplicative hashes of `base` — one IMAD
// and one compare per element.  Checked offline on 4 M vectors: per-lane rate p +- 4e-4, joint drop probability of any two
// lanes / neighbouring vectors / neighbouring seeds p^2 +- 2 %, drops-per-vector histogram binomial.
struct DropCtx {
    uint32_t s0, s1, thr;
    float keep;  // 1 / (1 - p)
};
__device__ __forceinline__ DropCtx drop_ctx(unsigned long long seed, float p) {
    unsigned long long z = seed * 0x9E3779B97F4A7C15ull;
    z ^= z >> 32;
    z *= 0xD6E8FEB86659FD93ull;
    z ^= z >> 32;
    DropCtx c;
    c.s0 = static_cast<uint32_t>(z);
    c.s1 = static_cast<uint32_t>(z >> 32);
    c.thr = p >= 1.f ? 0xFFFFFFFFu : static_cast<uint32_t>(static_cast<double>(p) * 4294967296.0);
    c.keep = __frcp_rn(1.f - p);
    return c;
}
__device__ __forceinline__ uint32_t drop_base(const DropCtx& c, uint32_t vec_index) {
    uint32_t h = (vec_index ^ c.s0) * 0x9E3779B1u;
    h = h ^ (h >> 15) ^ c.s1;
    h *= 0x85EBCA77u;
    h ^= h >> 13;
    return h;
}
__device__ __forceinline__ bool drop_keep(const DropCtx& c, uint32_t base, int lane) {
    constexpr uint32_t M[8] = {0x9E3779B1u, 0x85EBCA6Bu, 0xC2B2AE35u, 0x27D4EB2Fu,
                               0x165667B1u, 0xD3A2646Du, 0xFD7046C5u, 0xB55A4F09u};
    return base * M[lane] >= c.thr;
}
// keep-scales of the 8 channels of one vector: 0 or 1 / (1 - p)
__device__ __forceinline__ void dropout_scales(const DropCtx& c, uint32_t vec_index, float (&s)[8]) {
    const uint32_t base = drop_base(c, vec_index);
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] = drop_keep(c, base, j) ? c.keep : 0.f;
}
__device__ __forceinline__ void dropout_scales2(const DropCtx& c, uint32_t vec_index, f32x2 (&s)[4]) {
    const uint32_t base = drop_base(c, vec_index);
#pragma unroll
    for (int j = 0; j < 4; ++j)
        s[j] = pack2(drop_keep(c, base, 2 * j) ? c.keep : 0.f, drop_keep(c, base, 2 * j + 1) ? c.keep : 0.f);
}

}  // namespace adm
