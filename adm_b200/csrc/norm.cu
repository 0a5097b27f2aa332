// GroupNorm family on NHWC bf16 (HBM-bound), replacing torch.nn.functional.group_norm + silu + addcmul + dropout +
// the depthwise 2x2 resample of the reference (unet/uncond_unet.py:128, :191-200, :105-108).
//
//   K7  chan_sums      : per-(n, c) sum and sum-of-squares over H*W (optionally over a fused channel concat of two
//                        tensors).  Group statistics are derived from these on the fly by the consumers.
//   K7b gn_apply       : y = act(x * A[n,c] + B[n,c]) with A/B folding mean, rstd, gamma, beta and the adaptive
//                        (1 + scale), shift of UNetBlock; optional Philox dropout; optional 2x2 avg-pool / nearest-up
//                        fused into the store.
//   K8  gn_bwd_reduce  : S1[n,c] = sum_p dv, S2[n,c] = sum_p dv * xhat        (dv = grad at the pre-activation)
//       gn_bwd_params  : dgamma, dbeta, d(scale), d(shift) from S1/S2
//       gn_bwd_apply   : dx = rstd * (dv*g' - mean_g(dv*g') - xhat * mean_g(dv*g'*xhat)) (+ residual gradient)
//   plus col_sums (bias gradients), resample (skip path) and silu for the embedding MLP.
// All kernels process 8 channels (one 16-byte vector) per thread and keep a thread on a fixed channel vector so the
// per-channel partials live in registers.
#include "adm_internal.h"
#include <cuda_bf16.h>
#include <stdint.h>
#include <cooperative_groups.h>

#include "vecmath.cuh"

namespace cg = cooperative_groups;

namespace adm {

struct Vec8 {
    float v[8];
};
__device__ __forceinline__ Vec8 load8(const __nv_bfloat16* p) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    Vec8 r;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&w[i]);
        r.v[2 * i] = __bfloat162float(b.x);
        r.v[2 * i + 1] = __bfloat162float(b.y);
    }
    return r;
}
__device__ __forceinline__ void store8(__nv_bfloat16* p, const Vec8& r) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 b = __floats2bfloat162_rn(r.v[2 * i], r.v[2 * i + 1]);
        w[i] = *reinterpret_cast<const uint32_t*>(&b);
    }
    *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}

// sigmoid via the hardware tanh (1 MUFU op, no division): s = 0.5 * tanh(0.5 v) + 0.5; |err| ~ 2^-12, far below bf16.
__device__ __forceinline__ float sigmoid_fast(float v) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * v));
    return fmaf(t, 0.5f, 0.5f);
}
__device__ __forceinline__ float silu_f(float v) { return v * sigmoid_fast(v); }
__device__ __forceinline__ float silu_grad(float v) {
    const float s = sigmoid_fast(v);
    return fmaf(v * s, 1.f - s, s);
}
// full-precision variants for the fp32 embedding MLP
__device__ __forceinline__ float silu_precise(float v) { return v * __frcp_rn(1.f + __expf(-v)); }
__device__ __forceinline__ float silu_grad_precise(float v) {
    const float s = __frcp_rn(1.f + __expf(-v));
    return s * (1.f + v * (1.f - s));
}

__device__ __forceinline__ Vec8 unpack8(const uint4 u) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    Vec8 r;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        r.v[2 * i] = __uint_as_float(w[i] << 16);
        r.v[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
    }
    return r;
}
// tanh-form SiLU on a pre-halved pre-activation h = v/2:  silu(v) = h*tanh(h) + h,
// silu'(v) = 0.5 * (1 + T + h * (1 - T^2)), T = tanh(h).
__device__ __forceinline__ float tanh_fast(float h) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    return t;
}

static inline int threads_for(int nvec) {  // a multiple of nvec (threads keep a fixed channel vector), <= 256
    if (nvec >= 256) return 256;
    return nvec * (256 / nvec);
}

// ------------------------------------------------------------------------------------------------ gn_stats
// Pass 1 of GroupNorm: per-(n, c) sum / sum of squares (atomics into `sums`), and — in the LAST block of each sample
// (ticket counter) — the per-(n, c) coefficient table coef[n][c] = {A, B, mean, rstd} with y = x*A + B folding
// mean, rstd, gamma, beta and the adaptive (1 + scale), shift.  grid (chunks, N); blockDim is a multiple of V = C/8 so
// each thread stays on one channel vector and keeps its partials in registers.
__device__ __forceinline__ void gn_finish_coef(const float* __restrict__ sums, const float* __restrict__ gamma,
                                               const float* __restrict__ beta, const float* __restrict__ params,
                                               long long ldp, int n, int C, int G, int hw, float eps,
                                               float4* __restrict__ coef) {
    const int cpg = C / G;
    const float inv_cnt = 1.f / (static_cast<float>(cpg) * static_cast<float>(hw));
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int g = c / cpg;
        float s = 0.f, q = 0.f;
        for (int j = 0; j < cpg; ++j) {
            const float2 t = __ldcg(reinterpret_cast<const float2*>(sums) + (1LL * n * C + g * cpg + j));
            s += t.x;
            q += t.y;
        }
        const float mean = s * inv_cnt;
        const float var = fmaxf(q * inv_cnt - mean * mean, 0.f);
        const float rstd = rsqrtf(var + eps);
        const float ga = gamma[c], be = beta[c];
        float a = rstd * ga, b = be - mean * rstd * ga;
        if (params != nullptr) {
            const float sc = 1.f + params[n * ldp + c], sh = params[n * ldp + C + c];
            a *= sc;
            b = b * sc + sh;
        }
        coef[1LL * n * C + c] = make_float4(a, b, mean, rstd);
    }
}

__global__ void __launch_bounds__(256) gn_stats_kernel(const __nv_bfloat16* __restrict__ x1, int c1, long long ld1,
                                                       const __nv_bfloat16* __restrict__ x2, int c2, long long ld2,
                                                       int hw, float* __restrict__ sums, unsigned int* __restrict__ tickets,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       const float* __restrict__ params, long long ldp, int G, float eps,
                                                       float4* __restrict__ coef) {
    const int C = c1 + c2, V = C >> 3, V1 = c1 >> 3;
    const int n = blockIdx.y;
    const int tpv = blockDim.x / V;
    extern __shared__ float sm[];  // [blockDim][16]
    __shared__ int s_last;
    const int v = threadIdx.x % V, lane = threadIdx.x / V;
    float s[8], q[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
    if (lane < tpv) {
        const __nv_bfloat16* base = v < V1 ? x1 + 1LL * n * hw * ld1 + v * 8 : x2 + 1LL * n * hw * ld2 + (v - V1) * 8;
        const long long ld = v < V1 ? ld1 : ld2;
        const int step = gridDim.x * tpv;
        int p = blockIdx.x * tpv + lane;
        for (; p + 3 * step < hw; p += 4 * step) {  // 4 independent 16 B loads in flight
            const Vec8 a0 = load8(base + p * ld), a1 = load8(base + (p + step) * ld);
            const Vec8 a2 = load8(base + (p + 2 * step) * ld), a3 = load8(base + (p + 3 * step) * ld);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                s[i] += (a0.v[i] + a1.v[i]) + (a2.v[i] + a3.v[i]);
                q[i] += (a0.v[i] * a0.v[i] + a1.v[i] * a1.v[i]) + (a2.v[i] * a2.v[i] + a3.v[i] * a3.v[i]);
            }
        }
        for (; p < hw; p += step) {
            const Vec8 a = load8(base + p * ld);
#pragma unroll
            for (int i = 0; i < 8; ++i) { s[i] += a.v[i]; q[i] += a.v[i] * a.v[i]; }
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) { sm[threadIdx.x * 16 + i] = s[i]; sm[threadIdx.x * 16 + 8 + i] = q[i]; }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int vv = c >> 3, i = c & 7;
        float a = 0.f, b = 0.f;
        for (int l = 0; l < tpv; ++l) {
            a += sm[(l * V + vv) * 16 + i];
            b += sm[(l * V + vv) * 16 + 8 + i];
        }
        atomicAdd(sums + (1LL * n * C + c) * 2, a);
        atomicAdd(sums + (1LL * n * C + c) * 2 + 1, b);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(tickets + n, 1u) == gridDim.x - 1);
    __syncthreads();
    if (s_last) {
        __threadfence();
        gn_finish_coef(sums, gamma, beta, params, ldp, n, C, G, hw, eps, coef);
    }
}

// ------------------------------------------------------------------------------------------------ gn_apply (forward)
// y = act(x*A + B) (+ dropout) (+ 2x2 avg-pool / nearest-up on the store).  grid (chunks, N); blockDim is a multiple of
// V = C/8: a thread owns ONE channel vector (its 16 coefficients live in registers) and walks pixels with a fixed stride,
// so the inner loop has no integer division and consecutive threads touch consecutive 16 B chunks.
__global__ void __launch_bounds__(256, 4) gn_apply_kernel(const __nv_bfloat16* __restrict__ x1, int c1, long long ld1,
                                                       const __nv_bfloat16* __restrict__ x2, int c2, long long ld2,
                                                       int H, int W, const float4* __restrict__ coef, int act,
                                                       float drop_p, unsigned long long seed, int resample,
                                                       __nv_bfloat16* __restrict__ out, long long ldo,
                                                       const unsigned long long* __restrict__ seed_dev) {
    if (seed_dev != nullptr) seed += *seed_dev * 0x9E3779B97F4A7C15ull;
    const DropCtx dc = drop_ctx(seed, drop_p);
    const int C = c1 + c2, V = C >> 3, V1 = c1 >> 3;
    const int n = blockIdx.y, hw = H * W;
    const int tpv = blockDim.x / V;
    const int v = threadIdx.x % V, lane = threadIdx.x / V;
    if (lane >= tpv) return;
    float a[8], b[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 t = coef[1LL * n * C + v * 8 + j];
        a[j] = t.x;
        b[j] = t.y;
    }
    const __nv_bfloat16* base = v < V1 ? x1 + 1LL * n * hw * ld1 + v * 8 : x2 + 1LL * n * hw * ld2 + (v - V1) * 8;
    const long long ld = v < V1 ? ld1 : ld2;
    const int step = gridDim.x * tpv;
    if (resample == 1) {
        const int Ho = H / 2, Wo = W / 2;
        __nv_bfloat16* ob = out + 1LL * n * Ho * Wo * ldo + v * 8;
        for (int p = blockIdx.x * tpv + lane; p < Ho * Wo; p += step) {
            const int ho = p / Wo, wo = p - ho * Wo;
            Vec8 xv[4];
#pragma unroll
            for (int d = 0; d < 4; ++d) xv[d] = load8(base + ((2 * ho + (d >> 1)) * W + 2 * wo + (d & 1)) * ld);
            Vec8 o;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float acc = 0.f;
#pragma unroll
                for (int d = 0; d < 4; ++d) {
                    float y = xv[d].v[j] * a[j] + b[j];
                    if (act) y = silu_f(y);
                    acc += y;
                }
                o.v[j] = 0.25f * acc;
            }
            store8(ob + p * ldo, o);
        }
        return;
    }
    const int Wo = 2 * W;
    __nv_bfloat16* ob = out + 1LL * n * (resample == 2 ? 4 * hw : hw) * ldo + v * 8;
    const unsigned long long vec0 = 1ULL * n * hw * V + v;
    if (act) {  // silu(v) = h*tanh(h) + h with h = v/2: halve the coefficients once
#pragma unroll
        for (int j = 0; j < 8; ++j) { a[j] *= 0.5f; b[j] *= 0.5f; }
    }
    auto emit = [&](int pp, const uint4 raw) {
        const Vec8 xv = unpack8(raw);
        float ds[8];
        if (drop_p > 0.f) dropout_scales(dc, static_cast<uint32_t>(vec0 + 1ULL * pp * V), ds);
        Vec8 o;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float y = fmaf(xv.v[j], a[j], b[j]);
            if (act) y = fmaf(y, tanh_fast(y), y);
            if (drop_p > 0.f) y *= ds[j];
            o.v[j] = y;
        }
        if (resample == 0) {
            store8(ob + pp * ldo, o);
        } else {
            const int h = pp / W, w = pp - h * W;
#pragma unroll
            for (int d = 0; d < 4; ++d) store8(ob + (1LL * (2 * h + (d >> 1)) * Wo + 2 * w + (d & 1)) * ldo, o);
        }
    };
    // a pure stream: eight 16 B loads in flight per thread, then the math and the stores
    int p = blockIdx.x * tpv + lane;
    for (; p + 7 * step < hw; p += 8 * step) {
        uint4 raw[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) raw[u] = __ldcs(reinterpret_cast<const uint4*>(base + (p + u * step) * ld));
#pragma unroll
        for (int u = 0; u < 8; ++u) emit(p + u * step, raw[u]);
    }
    for (; p + 1 * step < hw; p += 2 * step) {
        const uint4 r0 = __ldcs(reinterpret_cast<const uint4*>(base + p * ld));
        const uint4 r1 = __ldcs(reinterpret_cast<const uint4*>(base + (p + step) * ld));
        emit(p, r0);
        emit(p + step, r1);
    }
    if (p < hw) emit(p, __ldcs(reinterpret_cast<const uint4*>(base + p * ld)));
}

// dv (gradient at the pre-activation v = x*A+B) for input pixel p (h, w), channel vector v.
__device__ __forceinline__ void grad_preact(const __nv_bfloat16* __restrict__ dyb, long long ldy, int H, int W, int p,
                                            int resample, int act, float drop_p, const DropCtx& dc,
                                            unsigned long long vec_index, const Vec8& xv, const float* a,
                                            const float* b, float (&dv)[8]) {
    Vec8 g;
    if (resample == 0) {
        g = load8(dyb + p * ldy);
    } else {
        const int h = p / W, w = p - h * W;
        if (resample == 1) {
            g = load8(dyb + ((h >> 1) * (W >> 1) + (w >> 1)) * ldy);
#pragma unroll
            for (int j = 0; j < 8; ++j) g.v[j] *= 0.25f;
        } else {
            Vec8 t[4];
#pragma unroll
            for (int d = 0; d < 4; ++d) t[d] = load8(dyb + (1LL * (2 * h + (d >> 1)) * (2 * W) + 2 * w + (d & 1)) * ldy);
#pragma unroll
            for (int j = 0; j < 8; ++j) g.v[j] = (t[0].v[j] + t[1].v[j]) + (t[2].v[j] + t[3].v[j]);
        }
    }
    float ds[8];
    if (drop_p > 0.f) dropout_scales(dc, static_cast<uint32_t>(vec_index), ds);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        float d = g.v[j];
        if (drop_p > 0.f) d *= ds[j];
        if (act) d *= silu_grad(xv.v[j] * a[j] + b[j]);
        dv[j] = d;
    }
}

// ------------------------------------------------------------------------------------------------ gn_bwd_reduce
// bsums [N][C][2]: S1 = sum_p dv, S2 = sum_p dv * xhat.  The last block of each sample turns them into
//   bcoef[n][c] = {K1, K2, K3, 0} with dx = dv*K1 + x*K2 + K3
//     (K1 = rstd*gamma', K2 = -rstd^2*M2, K3 = -rstd*M1 + mean*rstd^2*M2, gamma' = gamma (1 + scale),
//      M1 = mean_g(gamma' S1), M2 = mean_g(gamma' S2))
// and the parameter gradients: dgamma[c] += (1+sc) S2, dbeta[c] += (1+sc) S1, dparams[n] = (gamma S2 + beta S1 | S1).
__global__ void __launch_bounds__(256, 3) gn_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ dy, long long ldy,
                                                            const __nv_bfloat16* __restrict__ x1, int c1, long long ld1,
                                                            const __nv_bfloat16* __restrict__ x2, int c2, long long ld2,
                                                            int H, int W, int G, const float4* __restrict__ coef,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta,
                                                            const float* __restrict__ params, long long ldp, int act,
                                                            float drop_p, unsigned long long seed, int resample,
                                                            float* __restrict__ bsums, unsigned int* __restrict__ tickets,
                                                            float4* __restrict__ bcoef, float* __restrict__ dgamma,
                                                            float* __restrict__ dbeta, float* __restrict__ dparams,
                                                            long long ld_dparams,
                                                            const unsigned long long* __restrict__ seed_dev) {
    if (seed_dev != nullptr) seed += *seed_dev * 0x9E3779B97F4A7C15ull;
    const DropCtx dc = drop_ctx(seed, drop_p);
    extern __shared__ float sm[];
    __shared__ int s_last;
    const int C = c1 + c2, V = C >> 3, V1 = c1 >> 3;
    float* red = sm;  // [blockDim][16]
    const int n = blockIdx.y, hw = H * W;
    const int tpv = blockDim.x / V;
    const int v = threadIdx.x % V, lane = threadIdx.x / V;
    float s1[8], sx[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) s1[j] = sx[j] = 0.f;
    if (lane < tpv) {
        const __nv_bfloat16* base = v < V1 ? x1 + 1LL * n * hw * ld1 + v * 8 : x2 + 1LL * n * hw * ld2 + (v - V1) * 8;
        const long long ld = v < V1 ? ld1 : ld2;
        const int out_hw = resample == 1 ? hw / 4 : (resample == 2 ? hw * 4 : hw);
        const __nv_bfloat16* dyb = dy + 1LL * n * out_hw * ldy + v * 8;
        const unsigned long long vec0 = 1ULL * n * hw * V + v;
        float a[8], b[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 t = coef[1LL * n * C + v * 8 + j];
            a[j] = t.x; b[j] = t.y;
        }
        const int step = gridDim.x * tpv;
        int p = blockIdx.x * tpv + lane;
        for (; p + step < hw; p += 2 * step) {  // two pixels in flight
            const Vec8 xa = load8(base + p * ld), xb = load8(base + (p + step) * ld);
            float da[8], db[8];
            grad_preact(dyb, ldy, H, W, p, resample, act, drop_p, dc, vec0 + 1ULL * p * V, xa, a, b, da);
            grad_preact(dyb, ldy, H, W, p + step, resample, act, drop_p, dc, vec0 + 1ULL * (p + step) * V, xb, a, b, db);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                s1[j] += da[j] + db[j];
                sx[j] += da[j] * xa.v[j] + db[j] * xb.v[j];
            }
        }
        for (; p < hw; p += step) {
            const Vec8 xv = load8(base + p * ld);
            float dv[8];
            grad_preact(dyb, ldy, H, W, p, resample, act, drop_p, dc, vec0 + 1ULL * p * V, xv, a, b, dv);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                s1[j] += dv[j];
                sx[j] += dv[j] * xv.v[j];
            }
        }
        // S2 = sum dv * xhat = rstd * (sum dv*x - mean * sum dv)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 t = coef[1LL * n * C + v * 8 + j];
            sx[j] = t.w * (sx[j] - t.z * s1[j]);
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) { red[threadIdx.x * 16 + j] = s1[j]; red[threadIdx.x * 16 + 8 + j] = sx[j]; }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int vv = c >> 3, j = c & 7;
        float a = 0.f, b = 0.f;
        for (int l = 0; l < tpv; ++l) {
            a += red[(l * V + vv) * 16 + j];
            b += red[(l * V + vv) * 16 + 8 + j];
        }
        atomicAdd(bsums + (1LL * n * C + c) * 2, a);
        atomicAdd(bsums + (1LL * n * C + c) * 2 + 1, b);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(tickets + n, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // ---- per-sample epilogue (one block per sample): gamma' S1 / gamma' S2 into smem, then group means
    float* gs1 = sm;       // [C]
    float* gs2 = sm + C;   // [C]
    const int cpg = C / G;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const float2 t = __ldcg(reinterpret_cast<const float2*>(bsums) + (1LL * n * C + c));
        const float ga = gamma[c], be = beta[c];
        const float sc = params != nullptr ? 1.f + params[n * ldp + c] : 1.f;
        gs1[c] = ga * sc * t.x;
        gs2[c] = ga * sc * t.y;
        if (dgamma != nullptr) {
            atomicAdd(dgamma + c, sc * t.y);
            atomicAdd(dbeta + c, sc * t.x);
        }
        if (dparams != nullptr) {
            dparams[n * ld_dparams + c] = ga * t.y + be * t.x;
            dparams[n * ld_dparams + C + c] = t.x;
        }
    }
    __syncthreads();
    const float inv_cnt = 1.f / (static_cast<float>(cpg) * static_cast<float>(hw));
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int g = c / cpg;
        float m1 = 0.f, m2 = 0.f;
        for (int j = 0; j < cpg; ++j) { m1 += gs1[g * cpg + j]; m2 += gs2[g * cpg + j]; }
        m1 *= inv_cnt;
        m2 *= inv_cnt;
        const float sc = params != nullptr ? 1.f + params[n * ldp + c] : 1.f;
        const float4 t = coef[1LL * n * C + c];
        const float mean = t.z, rstd = t.w;
        bcoef[1LL * n * C + c] = make_float4(rstd * gamma[c] * sc, -rstd * rstd * m2, -rstd * m1 + mean * rstd * rstd * m2, 0.f);
    }
}

// ------------------------------------------------------------------------------------------------ gn_bwd_apply
// dx = dv*K1 + x*K2 + K3 (+ add).  add: optional skip-path gradient over the full channel range;
// add_mode 0: same resolution; 1: half resolution, spread as add/4; 2: double resolution, summed over the 2x2 patch.
// Same thread mapping as gn_apply (one channel vector per thread, coefficients in registers, no division in the loop).
__global__ void __launch_bounds__(256, 3) gn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ dy, long long ldy,
                                                           const __nv_bfloat16* __restrict__ x1, int c1, long long ld1,
                                                           const __nv_bfloat16* __restrict__ x2, int c2, long long ld2,
                                                           int H, int W, const float4* __restrict__ coef,
                                                           const float4* __restrict__ bcoef, int act, float drop_p,
                                                           unsigned long long seed, int resample,
                                                           const __nv_bfloat16* __restrict__ add, long long ldadd,
                                                           int add_mode, __nv_bfloat16* __restrict__ dx1, long long ldx1,
                                                           __nv_bfloat16* __restrict__ dx2, long long ldx2,
                                                           const unsigned long long* __restrict__ seed_dev) {
    if (seed_dev != nullptr) seed += *seed_dev * 0x9E3779B97F4A7C15ull;
    const DropCtx dc = drop_ctx(seed, drop_p);
    const int C = c1 + c2, V = C >> 3, V1 = c1 >> 3;
    const int n = blockIdx.y, hw = H * W;
    const int tpv = blockDim.x / V;
    const int v = threadIdx.x % V, lane = threadIdx.x / V;
    if (lane >= tpv) return;
    float a[8], b[8], k1[8], k2[8], k3[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 t = coef[1LL * n * C + v * 8 + j];
        const float4 u = bcoef[1LL * n * C + v * 8 + j];
        a[j] = t.x; b[j] = t.y;
        k1[j] = u.x; k2[j] = u.y; k3[j] = u.z;
    }
    const bool first = v < V1;
    const __nv_bfloat16* base = first ? x1 + 1LL * n * hw * ld1 + v * 8 : x2 + 1LL * n * hw * ld2 + (v - V1) * 8;
    const long long ld = first ? ld1 : ld2;
    __nv_bfloat16* ob = first ? dx1 + 1LL * n * hw * ldx1 + v * 8 : dx2 + 1LL * n * hw * ldx2 + (v - V1) * 8;
    const long long ldo = first ? ldx1 : ldx2;
    const int out_hw = resample == 1 ? hw / 4 : (resample == 2 ? hw * 4 : hw);
    const __nv_bfloat16* dyb = dy + 1LL * n * out_hw * ldy + v * 8;
    const int add_hw = add_mode == 1 ? hw / 4 : (add_mode == 2 ? hw * 4 : hw);
    const __nv_bfloat16* addb = add != nullptr ? add + 1LL * n * add_hw * ldadd + v * 8 : nullptr;
    const unsigned long long vec0 = 1ULL * n * hw * V + v;
    const int step = gridDim.x * tpv;
    for (int p = blockIdx.x * tpv + lane; p < hw; p += step) {
        const Vec8 xv = load8(base + p * ld);
        Vec8 addv;
        if (addb != nullptr) {  // issue the skip-gradient loads before the math
            if (add_mode == 0) {
                addv = load8(addb + p * ldadd);
            } else {
                const int h = p / W, w = p - h * W;
                if (add_mode == 1) {
                    addv = load8(addb + ((h >> 1) * (W >> 1) + (w >> 1)) * ldadd);
#pragma unroll
                    for (int j = 0; j < 8; ++j) addv.v[j] *= 0.25f;
                } else {
                    Vec8 t[4];
#pragma unroll
                    for (int d = 0; d < 4; ++d)
                        t[d] = load8(addb + (1LL * (2 * h + (d >> 1)) * (2 * W) + 2 * w + (d & 1)) * ldadd);
#pragma unroll
                    for (int j = 0; j < 8; ++j) addv.v[j] = (t[0].v[j] + t[1].v[j]) + (t[2].v[j] + t[3].v[j]);
                }
            }
        }
        float dv[8];
        grad_preact(dyb, ldy, H, W, p, resample, act, drop_p, dc, vec0 + 1ULL * p * V, xv, a, b, dv);
        Vec8 o;
#pragma unroll
        for (int j = 0; j < 8; ++j) o.v[j] = dv[j] * k1[j] + xv.v[j] * k2[j] + k3[j];
        if (addb != nullptr) {
#pragma unroll
            for (int j = 0; j < 8; ++j) o.v[j] += addv.v[j];
        }
        store8(ob + p * ldo, o);
    }
}

// ------------------------------------------------------------------------------------------------ col_sums (bias grad)
// out[c] += sum over rows of x[row][c]; x bf16 [rows][ld].  grid (chunks).
__global__ void __launch_bounds__(256) col_sums_kernel(const __nv_bfloat16* __restrict__ x, long long ld,
                                                       long long rows, int C_total, float* __restrict__ out,
                                                       const int* __restrict__ out_map) {
    extern __shared__ float sm[];  // [blockDim][8]
    const int col0 = blockIdx.y * 2048;
    const int C = min(2048, C_total - col0);
    x += col0;
    if (out_map != nullptr) out_map += col0; else out += col0;
    const int V = C >> 3;
    const int tpv = blockDim.x / V;
    const int v = threadIdx.x % V, lane = threadIdx.x / V;
    float s[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] = 0.f;
    if (lane < tpv && tpv > 0) {
        // four independent 16 B loads in flight per thread (a narrow tensor leaves few threads per row: one load at a time
        // kept ~18 KB per SM in flight, 1.4 TB/s)
        const long long stride = 1LL * gridDim.x * tpv;
        const __nv_bfloat16* px = x + v * 8;
        for (long long r = blockIdx.x * 1LL * tpv + lane; r < rows; r += 4 * stride) {
            uint4 raw[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                raw[u] = r + u * stride < rows ? __ldg(reinterpret_cast<const uint4*>(px + (r + u * stride) * ld))
                                               : make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t w[4] = {raw[u].x, raw[u].y, raw[u].z, raw[u].w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    s[2 * j] += __uint_as_float(w[j] << 16);
                    s[2 * j + 1] += __uint_as_float(w[j] & 0xFFFF0000u);
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) sm[threadIdx.x * 8 + j] = s[j];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float a = 0.f;
        for (int l = 0; l < tpv; ++l) a += sm[(l * V + (c >> 3)) * 8 + (c & 7)];
        atomicAdd(out + (out_map != nullptr ? out_map[c] : c), a);
    }
}

// out = a + b (+ c), bf16 rows of C channels with independent row strides.
__global__ void __launch_bounds__(256) add_bf16_kernel(const __nv_bfloat16* __restrict__ a, long long lda,
                                                       const __nv_bfloat16* __restrict__ b, long long ldb,
                                                       const __nv_bfloat16* __restrict__ c, long long ldc,
                                                       __nv_bfloat16* __restrict__ out, long long ldo, long long rows,
                                                       int C) {
    const int V = C >> 3;
    const unsigned total = static_cast<unsigned>(rows * V);  // < 2^31 vectors (checked by the launcher): 32-bit divisions
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const long long r = i / V;
        const int v = static_cast<int>(i % V);
        Vec8 x = load8(a + r * lda + v * 8);
        const Vec8 y = load8(b + r * ldb + v * 8);
#pragma unroll
        for (int j = 0; j < 8; ++j) x.v[j] += y.v[j];
        if (c != nullptr) {
            const Vec8 z = load8(c + r * ldc + v * 8);
#pragma unroll
            for (int j = 0; j < 8; ++j) x.v[j] += z.v[j];
        }
        store8(out + r * ldo + v * 8, x);
    }
}

// ------------------------------------------------------------------------------------------------ resample (skip path)
// mode 1: 2x2 average pool; mode 2: nearest x2.  NHWC bf16.
__global__ void __launch_bounds__(256) resample_kernel(const __nv_bfloat16* __restrict__ x, long long ldx, int N, int H,
                                                       int W, int C, int mode, __nv_bfloat16* __restrict__ out,
                                                       long long ldo) {
    const int V = C >> 3;
    const int Ho = mode == 1 ? H / 2 : H * 2, Wo = mode == 1 ? W / 2 : W * 2;
    // 32-bit index math (the launcher checks the element count): three 64-bit divisions per vector made this kernel
    // run at 1.1 TB/s
    const unsigned total = static_cast<unsigned>(N) * Ho * Wo * V;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int v = static_cast<int>(i % V);
        unsigned r = i / V;
        const int wo = static_cast<int>(r % Wo);
        r /= Wo;
        const int ho = static_cast<int>(r % Ho);
        const int n = static_cast<int>(r / Ho);
        Vec8 o;
        if (mode == 1) {
#pragma unroll
            for (int j = 0; j < 8; ++j) o.v[j] = 0.f;
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                const Vec8 t = load8(x + ((1LL * n * H + 2 * ho + (d >> 1)) * W + 2 * wo + (d & 1)) * ldx + v * 8);
#pragma unroll
                for (int j = 0; j < 8; ++j) o.v[j] += 0.25f * t.v[j];
            }
        } else {
            o = load8(x + ((1LL * n * H + (ho >> 1)) * W + (wo >> 1)) * ldx + v * 8);
        }
        store8(out + ((1LL * n * Ho + ho) * Wo + wo) * ldo + v * 8, o);
    }
}

// ------------------------------------------------------------------------------------------------ silu (embedding MLP)
__global__ void __launch_bounds__(256) silu_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                   __nv_bfloat16* __restrict__ y_bf16, long long n) {
    for (long long i = blockIdx.x * 1LL * blockDim.x + threadIdx.x; i < n; i += 1LL * gridDim.x * blockDim.x) {
        const float v = silu_precise(x[i]);
        if (y != nullptr) y[i] = v;
        if (y_bf16 != nullptr) y_bf16[i] = __float2bfloat16(v);
    }
}
__global__ void __launch_bounds__(256) silu_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy,
                                                       float* __restrict__ dx, __nv_bfloat16* __restrict__ dx_bf16,
                                                       long long n) {
    for (long long i = blockIdx.x * 1LL * blockDim.x + threadIdx.x; i < n; i += 1LL * gridDim.x * blockDim.x) {
        const float v = dy[i] * silu_grad_precise(x[i]);
        if (dx != nullptr) dx[i] = v;
        if (dx_bf16 != nullptr) dx_bf16[i] = __float2bfloat16(v);
    }
}


// ================================================================================================ fused cluster kernels
// One thread-block CLUSTER per sample (K = 1, 2, 4 or 8 CTAs; per-channel partials are exchanged through distributed
// shared memory), so the statistics pass and the apply pass of a GroupNorm live in ONE kernel separated by a cluster
// barrier instead of two kernels separated by a grid-wide dependency: no atomics, no memset, no ticket, and the second
// read of the sample comes from L2/L1.  Each thread owns one 8-channel vector (coefficients in registers) and streams
// its pixels through a private 4-deep cp.async ring in shared memory, so ~100 KB per SM are in flight without holding
// registers for them.  Used when the batch is large enough to fill the SMs (see gn_cluster_size); the multi-block
// kernels above remain the general path.
constexpr int GNF_STAGES = 4;

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(
                     static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst))),
                 "l"(gsrc)
                 : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__global__ void __launch_bounds__(512, 1) gn_fwd_fused_kernel(
    const __nv_bfloat16* __restrict__ x1, int c1, long long ld1, const __nv_bfloat16* __restrict__ x2, int c2,
    long long ld2, int H, int W, int G, float eps, const float* __restrict__ gamma, const float* __restrict__ beta,
    const float* __restrict__ params, long long ldp, float4* __restrict__ coef, int act, float drop_p,
    unsigned long long seed, int resample, __nv_bfloat16* __restrict__ out, long long ldo,
    const unsigned long long* __restrict__ seed_dev) {
    cg::cluster_group cluster = cg::this_cluster();
    const int K = static_cast<int>(cluster.num_blocks()), r = static_cast<int>(cluster.block_rank());
    if (seed_dev != nullptr) seed += *seed_dev * 0x9E3779B97F4A7C15ull;
    const DropCtx dc = drop_ctx(seed, drop_p);
    const int C = c1 + c2, V = C >> 3, V1 = c1 >> 3;
    const int n = blockIdx.x / K, hw = H * W;
    const int tpv = blockDim.x / V;
    const int v = threadIdx.x % V, lane = threadIdx.x / V;
    const bool active = lane < tpv;
    extern __shared__ __align__(16) float sm[];
    float* chan = sm;          // [2C] this CTA's per-channel (sum, sum of squares)
    float* tot = sm + 2 * C;   // [2C] cluster totals
    float* tabA = sm + 4 * C;  // [C]
    float* tabB = sm + 5 * C;  // [C]
    float* red = sm + 6 * C;   // [blockDim][16]; re-used as the cp.async ring [STAGES][blockDim] of uint4 in pass 2
    const __nv_bfloat16* base = v < V1 ? x1 + 1LL * n * hw * ld1 + v * 8 : x2 + 1LL * n * hw * ld2 + (v - V1) * 8;
    const long long ld = v < V1 ? ld1 : ld2;
    const int step = K * tpv;
    const int p0 = r * tpv + lane;
    // ---- pass 1: per-channel sums over this CTA's pixels (eight 16 B loads in flight per thread; packed fp32 math)
    {
        f32x2 s[4], q[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) s[i] = q[i] = 0ull;
        if (active) {
            const long long stride = step * ld;
            const __nv_bfloat16* px = base + p0 * ld;
            int p = p0;
            for (; p + 7 * step < hw; p += 8 * step) {
                uint4 raw[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) raw[u] = *reinterpret_cast<const uint4*>(px + u * stride);
                px += 8 * stride;
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const uint32_t w[4] = {raw[u].x, raw[u].y, raw[u].z, raw[u].w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const f32x2 t = bf2_to_f2(w[i]);
                        s[i] = fadd2(s[i], t);
                        q[i] = ffma2(t, t, q[i]);
                    }
                }
            }
            if (p < hw) {  // remainder (< 8 pixels; the WHOLE sample at 8x8 / 4x4): predicated, still all loads in flight
                uint4 raw[7];
#pragma unroll
                for (int u = 0; u < 7; ++u)
                    raw[u] = p + u * step < hw ? *reinterpret_cast<const uint4*>(px + u * stride) : make_uint4(0, 0, 0, 0);
#pragma unroll
                for (int u = 0; u < 7; ++u) {
                    const uint32_t w[4] = {raw[u].x, raw[u].y, raw[u].z, raw[u].w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const f32x2 t = bf2_to_f2(w[i]);
                        s[i] = fadd2(s[i], t);
                        q[i] = ffma2(t, t, q[i]);
                    }
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            unpack2(s[i], red[threadIdx.x * 16 + 2 * i], red[threadIdx.x * 16 + 2 * i + 1]);
            unpack2(q[i], red[threadIdx.x * 16 + 8 + 2 * i], red[threadIdx.x * 16 + 8 + 2 * i + 1]);
        }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int vv = c >> 3, i = c & 7;
        float a = 0.f, b = 0.f;
        for (int l = 0; l < tpv; ++l) {
            a += red[(l * V + vv) * 16 + i];
            b += red[(l * V + vv) * 16 + 8 + i];
        }
        chan[2 * c] = a;
        chan[2 * c + 1] = b;
    }
    cluster.sync();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float a = 0.f, b = 0.f;
        for (int rr = 0; rr < K; ++rr) {
            const float* rc = cluster.map_shared_rank(chan, rr);
            a += rc[2 * c];
            b += rc[2 * c + 1];
        }
        tot[2 * c] = a;
        tot[2 * c + 1] = b;
    }
    cluster.sync();  // every remote read of `chan` is done; also orders `tot` inside the CTA
    {
        const int cpg = C / G;
        const float inv_cnt = 1.f / (static_cast<float>(cpg) * static_cast<float>(hw));
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            const int g0 = (c / cpg) * cpg;
            float s = 0.f, q = 0.f;
            for (int j = 0; j < cpg; ++j) { s += tot[2 * (g0 + j)]; q += tot[2 * (g0 + j) + 1]; }
            const float mean = s * inv_cnt;
            const float var = fmaxf(q * inv_cnt - mean * mean, 0.f);
            const float rstd = rsqrtf(var + eps);
            const float ga = gamma[c], be = beta[c];
            float a = rstd * ga, b = be - mean * rstd * ga;
            if (params != nullptr) {
                const float sc = 1.f + params[n * ldp + c], sh = params[n * ldp + C + c];
                a *= sc;
                b = b * sc + sh;
            }
            tabA[c] = a;
            tabB[c] = b;
            if (r == 0) coef[1LL * n * C + c] = make_float4(a, b, mean, rstd);
        }
    }
    __syncthreads();
    if (!active) return;
    // ---- pass 2: y = act(x*A + B) (+ dropout) (+ resample on the store); second read of x hits L2
    float a[8], b[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { a[j] = tabA[v * 8 + j]; b[j] = tabB[v * 8 + j]; }
    if (resample == 1) {
        const int Ho = H / 2, Wo = W / 2;
        __nv_bfloat16* ob = out + 1LL * n * Ho * Wo * ldo + v * 8;
        for (int p = p0; p < Ho * Wo; p += step) {
            const int ho = p / Wo, wo = p - ho * Wo;
            Vec8 xv[4];
#pragma unroll
            for (int d = 0; d < 4; ++d) xv[d] = load8(base + ((2 * ho + (d >> 1)) * W + 2 * wo + (d & 1)) * ld);
            Vec8 o;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float acc = 0.f;
#pragma unroll
                for (int d = 0; d < 4; ++d) {
                    float y = xv[d].v[j] * a[j] + b[j];
                    if (act) y = silu_f(y);
                    acc += y;
                }
                o.v[j] = 0.25f * acc;
            }
            store8(ob + p * ldo, o);
        }
        return;
    }
    if (act) {  // halve the coefficients once: silu(v) = h*tanh(h) + h with h = v/2
#pragma unroll
        for (int j = 0; j < 8; ++j) { a[j] *= 0.5f; b[j] *= 0.5f; }
    }
    f32x2 a2[4], b2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { a2[j] = pack2(a[2 * j], a[2 * j + 1]); b2[j] = pack2(b[2 * j], b[2 * j + 1]); }
    const int Wo = 2 * W;
    __nv_bfloat16* ob = out + 1LL * n * (resample == 2 ? 4 * hw : hw) * ldo + v * 8;
    const uint32_t vec0 = static_cast<uint32_t>(1ULL * n * hw * V + v);
    uint4* ring = reinterpret_cast<uint4*>(red);  // [STAGES][blockDim]; `red` is dead (all threads passed the barriers)
    const long long stride = step * ld;
    const __nv_bfloat16* pfp = base + p0 * ld;  // prefetch cursor
    int pf = p0;
#pragma unroll
    for (int st = 0; st < GNF_STAGES; ++st) {
        if (pf < hw) cp_async16(ring + st * blockDim.x + threadIdx.x, pfp);
        cp_async_commit();
        pf += step;
        pfp += stride;
    }
    int st = 0;
    const long long ostride = 1LL * step * ldo;
    __nv_bfloat16* op = ob + p0 * ldo;
    uint32_t vec = vec0 + static_cast<uint32_t>(p0) * V;
    const uint32_t vstep = static_cast<uint32_t>(step) * V;
    for (int p = p0; p < hw; p += step) {
        cp_async_wait<GNF_STAGES - 1>();
        uint4* slot = ring + st * blockDim.x + threadIdx.x;
        const uint4 raw = *slot;
        if (pf < hw) cp_async16(slot, pfp);
        cp_async_commit();
        pf += step;
        pfp += stride;
        if (++st == GNF_STAGES) st = 0;
        const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
        f32x2 y[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            y[j] = ffma2(bf2_to_f2(w[j]), a2[j], b2[j]);
            if (act) y[j] = ffma2(y[j], tanh2_fast(y[j]), y[j]);
        }
        if (drop_p > 0.f) {
            f32x2 ds[4];
            dropout_scales2(dc, vec, ds);
#pragma unroll
            for (int j = 0; j < 4; ++j) y[j] = fmul2(y[j], ds[j]);
        }
        vec += vstep;
        const uint4 o = make_uint4(f2_to_bf2(y[0]), f2_to_bf2(y[1]), f2_to_bf2(y[2]), f2_to_bf2(y[3]));
        if (resample == 0) {
            *reinterpret_cast<uint4*>(op) = o;
            op += ostride;
        } else {
            const int h = p / W, w_ = p - h * W;
#pragma unroll
            for (int d = 0; d < 4; ++d)
                *reinterpret_cast<uint4*>(ob + (1LL * (2 * h + (d >> 1)) * Wo + 2 * w_ + (d & 1)) * ldo) = o;
        }
    }
}

// dv (gradient at the pre-activation) of one 8-channel vector in packed fp32: g = upstream gradient, x = GroupNorm input,
// ah/bh = coefficient pairs, pre-halved when act (h = v/2).  silu'(v) = s * (1 + h * Q) with T = tanh(h), s = (1 + T)/2
// (the sigmoid) and Q = 1 - T = 2 (1 - s).
__device__ __forceinline__ void dv_from2(const f32x2 (&g)[4], const f32x2 (&x)[4], const f32x2 (&ah)[4],
                                         const f32x2 (&bh)[4], int act, float drop_p, const DropCtx& dc, uint32_t vec,
                                         f32x2 (&dv)[4]) {
    f32x2 ds[4];
    if (drop_p > 0.f) dropout_scales2(dc, vec, ds);
    const f32x2 half = splat2(0.5f), one = splat2(1.f), neg1 = splat2(-1.f);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        f32x2 d = g[j];
        if (drop_p > 0.f) d = fmul2(d, ds[j]);
        if (act) {
            const f32x2 h = ffma2(x[j], ah[j], bh[j]);
            const f32x2 T = tanh2_fast(h);
            const f32x2 sg = ffma2(T, half, half);
            const f32x2 Q = ffma2(T, neg1, one);
            d = fmul2(d, fmul2(sg, ffma2(h, Q, one)));
        }
        dv[j] = d;
    }
}

// Backward twin: pass 1 = S1/S2 reduction, cluster exchange, parameter gradients and the {K1,K2,K3} table;
// pass 2 = dx (+ skip-path gradient `add`), optionally also the column sums of dx1 (the bias gradient of the conv
// that produced x1) accumulated into dbias1[c1].
__global__ void __launch_bounds__(512, 1) gn_bwd_fused_kernel(
    const __nv_bfloat16* __restrict__ dy, long long ldy, const __nv_bfloat16* __restrict__ x1, int c1, long long ld1,
    const __nv_bfloat16* __restrict__ x2, int c2, long long ld2, int H, int W, int G,
    const float4* __restrict__ coef, const float* __restrict__ gamma, const float* __restrict__ beta,
    const float* __restrict__ params, long long ldp, int act, float drop_p, unsigned long long seed, int resample,
    float* __restrict__ dgamma, float* __restrict__ dbeta, float* __restrict__ dparams, long long ld_dparams,
    const __nv_bfloat16* __restrict__ add, long long ldadd, int add_mode, __nv_bfloat16* __restrict__ dx1,
    long long ldx1, __nv_bfloat16* __restrict__ dx2, long long ldx2, float* __restrict__ dbias1,
    float* __restrict__ dbias1b, const unsigned long long* __restrict__ seed_dev, int dy_scratch) {
    cg::cluster_group cluster = cg::this_cluster();
    const int K = static_cast<int>(cluster.num_blocks()), r = static_cast<int>(cluster.block_rank());
    if (seed_dev != nullptr) seed += *seed_dev * 0x9E3779B97F4A7C15ull;
    const DropCtx dc = drop_ctx(seed, drop_p);
    const int C = c1 + c2, V = C >> 3, V1 = c1 >> 3;
    const int n = blockIdx.x / K, hw = H * W;
    const int tpv = blockDim.x / V;
    const int v = threadIdx.x % V, lane = threadIdx.x / V;
    const bool active = lane < tpv;
    extern __shared__ __align__(16) float sm[];
    float* chan = sm;          // [2C] this CTA's raw (sum dv, sum dv*x)
    float* tot = sm + 2 * C;   // [2C] cluster totals -> (gamma' S1, gamma' S2)
    float* tab = sm + 4 * C;   // [3C] k1, k2, k3
    float* red = sm + 7 * C;   // [blockDim][16] reduction scratch
    uint4* ring = reinterpret_cast<uint4*>(sm + 7 * C + 16 * blockDim.x);  // [STAGES][3][blockDim] cp.async ring
    const bool first = v < V1;
    const __nv_bfloat16* base = first ? x1 + 1LL * n * hw * ld1 + v * 8 : x2 + 1LL * n * hw * ld2 + (v - V1) * 8;
    const long long ld = first ? ld1 : ld2;
    const int out_hw = resample == 1 ? hw / 4 : (resample == 2 ? hw * 4 : hw);
    const __nv_bfloat16* dyb = dy + 1LL * n * out_hw * ldy + v * 8;
    const uint32_t vec0 = static_cast<uint32_t>(1ULL * n * hw * V + v);
    const int step = K * tpv;
    const int p0 = r * tpv + lane;
    const bool piped = resample == 0 && (add == nullptr || add_mode == 0);  // the common, fully pipelined shape
    // dy_scratch: the caller does not need dy afterwards.  Pass 1 then overwrites it with dv (the gradient at the
    // pre-activation, bf16) and pass 2 reads that back instead of re-deriving it: the SiLU derivative and the dropout hash
    // are evaluated once per element instead of twice (this kernel is instruction-issue bound, not DRAM bound).
    const bool reuse_dv = dy_scratch != 0 && piped && dx1 != nullptr && (act != 0 || drop_p > 0.f);
    float a[8], b[8];      // pre-activation coefficients (as stored)
    float ah[8], bh[8];    // halved when act (tanh-form SiLU); used by the pipelined path
    if (active) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 t = coef[1LL * n * C + v * 8 + j];
            a[j] = t.x;
            b[j] = t.y;
            ah[j] = act ? 0.5f * t.x : t.x;
            bh[j] = act ? 0.5f * t.y : t.y;
        }
    }
    f32x2 ah2[4], bh2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { ah2[j] = pack2(ah[2 * j], ah[2 * j + 1]); bh2[j] = pack2(bh[2 * j], bh[2 * j + 1]); }
    // ---- pass 1
    {
        float s1[8], sx[8];
        f32x2 s1p[4], sxp[4];  // the pipelined path accumulates in packed fp32
#pragma unroll
        for (int j = 0; j < 8; ++j) s1[j] = sx[j] = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) s1p[j] = sxp[j] = 0ull;
        if (active && piped) {
            const long long xstride = step * ld, gstride = step * ldy;
            const __nv_bfloat16* xpf = base + p0 * ld;
            const __nv_bfloat16* gpf = dyb + p0 * ldy;
            __nv_bfloat16* gst = const_cast<__nv_bfloat16*>(dyb) + p0 * ldy;  // dv goes where dy was (reuse_dv)
            uint32_t vec = vec0 + static_cast<uint32_t>(p0) * V;
            const uint32_t vstep = static_cast<uint32_t>(step) * V;
            int pf = p0;
#pragma unroll
            for (int st = 0; st < GNF_STAGES; ++st) {
                if (pf < hw) {
                    cp_async16(ring + (st * 3 + 0) * blockDim.x + threadIdx.x, xpf);
                    cp_async16(ring + (st * 3 + 1) * blockDim.x + threadIdx.x, gpf);
                }
                cp_async_commit();
                pf += step;
                xpf += xstride;
                gpf += gstride;
            }
            int st = 0;
            for (int p = p0; p < hw; p += step) {
                cp_async_wait<GNF_STAGES - 1>();
                uint4* sx_ = ring + (st * 3 + 0) * blockDim.x + threadIdx.x;
                uint4* sd_ = ring + (st * 3 + 1) * blockDim.x + threadIdx.x;
                const uint4 xr = *sx_, gr = *sd_;
                if (pf < hw) {
                    cp_async16(sx_, xpf);
                    cp_async16(sd_, gpf);
                }
                cp_async_commit();
                pf += step;
                xpf += xstride;
                gpf += gstride;
                if (++st == GNF_STAGES) st = 0;
                const uint32_t xw[4] = {xr.x, xr.y, xr.z, xr.w}, gw[4] = {gr.x, gr.y, gr.z, gr.w};
                f32x2 x2[4], g2[4], dv[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) { x2[j] = bf2_to_f2(xw[j]); g2[j] = bf2_to_f2(gw[j]); }
                dv_from2(g2, x2, ah2, bh2, act, drop_p, dc, vec, dv);
                vec += vstep;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    s1p[j] = fadd2(s1p[j], dv[j]);
                    sxp[j] = ffma2(dv[j], x2[j], sxp[j]);
                }
                if (reuse_dv) {
                    *reinterpret_cast<uint4*>(gst) =
                        make_uint4(f2_to_bf2(dv[0]), f2_to_bf2(dv[1]), f2_to_bf2(dv[2]), f2_to_bf2(dv[3]));
                    gst += gstride;
                }
            }
            cp_async_wait<0>();
        } else if (active) {
            for (int p = p0; p < hw; p += step) {
                const Vec8 xv = load8(base + p * ld);
                float dv[8];
                grad_preact(dyb, ldy, H, W, p, resample, act, drop_p, dc, vec0 + 1ULL * p * V, xv, a, b, dv);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    s1[j] += dv[j];
                    sx[j] += dv[j] * xv.v[j];
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float lo, hi;
            unpack2(s1p[j], lo, hi);
            s1[2 * j] += lo;
            s1[2 * j + 1] += hi;
            unpack2(sxp[j], lo, hi);
            sx[2 * j] += lo;
            sx[2 * j + 1] += hi;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) { red[threadIdx.x * 16 + j] = s1[j]; red[threadIdx.x * 16 + 8 + j] = sx[j]; }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int vv = c >> 3, j = c & 7;
        float s = 0.f, q = 0.f;
        for (int l = 0; l < tpv; ++l) {
            s += red[(l * V + vv) * 16 + j];
            q += red[(l * V + vv) * 16 + 8 + j];
        }
        chan[2 * c] = s;
        chan[2 * c + 1] = q;
    }
    cluster.sync();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float s = 0.f, q = 0.f;
        for (int rr = 0; rr < K; ++rr) {
            const float* rc = cluster.map_shared_rank(chan, rr);
            s += rc[2 * c];
            q += rc[2 * c + 1];
        }
        const float4 t = coef[1LL * n * C + c];
        const float S1 = s, S2 = t.w * (q - t.z * s);  // sum dv*xhat = rstd * (sum dv*x - mean * sum dv)
        const float ga = gamma[c], be = beta[c];
        const float sc = params != nullptr ? 1.f + params[n * ldp + c] : 1.f;
        tot[2 * c] = ga * sc * S1;
        tot[2 * c + 1] = ga * sc * S2;
        if (r == 0) {
            if (dgamma != nullptr) {
                atomicAdd(dgamma + c, sc * S2);
                atomicAdd(dbeta + c, sc * S1);
            }
            if (dparams != nullptr) {
                dparams[n * ld_dparams + c] = ga * S2 + be * S1;
                dparams[n * ld_dparams + C + c] = S1;
            }
        }
    }
    cluster.sync();
    if (dx1 == nullptr) return;
    {
        const int cpg = C / G;
        const float inv_cnt = 1.f / (static_cast<float>(cpg) * static_cast<float>(hw));
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            const int g0 = (c / cpg) * cpg;
            float m1 = 0.f, m2 = 0.f;
            for (int j = 0; j < cpg; ++j) { m1 += tot[2 * (g0 + j)]; m2 += tot[2 * (g0 + j) + 1]; }
            m1 *= inv_cnt;
            m2 *= inv_cnt;
            const float sc = params != nullptr ? 1.f + params[n * ldp + c] : 1.f;
            const float4 t = coef[1LL * n * C + c];
            const float mean = t.z, rstd = t.w;
            tab[c] = rstd * gamma[c] * sc;
            tab[C + c] = -rstd * rstd * m2;
            tab[2 * C + c] = -rstd * m1 + mean * rstd * rstd * m2;
        }
    }
    __syncthreads();
    // ---- pass 2
    float bs[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) bs[j] = 0.f;
    if (active) {
        float k1[8], k2[8], k3[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            k1[j] = tab[v * 8 + j];
            k2[j] = tab[C + v * 8 + j];
            k3[j] = tab[2 * C + v * 8 + j];
        }
        __nv_bfloat16* ob = first ? dx1 + 1LL * n * hw * ldx1 + v * 8 : dx2 + 1LL * n * hw * ldx2 + (v - V1) * 8;
        const long long ldo = first ? ldx1 : ldx2;
        const int add_hw = add_mode == 1 ? hw / 4 : (add_mode == 2 ? hw * 4 : hw);
        const __nv_bfloat16* addb = add != nullptr ? add + 1LL * n * add_hw * ldadd + v * 8 : nullptr;
        const bool want_bs = dbias1 != nullptr && first;
        if (piped) {
            f32x2 k1p[4], k2p[4], k3p[4], bsp[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                k1p[j] = pack2(k1[2 * j], k1[2 * j + 1]);
                k2p[j] = pack2(k2[2 * j], k2[2 * j + 1]);
                k3p[j] = pack2(k3[2 * j], k3[2 * j + 1]);
                bsp[j] = 0ull;
            }
            const long long xstride = step * ld, gstride = step * ldy, ostride = step * ldo;
            const long long astride = addb != nullptr ? step * ldadd : 0;
            const __nv_bfloat16* xpf = base + p0 * ld;
            const __nv_bfloat16* gpf = dyb + p0 * ldy;
            const __nv_bfloat16* apf = addb != nullptr ? addb + p0 * ldadd : nullptr;
            __nv_bfloat16* op = ob + p0 * ldo;
            uint32_t vec = vec0 + static_cast<uint32_t>(p0) * V;
            const uint32_t vstep = static_cast<uint32_t>(step) * V;
            int pf = p0;
#pragma unroll
            for (int st = 0; st < GNF_STAGES; ++st) {
                if (pf < hw) {
                    cp_async16(ring + (st * 3 + 0) * blockDim.x + threadIdx.x, xpf);
                    cp_async16(ring + (st * 3 + 1) * blockDim.x + threadIdx.x, gpf);
                    if (addb != nullptr) cp_async16(ring + (st * 3 + 2) * blockDim.x + threadIdx.x, apf);
                }
                cp_async_commit();
                pf += step;
                xpf += xstride;
                gpf += gstride;
                apf += astride;
            }
            int st = 0;
            for (int p = p0; p < hw; p += step) {
                cp_async_wait<GNF_STAGES - 1>();
                uint4* sx_ = ring + (st * 3 + 0) * blockDim.x + threadIdx.x;
                uint4* sd_ = ring + (st * 3 + 1) * blockDim.x + threadIdx.x;
                uint4* sa_ = ring + (st * 3 + 2) * blockDim.x + threadIdx.x;
                const uint4 xr = *sx_, gr = *sd_;
                uint4 ar = make_uint4(0u, 0u, 0u, 0u);
                if (addb != nullptr) ar = *sa_;
                if (pf < hw) {
                    cp_async16(sx_, xpf);
                    cp_async16(sd_, gpf);
                    if (addb != nullptr) cp_async16(sa_, apf);
                }
                cp_async_commit();
                pf += step;
                xpf += xstride;
                gpf += gstride;
                apf += astride;
                if (++st == GNF_STAGES) st = 0;
                const uint32_t xw[4] = {xr.x, xr.y, xr.z, xr.w}, gw[4] = {gr.x, gr.y, gr.z, gr.w};
                const uint32_t aw[4] = {ar.x, ar.y, ar.z, ar.w};
                f32x2 x2[4], g2[4], dv[4], o[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) { x2[j] = bf2_to_f2(xw[j]); g2[j] = bf2_to_f2(gw[j]); }
                if (reuse_dv) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) dv[j] = g2[j];  // pass 1 left dv in dy's place
                } else {
                    dv_from2(g2, x2, ah2, bh2, act, drop_p, dc, vec, dv);
                }
                vec += vstep;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    o[j] = ffma2(dv[j], k1p[j], ffma2(x2[j], k2p[j], k3p[j]));
                    if (addb != nullptr) o[j] = fadd2(o[j], bf2_to_f2(aw[j]));
                    if (want_bs) bsp[j] = fadd2(bsp[j], o[j]);
                }
                *reinterpret_cast<uint4*>(op) = make_uint4(f2_to_bf2(o[0]), f2_to_bf2(o[1]), f2_to_bf2(o[2]), f2_to_bf2(o[3]));
                op += ostride;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) unpack2(bsp[j], bs[2 * j], bs[2 * j + 1]);
        } else {
            for (int p = p0; p < hw; p += step) {
                const Vec8 xv = load8(base + p * ld);
                Vec8 addv;
                if (addb != nullptr) {
                    if (add_mode == 0) {
                        addv = load8(addb + p * ldadd);
                    } else {
                        const int h = p / W, w = p - h * W;
                        if (add_mode == 1) {
                            addv = load8(addb + ((h >> 1) * (W >> 1) + (w >> 1)) * ldadd);
#pragma unroll
                            for (int j = 0; j < 8; ++j) addv.v[j] *= 0.25f;
                        } else {
                            Vec8 t[4];
#pragma unroll
                            for (int d = 0; d < 4; ++d)
                                t[d] = load8(addb + (1LL * (2 * h + (d >> 1)) * (2 * W) + 2 * w + (d & 1)) * ldadd);
#pragma unroll
                            for (int j = 0; j < 8; ++j) addv.v[j] = (t[0].v[j] + t[1].v[j]) + (t[2].v[j] + t[3].v[j]);
                        }
                    }
                }
                float dv[8];
                grad_preact(dyb, ldy, H, W, p, resample, act, drop_p, dc, vec0 + 1ULL * p * V, xv, a, b, dv);
                Vec8 o;
#pragma unroll
                for (int j = 0; j < 8; ++j) o.v[j] = dv[j] * k1[j] + xv.v[j] * k2[j] + k3[j];
                if (addb != nullptr) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) o.v[j] += addv.v[j];
                }
                if (want_bs) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) bs[j] += o.v[j];
                }
                store8(ob + p * ldo, o);
            }
        }
    }
    if (dbias1 != nullptr) {  // column sums of dx1 -> bias gradient of the conv that produced x1
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; ++j) red[threadIdx.x * 8 + j] = bs[j];
        __syncthreads();
        for (int c = threadIdx.x; c < c1; c += blockDim.x) {
            float s = 0.f;
            for (int l = 0; l < tpv; ++l) s += red[(l * V + (c >> 3)) * 8 + (c & 7)];
            atomicAdd(dbias1 + c, s);
            if (dbias1b != nullptr) atomicAdd(dbias1b + c, s);
        }
    }
}

static int grid_for(long long work, int threads, int n_batch) {
    long long blocks = (work + threads - 1) / threads;
    long long cap = (8LL * num_sms() + n_batch - 1) / n_batch;
    if (cap < 1) cap = 1;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return static_cast<int>(blocks);
}


// Cluster size for the one-cluster-per-sample kernels: the smallest K in {1,2,4,8} with n*K CTAs covering >= 60 % of
// the SMs; 0 when even K = 8 cannot (small batches use the multi-block kernels).
static int gn_cluster_size(int n) {
    const int want = (num_sms() * 6 + 9) / 10;
    int k = 1;
    while (k < 8 && n * k < want) k *= 2;
    return n * k >= want ? k : 0;
}

static int gn_fused_threads(int V, int hw, int k) {
    int tpv = 512 / V;
    const int per_cta = (hw + k - 1) / k;
    if (tpv > per_cta) tpv = per_cta;
    if (tpv < 1) tpv = 1;
    return tpv * V;
}

// Dynamic shared-memory limit of the two cluster kernels: covers their largest launch (gn_bwd_fused_kernel at C = 2048
// with 512 threads, 184 KB).
constexpr int GNF_SMEM_LIMIT = 200 * 1024;

}  // namespace adm

using namespace adm;
typedef __nv_bfloat16 bf16;

#define ADM_REQUIRE(cond, msg)        \
    do {                              \
        if (!(cond)) {                \
            set_error(msg);           \
            return ADM_ERR_SHAPE;     \
        }                             \
    } while (0)

extern "C" {

int adm_gn_stats(const void* x1, int c1, long long ld1, const void* x2, int c2, long long ld2, int n, int hw,
                 int groups, float eps, const float* gamma, const float* beta, const float* params,
                 long long ld_params, float* work, float* coef, void* stream) {
    const int C = c1 + c2;
    ADM_REQUIRE(c1 > 0 && c1 % 8 == 0 && c2 % 8 == 0 && (x2 != nullptr || c2 == 0) && C % groups == 0,
                "gn_stats: channels must be multiples of 8 and divisible by groups");
    ADM_REQUIRE(C <= 2048, "gn_stats: C too large");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cudaMemsetAsync(work, 0, sizeof(float) * (2LL * n * C + n), s);
    const int V = C / 8;
    const int threads = threads_for(V);
    const int tpv = threads / V;
    dim3 grid(grid_for(hw, tpv, n), n);
    gn_stats_kernel<<<grid, threads, threads * 16 * sizeof(float), s>>>(
        static_cast<const bf16*>(x1), c1, ld1, static_cast<const bf16*>(x2), c2, ld2, hw, work,
        reinterpret_cast<unsigned int*>(work + 2LL * n * C), gamma, beta, params, ld_params, groups, eps,
        reinterpret_cast<float4*>(coef));
    ADM_CHECK_LAUNCH("gn_stats");
    return 0;
}

int adm_gn_apply(const void* x1, int c1, long long ld1, const void* x2, int c2, long long ld2, int n, int h, int w,
                 const float* coef, int act, float drop_p, unsigned long long seed,
                 const unsigned long long* seed_counter, int resample, void* out, long long ldo, void* stream) {
    const unsigned long long* g_seed_dev = drop_p > 0.f ? seed_counter : nullptr;
    const int C = c1 + c2;
    ADM_REQUIRE(c1 > 0 && c1 % 8 == 0 && c2 % 8 == 0, "gn_apply: channels must be multiples of 8");
    ADM_REQUIRE(resample == 0 || (resample == 1 && h % 2 == 0 && w % 2 == 0) || resample == 2, "gn_apply: bad resample");
    ADM_REQUIRE(C <= 2048, "gn_apply: C too large");
    const int threads = threads_for(C / 8);
    const int tpv = threads / (C / 8);
    // ~3 CTAs per SM in total, each thread streaming >= 8 pixels of its channel vector when the image has that many
    const int pixels = resample == 1 ? (h / 2) * (w / 2) : h * w;
    int bps = (3 * num_sms() + n - 1) / n;
    const int maxb = (pixels + tpv * 8 - 1) / (tpv * 8);
    if (bps > maxb) bps = maxb;
    if (bps < 1) bps = 1;
    dim3 grid(bps, n);
    gn_apply_kernel<<<grid, threads, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const bf16*>(x1), c1, ld1, static_cast<const bf16*>(x2), c2, ld2, h, w,
        reinterpret_cast<const float4*>(coef), act, drop_p, seed, resample, static_cast<bf16*>(out), ldo, g_seed_dev);
    ADM_CHECK_LAUNCH("gn_apply");
    return 0;
}

int adm_gn_forward(const void* x1, int c1, long long ld1, const void* x2, int c2, long long ld2, int n, int h, int w,
                   int groups, float eps, const float* gamma, const float* beta, const float* params,
                   long long ld_params, float* work, float* coef, int act, float drop_p, unsigned long long seed,
                   const unsigned long long* seed_counter, int resample, void* out, long long ldo, void* stream) {
    const unsigned long long* g_seed_dev = drop_p > 0.f ? seed_counter : nullptr;
    const int C = c1 + c2;
    ADM_REQUIRE(c1 > 0 && c1 % 8 == 0 && c2 % 8 == 0 && (x2 != nullptr || c2 == 0) && C % groups == 0,
                "gn_forward: channels must be multiples of 8 and divisible by groups");
    ADM_REQUIRE(C <= 2048, "gn_forward: C too large");
    ADM_REQUIRE(resample == 0 || (resample == 1 && h % 2 == 0 && w % 2 == 0) || resample == 2, "gn_forward: bad resample");
    ADM_REQUIRE(out != nullptr, "gn_forward: out is required");
    const int k = gn_cluster_size(n);
    if (k == 0) {
        int rc = adm_gn_stats(x1, c1, ld1, x2, c2, ld2, n, h * w, groups, eps, gamma, beta, params, ld_params, work, coef,
                              stream);
        if (rc != 0) return rc;
        return adm_gn_apply(x1, c1, ld1, x2, c2, ld2, n, h, w, coef, act, drop_p, seed, seed_counter, resample, out, ldo,
                            stream);
    }
    const int V = C / 8;
    const int threads = gn_fused_threads(V, h * w, k);
    const size_t smem = sizeof(float) * (6 * C + 16 * threads);  // ring (4 x 16 B per thread) aliases the scratch
    cudaError_t e = set_smem_limit_once<gn_fwd_fused_kernel>(GNF_SMEM_LIMIT);
    if (e == cudaSuccess)
        e = launch_k(gn_fwd_fused_kernel, dim3(n * k), dim3(threads), smem, static_cast<cudaStream_t>(stream), k,
                     static_cast<const bf16*>(x1), c1, ld1, static_cast<const bf16*>(x2), c2, ld2, h, w, groups, eps, gamma,
                     beta, params, ld_params, reinterpret_cast<float4*>(coef), act, drop_p, seed, resample,
                     static_cast<bf16*>(out), ldo, g_seed_dev);
    if (e != cudaSuccess) {
        set_error("gn_forward launch: %s", cudaGetErrorString(e));
        return ADM_ERR_CUDA;
    }
    ADM_CHECK_LAUNCH("gn_forward");
    return 0;
}

int adm_gn_bwd(const void* dy, long long ldy, const void* x1, int c1, long long ld1, const void* x2, int c2,
               long long ld2, int n, int h, int w, int groups, const float* coef, const float* gamma,
               const float* beta, const float* params, long long ld_params, int act, float drop_p,
               unsigned long long seed, const unsigned long long* seed_counter, int resample, float* work,
               float* bcoef, float* dgamma, float* dbeta, float* dparams, long long ld_dparams, const void* add,
               long long ldadd, int add_mode, void* dx1, long long ldx1, void* dx2, long long ldx2, float* dbias1,
               float* dbias1b, int dy_scratch, void* stream) {
    const unsigned long long* g_seed_dev = drop_p > 0.f ? seed_counter : nullptr;
    const int C = c1 + c2;
    ADM_REQUIRE(c1 > 0 && c1 % 8 == 0 && c2 % 8 == 0 && C % groups == 0, "gn_bwd: bad channels / groups");
    ADM_REQUIRE(C <= 2048, "gn_bwd: C too large");
    // a half-resolution dy (or add) covers an H x W input only when both are even: pixel (H - 1, .) of an odd H would
    // read row H / 2 of dy, which belongs to the next sample (past the tensor for the last one)
    ADM_REQUIRE((resample == 0 || (resample == 1 && h % 2 == 0 && w % 2 == 0) || resample == 2) &&
                    (add == nullptr || add_mode == 0 || (add_mode == 1 && h % 2 == 0 && w % 2 == 0) || add_mode == 2),
                "gn_bwd: bad resample / add_mode");
    ADM_REQUIRE((dbias1 == nullptr || dx1 != nullptr) && (dbias1b == nullptr || dbias1 != nullptr),
                "gn_bwd: dbias1 needs dx1 (and dbias1b needs dbias1)");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bf16* dyp = static_cast<const bf16*>(dy);
    const bf16* x1p = static_cast<const bf16*>(x1);
    const bf16* x2p = static_cast<const bf16*>(x2);
    const int kc = gn_cluster_size(n);
    if (kc > 0) {
        const int threads = gn_fused_threads(C / 8, h * w, kc);
        const size_t smem = sizeof(float) * (7 * C + 16 * threads) + 16 * GNF_STAGES * 3 * threads;
        cudaError_t e = set_smem_limit_once<gn_bwd_fused_kernel>(GNF_SMEM_LIMIT);
        if (e == cudaSuccess)
            e = launch_k(gn_bwd_fused_kernel, dim3(n * kc), dim3(threads), smem, s, kc, dyp, ldy, x1p, c1, ld1, x2p, c2, ld2,
                         h, w, groups, reinterpret_cast<const float4*>(coef), gamma, beta, params, ld_params, act, drop_p,
                         seed, resample, dgamma, dbeta, dparams, ld_dparams, static_cast<const bf16*>(add), ldadd, add_mode,
                         static_cast<bf16*>(dx1), ldx1, static_cast<bf16*>(dx2), ldx2, dbias1, dbias1b, g_seed_dev,
                         dy_scratch);
        if (e != cudaSuccess) {
            set_error("gn_bwd (fused) launch: %s", cudaGetErrorString(e));
            return ADM_ERR_CUDA;
        }
        ADM_CHECK_LAUNCH("gn_bwd_fused");
        return 0;
    }
    cudaMemsetAsync(work, 0, sizeof(float) * (2LL * n * C + n), s);
    const int V = C / 8;
    const int threads = threads_for(V);
    const int tpv = threads / V;
    {
        dim3 grid(grid_for(h * w, tpv * 2, n), n);
        size_t smem = threads * 16 * sizeof(float);
        if (smem < 2 * C * sizeof(float)) smem = 2 * C * sizeof(float);
        gn_bwd_reduce_kernel<<<grid, threads, smem, s>>>(
            dyp, ldy, x1p, c1, ld1, x2p, c2, ld2, h, w, groups, reinterpret_cast<const float4*>(coef), gamma, beta,
            params, ld_params, act, drop_p, seed, resample, work, reinterpret_cast<unsigned int*>(work + 2LL * n * C),
            reinterpret_cast<float4*>(bcoef), dgamma, dbeta, dparams, ld_dparams, g_seed_dev);
        ADM_CHECK_LAUNCH("gn_bwd_reduce");
    }
    if (dx1 != nullptr) {
        dim3 grid(grid_for(h * w, tpv * 2, n), n);
        gn_bwd_apply_kernel<<<grid, threads, 0, s>>>(
            dyp, ldy, x1p, c1, ld1, x2p, c2, ld2, h, w, reinterpret_cast<const float4*>(coef),
            reinterpret_cast<const float4*>(bcoef), act, drop_p, seed, resample, static_cast<const bf16*>(add), ldadd,
            add_mode, static_cast<bf16*>(dx1), ldx1, static_cast<bf16*>(dx2), ldx2, g_seed_dev);
        ADM_CHECK_LAUNCH("gn_bwd_apply");
        if (dbias1 != nullptr) {
            int rc = adm_col_sums(dx1, ldx1, 1LL * n * h * w, c1, dbias1, stream);
            if (rc != 0 || dbias1b == nullptr) return rc;
            return adm_col_sums(dx1, ldx1, 1LL * n * h * w, c1, dbias1b, stream);
        }
    }
    return 0;
}

int adm_col_sums(const void* x, long long ld, long long rows, int c, float* out, void* stream) {
    return adm_col_sums_mapped(x, ld, rows, c, out, nullptr, stream);
}

int adm_col_sums_mapped(const void* x, long long ld, long long rows, int c, float* out, const int* out_map,
                        void* stream) {
    ADM_REQUIRE(c > 0 && c % 8 == 0, "col_sums: C must be a multiple of 8");
    const int chunks = (c + 2047) / 2048;
    // all chunks but the last are 2048 wide (V = 256 -> 256 threads); size the block for the narrowest chunk
    const int last = c - (chunks - 1) * 2048;
    const int threads = chunks > 1 ? 256 : threads_for(last / 8);
    ADM_REQUIRE(chunks == 1 || last % 8 == 0, "col_sums: bad width");
    const int tpv = threads / ((chunks > 1 ? 2048 : last) / 8);
    dim3 grid(grid_for(rows, tpv > 0 ? tpv : 1, chunks), chunks);
    launch_k(col_sums_kernel, grid, dim3(threads), threads * 8 * sizeof(float), static_cast<cudaStream_t>(stream), 0,
             static_cast<const bf16*>(x), ld, rows, c, out, out_map);
    ADM_CHECK_LAUNCH("col_sums");
    return 0;
}

int adm_add_bf16(const void* a, long long lda, const void* b, long long ldb, const void* c, long long ldc, void* out,
                 long long ldo, long long rows, int ch, void* stream) {
    ADM_REQUIRE(ch > 0 && ch % 8 == 0, "add_bf16: channels must be a multiple of 8");
    ADM_REQUIRE(rows * (ch / 8) < (1LL << 31), "add_bf16: tensor too large (32-bit vector index)");
    launch_k(add_bf16_kernel, dim3(grid_for(rows * (ch / 8), 256, 1)), dim3(256), 0, static_cast<cudaStream_t>(stream), 0,
             static_cast<const bf16*>(a), lda, static_cast<const bf16*>(b), ldb, static_cast<const bf16*>(c), ldc,
             static_cast<bf16*>(out), ldo, rows, ch);
    ADM_CHECK_LAUNCH("add_bf16");
    return 0;
}

int adm_resample(const void* x, long long ldx, int n, int h, int w, int c, int mode, void* out, long long ldo,
                 void* stream) {
    ADM_REQUIRE(c % 8 == 0 && (mode == 1 || mode == 2), "resample: bad arguments");
    ADM_REQUIRE(mode == 2 || (h % 2 == 0 && w % 2 == 0), "resample: odd size");
    const long long total = 1LL * n * (mode == 1 ? (h / 2) * (w / 2) : 4 * h * w) * (c / 8);
    ADM_REQUIRE(total < (1LL << 31), "resample: tensor too large (32-bit vector index)");
    resample_kernel<<<grid_for(total, 256, 1), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const bf16*>(x), ldx, n, h, w, c, mode, static_cast<bf16*>(out), ldo);
    ADM_CHECK_LAUNCH("resample");
    return 0;
}

int adm_silu(const float* x, float* y, void* y_bf16, long long numel, void* stream) {
    silu_kernel<<<grid_for(numel, 256, 1), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, y, static_cast<bf16*>(y_bf16),
                                                                                       numel);
    ADM_CHECK_LAUNCH("silu");
    return 0;
}

int adm_silu_bwd(const float* x, const float* dy, float* dx, void* dx_bf16, long long numel, void* stream) {
    silu_bwd_kernel<<<grid_for(numel, 256, 1), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        x, dy, dx, static_cast<bf16*>(dx_bf16), numel);
    ADM_CHECK_LAUNCH("silu_bwd");
    return 0;
}

}  // extern "C"
