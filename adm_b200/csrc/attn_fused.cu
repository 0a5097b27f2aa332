// K9: fused softmax attention over pixels for the low-resolution UNet levels (reference unet/uncond_unet.py:204-208:
// w = softmax_k(q^T k / sqrt(d)); a = v w^T), forward AND backward, with the N x N probability matrix living only in
// TENSOR MEMORY — it is never written to shared memory or HBM, in inference or in training:
//
//   forward   S = Q K^T (tcgen05, fp32 in TMEM) -> per-row softmax by 128 threads (lane = query row) -> P written back
//             IN PLACE as bf16 pairs (tcgen05.st) -> O = P V with the A operand read from TMEM (tcgen05.mma [d], [a], b)
//             -> O / rowsum -> bf16 [B, N, C]; the per-row log-sum-exp goes to HBM (4 B per row) for the backward.
//   backward  recomputes the probabilities instead of re-reading them (P-free), in the TRANSPOSED orientation so that
//             every product that consumes P or dS has it as a TMEM A operand:
//               S^T = K Q^T, dP^T = V dO^T            (lanes = key rows, columns = queries)
//               P^T = exp2(c1 S^T - L_q), dS^T = scale P^T (dP^T - D_q),  D_q = sum_d dO_qd O_qd
//               dV += P^T dO, dK += dS^T Q            (A from TMEM, B = dO / Q consumed MN-major from shared memory)
//               dQ += dS K                            (dS^T also goes to shared memory: the same tile read MN-major is dS)
//             dK, dV, dQ accumulate in TMEM across the whole (sample, head) and are stored once.
//
// Persistent, warp-specialised CTAs (320 threads, 1 per SM): warp 0 = TMA producer, warp 1 = tcgen05 issuer, warps 2-5 and
// 6-9 = two softmax groups that ping-pong over tiles (forward) / 64-query sub-blocks (backward), so the tensor core works
// on one group's tile while the other group is in its exponentials.  Operand stages are multi-buffered in shared memory,
// i.e. the TMA loads of the next (sample, head) fly under the current one.
// Small images are PACKED: 128 tile rows hold 2 samples of 64 pixels or 8 samples of 16 pixels (one TMA box over
// (channel, pixel, sample)); the off-diagonal blocks of S are masked to zero probability.
// Shapes: pixels N in {16, 64, 256}, head dim 64 (32 / 72 run zero-padded by the caller).
// Longer sequences (N = nblk * 256, e.g. the 32 x 32 level of the CelebAHQ-latent UNet, configs/celebahq/...ldm.yaml:55) run
// BLOCKED on the same kernels: a work unit is (sample, head, query block, key block) of 256 x 256.  Forward units emit a
// block-normalised partial O and a partial log-sum-exp per key block, merged by attn_combine_kernel; backward units use
// the merged log-sum-exp (so P is already the global probability) and emit partial dQ (per key block) and dK / dV (per
// query block) into nblk dqkv-shaped buffers that attn_reduce_kernel sums.  No N x N tensor exists in either direction.
#include <algorithm>
#include <climits>

#include "adm_internal.h"
#include "ptx.cuh"

namespace adm {

constexpr int AT_THREADS = 320;
constexpr int AT_RING = 192 * 1024;          // forward: operand stages; backward: operand stages + the dS tile
constexpr int AT_SMEM_TOTAL = AT_RING + 8192 + 1024;  // ring + (barriers 1 KB, backward's L / D tables 4 KB) + alignment slack
constexpr int AT_MAX_STAGES = 4;

__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    const __nv_bfloat162 b2 = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&b2);
}
__device__ __forceinline__ void st_row16(__nv_bfloat16* dst, const uint32_t (&w)[8]) {  // 16 bf16 = 32 B
    if ((reinterpret_cast<uintptr_t>(dst) & 31) == 0) {
        asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(w[0]), "r"(w[1]),
                     "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
                     : "memory");
    } else {
        *reinterpret_cast<uint4*>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<uint4*>(dst + 8) = make_uint4(w[4], w[5], w[6], w[7]);
    }
}

struct AttnParams {
    int n_pix;    // N: 16, 64 or 256 (queries = keys per sample)
    int pack;     // samples per 128-row tile: 8, 2 or 1
    int heads, batch, c;  // C = heads * 64
    int units;    // work units: (sample group, head)
    int tiles;    // 128-query tiles per unit: 2 when N = 256, else 1
    int ncols;    // key columns per unit: 256 or 128
    int stages;   // operand stages in shared memory
    float scale, c1;  // softmax(scale * q.k);  c1 = scale * log2(e)
    __nv_bfloat16* out;        // fwd: O [B, N, C];  bwd: dqkv [B, N, 3C]
    float* lse;                // [B, heads, N]  (log2 domain: c1 * max + log2(sum))
    const __nv_bfloat16* o_in; // bwd: the forward output O
    int nblk;                  // 1, or the number of 256-pixel blocks of a long sequence (blocked units, see above)
    long long out_stride;      // blocked: elements between consecutive partial buffers of `out`
    long long lse_stride;      // blocked forward: elements between consecutive partial log-sum-exp buffers
};

// work unit -> (first sample, head, query block, key block)
__device__ __forceinline__ void attn_unit(const AttnParams& p, int u, int& b0, int& h, int& qb, int& kb) {
    if (p.nblk == 1) {
        b0 = (u / p.heads) * p.pack;
        h = u % p.heads;
        qb = kb = 0;
    } else {
        kb = u % p.nblk;
        u /= p.nblk;
        qb = u % p.nblk;
        u /= p.nblk;
        h = u % p.heads;
        b0 = u / p.heads;
    }
}

// ------------------------------------------------------------------------------------------------ forward
__global__ void __launch_bounds__(AT_THREADS, 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ AttnParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + AT_RING);
    uint64_t* empty = full + AT_MAX_STAGES;
    uint64_t* s_full = empty + AT_MAX_STAGES;  // [2] S of slot g is in TMEM
    uint64_t* p_full = s_full + 2;             // [2] P of slot g is in TMEM (softmax done)
    uint64_t* o_full = p_full + 2;             // [2] O of slot g is in TMEM
    uint64_t* o_done = o_full + 2;             // [2] slot g has been drained
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(o_done + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q_bytes = p.tiles * 16384, kv_bytes = p.ncols * 128;
    const int stage_bytes = q_bytes + 2 * kv_bytes;
    const int n_local = static_cast<int>(blockIdx.x) < p.units
                            ? (p.units - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x)
                            : 0;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmQKV);
        for (int i = 0; i < p.stages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], p.tiles); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&s_full[i], 1); mbar_init(&p_full[i], 4); mbar_init(&o_full[i], 1); mbar_init(&o_done[i], 4);
        }
        fence_barrier_init();
        fence_proxy_async_smem();
    }
    if (warp == 1) tmem_alloc(tmem_ptr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // =========================================================== TMA producer
        if (lane == 0) {
            for (int ul = 0; ul < n_local; ++ul) {
                int b0, h, qb, kb;
                attn_unit(p, blockIdx.x + ul * gridDim.x, b0, h, qb, kb);
                const int st = ul % p.stages;
                mbar_wait(&empty[st], ((ul / p.stages) & 1) ^ 1, 21);
                mbar_expect_tx(&full[st], stage_bytes);
                uint8_t* sq = smem + st * stage_bytes;
                tma_load_3d(sq, &tmQKV, &full[st], h * 64, qb * 256, b0);
                tma_load_3d(sq + q_bytes, &tmQKV, &full[st], p.c + h * 64, kb * 256, b0);
                tma_load_3d(sq + q_bytes + kv_bytes, &tmQKV, &full[st], 2 * p.c + h * 64, kb * 256, b0);
            }
        }
    } else if (warp == 1) {
        // =========================================================== tcgen05 issuer
        if (lane == 0) {
            const uint32_t idesc_s = make_idesc_bf16(128, p.ncols, 0, 0);
            const uint32_t idesc_o = make_idesc_bf16(128, 64, 0, 1);
            const int total = n_local * p.tiles;
            const int ksteps = p.ncols >> 4;
            auto issue_pv = [&](int k) {
                const int ul = k / p.tiles, tl = k % p.tiles;
                const int g = p.tiles == 2 ? tl : (ul & 1), it = p.tiles == 2 ? ul : (ul >> 1);
                const int st = ul % p.stages;
                mbar_wait(&p_full[g], it & 1, 22);
                tc_fence_after();
                const uint32_t sv = smem_u32(smem + st * stage_bytes + q_bytes + kv_bytes);
                const uint32_t slot = tmem_base + g * 256;
                for (int kk = 0; kk < ksteps; ++kk)  // O = P V: A = P from TMEM (8 columns per 16 keys), B = V MN-major
                    umma_bf16_ts(slot + (p.ncols >> 1), slot + kk * 8, make_smem_desc(sv + kk * 2048u, 8192u, 1024), idesc_o,
                                 kk > 0 ? 1u : 0u);
                umma_commit(&o_full[g]);
                umma_commit(&empty[st]);
            };
            for (int k = 0; k < total; ++k) {
                const int ul = k / p.tiles, tl = k % p.tiles;
                const int g = p.tiles == 2 ? tl : (ul & 1), it = p.tiles == 2 ? ul : (ul >> 1);
                const int st = ul % p.stages;
                mbar_wait(&full[st], (ul / p.stages) & 1, 23);
                mbar_wait(&o_done[g], (it & 1) ^ 1, 24);
                tc_fence_after();
                const uint32_t sq = smem_u32(smem + st * stage_bytes + tl * 16384);
                const uint32_t sk = smem_u32(smem + st * stage_bytes + q_bytes);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)  // S = Q K^T, K-major x K-major
                    umma_bf16(tmem_base + g * 256, make_smem_desc(sq + kk * 32u, 16u, 1024),
                              make_smem_desc(sk + kk * 32u, 16u, 1024), idesc_s, kk > 0 ? 1u : 0u);
                umma_commit(&s_full[g]);
                if (k >= 1) issue_pv(k - 1);
            }
            if (total > 0) issue_pv(total - 1);
        }
    } else {
        // =========================================================== softmax groups (128 threads each, lane = query row)
        const int g = (warp - 2) >> 2;
        const int quad = warp & 3;             // TMEM lane quadrant this warp may access
        const int row = quad * 32 + lane;      // row inside the 128-row tile
        const uint32_t taddr = tmem_base + g * 256 + (static_cast<uint32_t>(quad * 32) << 16);
        const int N = p.n_pix;
        const int wn = N < 32 ? 32 : (N > 256 ? 256 : N);  // key window this warp reads (warp-uniform), a multiple of 32
        const int wbeg = p.ncols == 256 ? 0 : (row / wn) * wn;
        const int my_blk = row / N;            // packed: the sample (inside the tile) this row belongs to
        int it = 0;
        for (int ul = (p.tiles == 2 ? 0 : g); ul < n_local; ul += (p.tiles == 2 ? 1 : 2), ++it) {
            const int tl = p.tiles == 2 ? g : 0;
            int b0, h, qb, kb;
            attn_unit(p, blockIdx.x + ul * gridDim.x, b0, h, qb, kb);
            mbar_wait(&s_full[g], it & 1, 25);
            tc_fence_after();
            // ---- pass 1: row maximum over this row's own keys
            float mx = -INFINITY;
            for (int c0 = 0; c0 < wn; c0 += 32) {
                uint32_t v[32];
                __syncwarp();
                tmem_ld_x32(taddr + wbeg + c0, v);
                tmem_ld_wait();
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    const bool valid = p.ncols == 256 || ((wbeg + c0 + 16 * hf) / N) == my_blk;
                    if (valid) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) mx = fmaxf(mx, __uint_as_float(v[16 * hf + j]));
                    }
                }
            }
            const float mc = mx * p.c1;
            // ---- pass 2: P = exp2(c1 s - c1 max) (unnormalised), row sum, P back to TMEM in place as bf16 pairs
            float sum = 0.f;
            for (int c0 = 0; c0 < wn; c0 += 32) {
                uint32_t v[32];
                __syncwarp();
                tmem_ld_x32(taddr + wbeg + c0, v);
                tmem_ld_wait();
                uint32_t w[16];
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    const bool valid = p.ncols == 256 || ((wbeg + c0 + 16 * hf) / N) == my_blk;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        float p0 = 0.f, p1 = 0.f;
                        if (valid) {
                            p0 = ex2(fmaf(__uint_as_float(v[16 * hf + 2 * j]), p.c1, -mc));
                            p1 = ex2(fmaf(__uint_as_float(v[16 * hf + 2 * j + 1]), p.c1, -mc));
                        }
                        sum += p0 + p1;
                        w[8 * hf + j] = pack_bf16(p0, p1);
                    }
                }
                __syncwarp();
                tmem_st_x16(taddr + ((wbeg + c0) >> 1), w);
            }
            if (p.ncols != 256) {  // packed tiles: zero probability for the other samples' keys (outside the window)
                uint32_t z[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) z[j] = 0u;
                for (int pc = 0; pc < 64; pc += 16)
                    if (pc < (wbeg >> 1) || pc >= ((wbeg + wn) >> 1)) {
                        __syncwarp();
                        tmem_st_x16(taddr + pc, z);
                    }
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&p_full[g]);
            // ---- epilogue: O / sum -> bf16, log-sum-exp
            const int smp = b0 + (p.ncols == 256 ? 0 : my_blk);
            const int pix = p.ncols == 256 ? qb * 256 + tl * 128 + row : row - my_blk * N;
            const bool row_ok = smp < p.batch;
            const float inv = 1.f / sum;
            mbar_wait(&o_full[g], it & 1, 26);
            tc_fence_after();
            __nv_bfloat16* op = p.out + kb * p.out_stride + (1LL * smp * N + pix) * p.c + h * 64;
#pragma unroll
            for (int c0 = 0; c0 < 64; c0 += 32) {
                uint32_t v[32];
                __syncwarp();
                tmem_ld_x32(taddr + (p.ncols >> 1) + c0, v);
                tmem_ld_wait();
                if (row_ok) {
#pragma unroll
                    for (int s = 0; s < 2; ++s) {
                        uint32_t w[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            w[j] = pack_bf16(__uint_as_float(v[16 * s + 2 * j]) * inv, __uint_as_float(v[16 * s + 2 * j + 1]) * inv);
                        st_row16(op + c0 + 16 * s, w);
                    }
                }
            }
            if (row_ok && p.lse != nullptr) p.lse[kb * p.lse_stride + (1LL * smp * p.heads + h) * N + pix] = mc + log2f(sum);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&o_done[g]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------------------------------ backward
// TMEM columns: [g*128, +64) S^T of group g's sub-block (P^T in place, 32 columns), [g*128+64, +64) dP^T (dS^T in place),
// [256, 320) dK_j, [320, 384) dV_j, [384, 448) dQ tile 0, [448, 512) dQ tile 1.
constexpr int BW_DK = 256, BW_DV = 320, BW_DQ = 384;

__global__ void __launch_bounds__(AT_THREADS, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO,
                const __grid_constant__ AttnParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + AT_RING);
    uint64_t* empty = full + AT_MAX_STAGES;
    uint64_t* sdp_full = empty + AT_MAX_STAGES;  // [2] S^T / dP^T of group g's sub-block are in TMEM
    uint64_t* p_full = sdp_full + 2;             // [2] P^T / dS^T (TMEM) and the dS chunk (smem) of group g are written
    uint64_t* ds_empty = p_full + 2;             // the dS tile in shared memory has been consumed by its dQ product
    uint64_t* acc_full = ds_empty + 1;           // dK_j / dV_j (and, on the last j, dQ) are complete in TMEM
    uint64_t* acc_done = acc_full + 1;           // ... and have been drained
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_done + 1);
    float* sLD = reinterpret_cast<float*>(smem + AT_RING + 1024);  // 2 x {L[256], D[256]}, double-buffered by unit parity

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nq = p.tiles * 128;                 // queries per unit (= keys per unit = ncols)
    const int t_bytes = nq * 128;                 // one operand (Q, K, V or dO) of a unit
    const int stage_bytes = 4 * t_bytes;
    uint8_t* sds = smem + p.stages * stage_bytes; // dS tile: [128 key rows] x 2 chunks of 64 queries (32 KB)
    const int nkt = p.ncols >> 7, nq4 = nq >> 6, nsb = nkt * nq4;
    const int n_local = static_cast<int>(blockIdx.x) < p.units
                            ? (p.units - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x)
                            : 0;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmQKV);
        tma_prefetch_desc(&tmDO);
        for (int i = 0; i < p.stages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&sdp_full[i], 1); mbar_init(&p_full[i], 4); }
        mbar_init(ds_empty, 1);
        mbar_init(acc_full, 1);
        mbar_init(acc_done, 8);
        fence_barrier_init();
        fence_proxy_async_smem();
    }
    if (warp == 1) tmem_alloc(tmem_ptr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // =========================================================== TMA producer
        if (lane == 0) {
            for (int ul = 0; ul < n_local; ++ul) {
                int b0, h, qb, kb;
                attn_unit(p, blockIdx.x + ul * gridDim.x, b0, h, qb, kb);
                const int st = ul % p.stages;
                mbar_wait(&empty[st], ((ul / p.stages) & 1) ^ 1, 31);
                mbar_expect_tx(&full[st], stage_bytes);
                uint8_t* s0 = smem + st * stage_bytes;
                tma_load_3d(s0, &tmQKV, &full[st], h * 64, qb * 256, b0);                        // Q
                tma_load_3d(s0 + t_bytes, &tmQKV, &full[st], p.c + h * 64, kb * 256, b0);         // K
                tma_load_3d(s0 + 2 * t_bytes, &tmQKV, &full[st], 2 * p.c + h * 64, kb * 256, b0); // V
                tma_load_3d(s0 + 3 * t_bytes, &tmDO, &full[st], h * 64, qb * 256, b0);            // dO
            }
        }
    } else if (warp == 1) {
        // =========================================================== tcgen05 issuer
        if (lane == 0) {
            const uint32_t idesc_sdp = make_idesc_bf16(128, 64, 0, 0);   // S^T / dP^T : K-major x K-major
            const uint32_t idesc_kv = make_idesc_bf16(128, 64, 0, 1);    // dV / dK    : A TMEM, B MN-major
            const uint32_t idesc_dq = make_idesc_bf16(128, 64, 1, 1);    // dQ         : A (dS tile) and B (K) MN-major
            const uint32_t sds_a = smem_u32(sds);
            for (int ul = 0; ul < n_local; ++ul) {
                const int st = ul % p.stages;
                const uint32_t sq = smem_u32(smem + st * stage_bytes), sk = sq + t_bytes, sv = sq + 2 * t_bytes,
                               sdo = sq + 3 * t_bytes;
                mbar_wait(&full[st], (ul / p.stages) & 1, 32);
                tc_fence_after();
                auto issue_sdp = [&](int sb) {
                    const int j = sb / nq4, i4 = sb % nq4, g = sb & 1;
                    const uint32_t d = tmem_base + g * 128;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        umma_bf16(d, make_smem_desc(sk + j * 16384 + kk * 32u, 16u, 1024),
                                  make_smem_desc(sq + i4 * 8192 + kk * 32u, 16u, 1024), idesc_sdp, kk > 0 ? 1u : 0u);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        umma_bf16(d + 64, make_smem_desc(sv + j * 16384 + kk * 32u, 16u, 1024),
                                  make_smem_desc(sdo + i4 * 8192 + kk * 32u, 16u, 1024), idesc_sdp, kk > 0 ? 1u : 0u);
                    umma_commit(&sdp_full[g]);
                };
                issue_sdp(0);
                if (nsb > 1) issue_sdp(1);
                for (int sb = 0; sb < nsb; ++sb) {
                    const int j = sb / nq4, i4 = sb % nq4, g = sb & 1;
                    const int gsb = ul * nsb + sb;  // running sub-block count; group g's iteration = gsb / 2
                    mbar_wait(&p_full[g], (gsb >> 1) & 1, 33);
                    if (i4 == 0) mbar_wait(acc_done, ((ul * nkt + j) & 1) ^ 1, 34);  // dK / dV (/ dQ) columns are free
                    tc_fence_after();
                    const uint32_t a = tmem_base + g * 128;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {  // 64 queries = 4 k-steps; A advances 8 columns
                        const uint32_t acc = (i4 > 0 || kk > 0) ? 1u : 0u;
                        umma_bf16_ts(tmem_base + BW_DV, a + kk * 8, make_smem_desc(sdo + i4 * 8192 + kk * 2048u, 8192u, 1024),
                                     idesc_kv, acc);
                        umma_bf16_ts(tmem_base + BW_DK, a + 64 + kk * 8, make_smem_desc(sq + i4 * 8192 + kk * 2048u, 8192u, 1024),
                                     idesc_kv, acc);
                    }
                    if (i4 & 1) {  // both 64-query chunks of this 128-query tile are in shared memory: dQ_i += dS K_j
                        const int i = i4 >> 1;
#pragma unroll
                        for (int kk = 0; kk < 8; ++kk)
                            umma_bf16(tmem_base + BW_DQ + i * 64, make_smem_desc(sds_a + kk * 2048u, 16384u, 1024),
                                      make_smem_desc(sk + j * 16384 + kk * 2048u, 8192u, 1024), idesc_dq,
                                      (j > 0 || kk > 0) ? 1u : 0u);
                        umma_commit(ds_empty);
                    }
                    if (i4 == nq4 - 1) umma_commit(acc_full);
                    if (sb + 2 < nsb) issue_sdp(sb + 2);
                }
                umma_commit(&empty[st]);
            }
        }
    } else {
        // =========================================================== softmax groups (lane = key row)
        const int g = (warp - 2) >> 2;
        const int quad = warp & 3;
        const int row = quad * 32 + lane;       // key row inside the 128-key tile
        const int tq = g * 128 + ((warp - 2) & 3) * 32 + lane;  // this thread's query for the D / L prologue
        const uint32_t trow = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
        const int N = p.n_pix;
        const bool packed = p.ncols != 256;
        int itg = 0;   // sub-blocks this group has processed
        for (int ul = 0; ul < n_local; ++ul) {
            // L_q / D_q tables: a group may run ahead of the other by less than one unit (the barrier below), so two
            // copies selected by the unit's parity are enough
            float* sL = sLD + (ul & 1) * 512;
            float* sD = sL + 256;
            int b0, h, qb, kb;
            attn_unit(p, blockIdx.x + ul * gridDim.x, b0, h, qb, kb);
            const int st = ul % p.stages;
            const uint8_t* sdo = smem + st * stage_bytes + 3 * t_bytes;
            mbar_wait(&full[st], (ul / p.stages) & 1, 35);
            // ---- prologue: D_q = sum_d dO_qd O_qd and L_q for every query of the unit
            if (tq < nq) {
                const int smp = b0 + (packed ? tq / N : 0), pix = packed ? tq % N : qb * 256 + tq;
                float d = 0.f, l = 0.f;
                if (smp < p.batch) {
                    const uint4* orow = reinterpret_cast<const uint4*>(p.o_in + (1LL * smp * N + pix) * p.c + h * 64);
#pragma unroll
                    for (int un = 0; un < 8; ++un) {
                        const uint4 a = *reinterpret_cast<const uint4*>(sdo + tq * 128 + ((un ^ (tq & 7)) << 4));
                        const uint4 b = __ldg(orow + un);
                        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            d = fmaf(__uint_as_float(aw[e] << 16), __uint_as_float(bw[e] << 16), d);
                            d = fmaf(__uint_as_float(aw[e] & 0xFFFF0000u), __uint_as_float(bw[e] & 0xFFFF0000u), d);
                        }
                    }
                    l = p.lse[(1LL * smp * p.heads + h) * N + pix];
                }
                sD[tq] = d;
                sL[tq] = l;
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            for (int sb = g; sb < nsb; sb += 2, ++itg) {
                const int j = sb / nq4, i4 = sb % nq4;
                mbar_wait(&sdp_full[g], itg & 1, 36);
                tc_fence_after();
                const uint32_t ts = trow + g * 128;
                const int kblk = row / N;  // packed: sample (inside the tile) of this key row
                uint32_t dsw[32];          // this row's dS^T (64 queries) as bf16 pairs, for the shared-memory tile
#pragma unroll
                for (int c0 = 0; c0 < 64; c0 += 32) {
                    uint32_t s[32], dp[32];
                    __syncwarp();
                    tmem_ld_x32(ts + c0, s);
                    tmem_ld_x32(ts + 64 + c0, dp);
                    tmem_ld_wait();
                    uint32_t pw[16];
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf) {
                        const int qc = i4 * 64 + c0 + 16 * hf;  // first query column of this 16-chunk
                        const bool valid = !packed || (qc / N) == kblk;
#pragma unroll
                        for (int e = 0; e < 16; e += 4) {
                            const float4 l4 = *reinterpret_cast<const float4*>(sL + qc + e);
                            const float4 d4 = *reinterpret_cast<const float4*>(sD + qc + e);
                            const float lv[4] = {l4.x, l4.y, l4.z, l4.w}, dv[4] = {d4.x, d4.y, d4.z, d4.w};
                            float pv[4], ds[4];
#pragma unroll
                            for (int t = 0; t < 4; ++t) {
                                const int idx = 16 * hf + e + t;
                                pv[t] = valid ? ex2(fmaf(__uint_as_float(s[idx]), p.c1, -lv[t])) : 0.f;
                                ds[t] = p.scale * pv[t] * (__uint_as_float(dp[idx]) - dv[t]);
                            }
                            pw[8 * hf + (e >> 1)] = pack_bf16(pv[0], pv[1]);
                            pw[8 * hf + (e >> 1) + 1] = pack_bf16(pv[2], pv[3]);
                            dsw[(c0 >> 1) + 8 * hf + (e >> 1)] = pack_bf16(ds[0], ds[1]);
                            dsw[(c0 >> 1) + 8 * hf + (e >> 1) + 1] = pack_bf16(ds[2], ds[3]);
                        }
                    }
                    uint32_t dw[16];
#pragma unroll
                    for (int t = 0; t < 16; ++t) dw[t] = dsw[(c0 >> 1) + t];
                    __syncwarp();
                    tmem_st_x16(ts + (c0 >> 1), pw);        // P^T in place over S^T
                    tmem_st_x16(ts + 64 + (c0 >> 1), dw);   // dS^T in place over dP^T
                }
                // dS^T row -> shared-memory tile (chunk i4 & 1), 128B-swizzled rows; read MN-major by the dQ product
                // (tile t = (key tile j, query tile i4 / 2) may be overwritten once the dQ product of tile t - 1 completed)
                mbar_wait(ds_empty, ((ul * (nsb >> 1) + (sb >> 1)) & 1) ^ 1, 37);
                uint8_t* drow = sds + (i4 & 1) * 16384 + row * 128;
#pragma unroll
                for (int un = 0; un < 8; ++un)
                    *reinterpret_cast<uint4*>(drow + ((un ^ (row & 7)) << 4)) =
                        make_uint4(dsw[4 * un], dsw[4 * un + 1], dsw[4 * un + 2], dsw[4 * un + 3]);
                fence_proxy_async_smem();
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&p_full[g]);
                // ---- at the end of a key tile: drain dK_j (group 0) / dV_j (group 1); on the last one also dQ
                if (i4 >= nq4 - 2) {
                    const int jj = ul * nkt + j;
                    mbar_wait(acc_full, jj & 1, 38);
                    tc_fence_after();
                    const int krow = j * 128 + row;
                    const int smp = b0 + (packed ? krow / N : 0), pix = packed ? krow % N : kb * 256 + krow;
                    // blocked: partial dK / dV of this query block go to buffer qb, partial dQ of this key block to buffer kb
                    __nv_bfloat16* gp =
                        p.out + qb * p.out_stride + (1LL * smp * N + pix) * 3 * p.c + (g == 0 ? p.c : 2 * p.c) + h * 64;
                    const uint32_t src = trow + (g == 0 ? BW_DK : BW_DV);
#pragma unroll
                    for (int c0 = 0; c0 < 64; c0 += 32) {
                        uint32_t v[32];
                        __syncwarp();
                        tmem_ld_x32(src + c0, v);
                        tmem_ld_wait();
                        if (smp < p.batch) {
#pragma unroll
                            for (int s2 = 0; s2 < 2; ++s2) {
                                uint32_t w[8];
#pragma unroll
                                for (int t = 0; t < 8; ++t)
                                    w[t] = pack_bf16(__uint_as_float(v[16 * s2 + 2 * t]), __uint_as_float(v[16 * s2 + 2 * t + 1]));
                                st_row16(gp + c0 + 16 * s2, w);
                            }
                        }
                    }
                    if (j == nkt - 1 && g < p.tiles) {  // dQ tile g: rows = queries g*128 + row
                        const int qrow = g * 128 + row;
                        const int qs = b0 + (packed ? qrow / N : 0), qp = packed ? qrow % N : qb * 256 + qrow;
                        __nv_bfloat16* qg = p.out + kb * p.out_stride + (1LL * qs * N + qp) * 3 * p.c + h * 64;
#pragma unroll
                        for (int c0 = 0; c0 < 64; c0 += 32) {
                            uint32_t v[32];
                            __syncwarp();
                            tmem_ld_x32(trow + BW_DQ + g * 64 + c0, v);
                            tmem_ld_wait();
                            if (qs < p.batch) {
#pragma unroll
                                for (int s2 = 0; s2 < 2; ++s2) {
                                    uint32_t w[8];
#pragma unroll
                                    for (int t = 0; t < 8; ++t)
                                        w[t] = pack_bf16(__uint_as_float(v[16 * s2 + 2 * t]), __uint_as_float(v[16 * s2 + 2 * t + 1]));
                                    st_row16(qg + c0 + 16 * s2, w);
                                }
                            }
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acc_done);
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------------------------------ blocked sequences
// Forward merge of the per-key-block partials: L = log2 sum_kb 2^L_kb, O = sum_kb 2^(L_kb - L) O_kb.
// One thread per (row, head, 8 channels); po [nblk][B, N, C] bf16, pl [nblk][B, heads, N] fp32.
__global__ void __launch_bounds__(256) attn_combine_kernel(const __nv_bfloat16* __restrict__ po, const float* __restrict__ pl,
                                                           int nblk, long long rows, int n_pix, int heads,
                                                           __nv_bfloat16* __restrict__ out, float* __restrict__ lse) {
    const long long total = rows * heads * 8;
    const long long ostride = rows * heads * 64, lstride = rows * heads;
    for (long long i = blockIdx.x * 1LL * blockDim.x + threadIdx.x; i < total; i += 1LL * gridDim.x * blockDim.x) {
        const int v = static_cast<int>(i & 7);
        const long long rh = i >> 3;  // row * heads + head
        const long long row = rh / heads;
        const int h = static_cast<int>(rh - row * heads);
        const long long li = ((row / n_pix) * heads + h) * n_pix + row % n_pix;
        float m = -INFINITY;
        for (int k = 0; k < nblk; ++k) m = fmaxf(m, pl[k * lstride + li]);
        float tot = 0.f;
        for (int k = 0; k < nblk; ++k) tot += ex2(pl[k * lstride + li] - m);
        const float inv = 1.f / tot;
        float acc[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = 0.f;
        const long long off = rh * 64 + v * 8;
        for (int k = 0; k < nblk; ++k) {
            const float w = ex2(pl[k * lstride + li] - m) * inv;
            const uint4 raw = *reinterpret_cast<const uint4*>(po + k * ostride + off);
            const uint32_t ww[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                acc[2 * e] = fmaf(w, __uint_as_float(ww[e] << 16), acc[2 * e]);
                acc[2 * e + 1] = fmaf(w, __uint_as_float(ww[e] & 0xFFFF0000u), acc[2 * e + 1]);
            }
        }
        *reinterpret_cast<uint4*>(out + off) = make_uint4(pack_bf16(acc[0], acc[1]), pack_bf16(acc[2], acc[3]),
                                                          pack_bf16(acc[4], acc[5]), pack_bf16(acc[6], acc[7]));
        if (v == 0 && lse != nullptr) lse[li] = m + log2f(tot);
    }
}

// Backward merge: dqkv = sum over the nblk partial buffers (fp32 accumulation, one rounding).
__global__ void __launch_bounds__(256) attn_reduce_kernel(const __nv_bfloat16* __restrict__ part, int nblk, long long nvec,
                                                          __nv_bfloat16* __restrict__ out) {
    for (long long i = blockIdx.x * 1LL * blockDim.x + threadIdx.x; i < nvec; i += 1LL * gridDim.x * blockDim.x) {
        float acc[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = 0.f;
        for (int k = 0; k < nblk; ++k) {
            const uint4 raw = *reinterpret_cast<const uint4*>(part + (k * nvec + i) * 8);
            const uint32_t ww[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                acc[2 * e] += __uint_as_float(ww[e] << 16);
                acc[2 * e + 1] += __uint_as_float(ww[e] & 0xFFFF0000u);
            }
        }
        *reinterpret_cast<uint4*>(out + i * 8) = make_uint4(pack_bf16(acc[0], acc[1]), pack_bf16(acc[2], acc[3]),
                                                            pack_bf16(acc[4], acc[5]), pack_bf16(acc[6], acc[7]));
    }
}

}  // namespace adm

using namespace adm;

// (channel, pixel, sample) view of a [B, N, ld] bf16 tensor; box = 64 channels x box_pix pixels x box_smp samples
static int af_map(CUtensorMap* m, const void* ptr, long long ld, int n_pix, int batch, int box_pix, int box_smp) {
    const long long dims[3] = {ld, n_pix, batch};
    const long long strides[2] = {ld, ld * n_pix};
    const int box[3] = {64, box_pix, box_smp};
    return encode_map(m, ptr, 3, dims, strides, box);
}

static int af_setup(const char* what, AttnParams* p, int batch, int n_pix, int heads, float scale) {
    if (n_pix != 16 && n_pix != 64 && n_pix != 256) {
        set_error("%s: n_pix must be 16, 64 or 256 (got %d)", what, n_pix);
        return ADM_ERR_SHAPE;
    }
    if (batch <= 0 || heads <= 0) {
        set_error("%s: bad arguments", what);
        return ADM_ERR_SHAPE;
    }
    p->n_pix = n_pix; p->heads = heads; p->batch = batch; p->c = heads * 64;
    p->pack = n_pix == 256 ? 1 : 128 / n_pix;
    p->tiles = n_pix == 256 ? 2 : 1;
    p->ncols = n_pix == 256 ? 256 : 128;
    p->units = ((batch + p->pack - 1) / p->pack) * heads;
    p->nblk = 1; p->out_stride = 0; p->lse_stride = 0;
    p->scale = scale;
    p->c1 = scale * 1.4426950408889634f;
    return 0;
}

extern "C" int adm_attn_fwd_fused(const void* qkv, int batch, int n_pix, int heads, float scale, void* out, float* lse,
                                  void* stream) {
    AttnParams p;
    if (int e = af_setup("attn_fwd_fused", &p, batch, n_pix, heads, scale)) return e;
    if (((reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(out)) & 15) != 0) {
        set_error("attn_fwd_fused: pointers must be 16 B aligned");
        return ADM_ERR_SHAPE;
    }
    p.stages = n_pix == 256 ? 2 : 4;
    p.out = static_cast<__nv_bfloat16*>(out); p.lse = lse; p.o_in = nullptr;
    CUtensorMap mq;
    if (int e = af_map(&mq, qkv, 3LL * p.c, n_pix, batch, n_pix, p.pack)) return e;
    if (const cudaError_t e = set_smem_limit_once<attn_fwd_kernel>(AT_SMEM_TOTAL)) {
        set_error("attn_fwd_fused launch: %s", cudaGetErrorString(e));
        return ADM_ERR_CUDA;
    }
    const int grid = p.units < num_sms() ? p.units : num_sms();
    launch_k(attn_fwd_kernel, dim3(grid), dim3(AT_THREADS), AT_SMEM_TOTAL, static_cast<cudaStream_t>(stream), 0, mq, p);
    ADM_CHECK_LAUNCH("attn_fwd_fused");
    return 0;
}

extern "C" int adm_attn_bwd_fused(const void* da, const void* qkv, const void* out_fwd, const float* lse, int batch,
                                  int n_pix, int heads, float scale, void* dqkv, void* stream) {
    AttnParams p;
    if (int e = af_setup("attn_bwd_fused", &p, batch, n_pix, heads, scale)) return e;
    if (out_fwd == nullptr || lse == nullptr ||
        ((reinterpret_cast<uintptr_t>(da) | reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(out_fwd) |
          reinterpret_cast<uintptr_t>(dqkv)) & 15) != 0) {
        set_error("attn_bwd_fused: the forward output and log-sum-exp are required; pointers must be 16 B aligned");
        return ADM_ERR_SHAPE;
    }
    p.stages = n_pix == 256 ? 1 : 2;  // 128 KB / 64 KB per stage, next to the 32 KB dS tile
    p.out = static_cast<__nv_bfloat16*>(dqkv); p.lse = const_cast<float*>(lse);
    p.o_in = static_cast<const __nv_bfloat16*>(out_fwd);
    CUtensorMap mq, mdo;
    if (int e = af_map(&mq, qkv, 3LL * p.c, n_pix, batch, n_pix, p.pack)) return e;
    if (int e = af_map(&mdo, da, p.c, n_pix, batch, n_pix, p.pack)) return e;
    if (const cudaError_t e = set_smem_limit_once<attn_bwd_kernel>(AT_SMEM_TOTAL)) {
        set_error("attn_bwd_fused launch: %s", cudaGetErrorString(e));
        return ADM_ERR_CUDA;
    }
    const int grid = p.units < num_sms() ? p.units : num_sms();
    launch_k(attn_bwd_kernel, dim3(grid), dim3(AT_THREADS), AT_SMEM_TOTAL, static_cast<cudaStream_t>(stream), 0, mq, mdo, p);
    ADM_CHECK_LAUNCH("attn_bwd_fused");
    return 0;
}

// ------------------------------------------------------------------------------------------------ long sequences (blocked)
static int af_setup_long(const char* what, AttnParams* p, int batch, int n_pix, int heads, float scale) {
    if (n_pix < 512 || n_pix > 4096 || n_pix % 256 != 0 || batch <= 0 || heads <= 0) {
        set_error("%s: n_pix must be a multiple of 256 in [512, 4096] (got %d)", what, n_pix);
        return ADM_ERR_SHAPE;
    }
    p->n_pix = n_pix; p->heads = heads; p->batch = batch; p->c = heads * 64;
    p->pack = 1; p->tiles = 2; p->ncols = 256;
    p->nblk = n_pix / 256;
    const long long units = 1LL * batch * heads * p->nblk * p->nblk;
    if (units > INT_MAX) {
        set_error("%s: too many work units", what);
        return ADM_ERR_SHAPE;
    }
    p->units = static_cast<int>(units);
    p->scale = scale;
    p->c1 = scale * 1.4426950408889634f;
    return 0;
}

// Bytes of scratch the blocked kernels need: forward = nblk partial outputs [B, N, C] bf16 + nblk partial log-sum-exps
// [B, heads, N] fp32; backward = nblk partial dqkv [B, N, 3C] bf16.
extern "C" long long adm_attn_long_workspace(int batch, int n_pix, int heads, int backward) {
    if (n_pix < 512 || n_pix % 256 != 0 || batch <= 0 || heads <= 0) return 0;
    const long long nblk = n_pix / 256, rows = 1LL * batch * n_pix, c = 64LL * heads;
    return backward ? nblk * rows * 3 * c * 2 : nblk * (rows * c * 2 + rows * heads * 4);
}

extern "C" int adm_attn_fwd_long(const void* qkv, int batch, int n_pix, int heads, float scale, void* out, float* lse,
                                 void* work, long long work_bytes, void* stream) {
    AttnParams p;
    if (int e = af_setup_long("attn_fwd_long", &p, batch, n_pix, heads, scale)) return e;
    if (work == nullptr || work_bytes < adm_attn_long_workspace(batch, n_pix, heads, 0) ||
        ((reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(work)) & 15) != 0) {
        set_error("attn_fwd_long: workspace too small or pointers not 16 B aligned");
        return ADM_ERR_SHAPE;
    }
    const long long rows = 1LL * batch * n_pix;
    p.stages = 2;
    p.out = static_cast<__nv_bfloat16*>(work);
    p.out_stride = rows * p.c;
    p.lse = reinterpret_cast<float*>(static_cast<__nv_bfloat16*>(work) + p.nblk * p.out_stride);
    p.lse_stride = rows * heads;
    p.o_in = nullptr;
    CUtensorMap mq;
    if (int e = af_map(&mq, qkv, 3LL * p.c, n_pix, batch, 256, 1)) return e;
    if (const cudaError_t e = set_smem_limit_once<attn_fwd_kernel>(AT_SMEM_TOTAL)) {
        set_error("attn_fwd_long launch: %s", cudaGetErrorString(e));
        return ADM_ERR_CUDA;
    }
    const int grid = p.units < num_sms() ? p.units : num_sms();
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    launch_k(attn_fwd_kernel, dim3(grid), dim3(AT_THREADS), AT_SMEM_TOTAL, st, 0, mq, p);
    ADM_CHECK_LAUNCH("attn_fwd_long");
    const long long total = rows * heads * 8;
    const int cgrid = static_cast<int>(std::min<long long>((total + 255) / 256, 8LL * num_sms()));
    attn_combine_kernel<<<cgrid, 256, 0, st>>>(p.out, p.lse, p.nblk, rows, n_pix, heads, static_cast<__nv_bfloat16*>(out), lse);
    ADM_CHECK_LAUNCH("attn_combine");
    return 0;
}

extern "C" int adm_attn_bwd_long(const void* da, const void* qkv, const void* out_fwd, const float* lse, int batch,
                                 int n_pix, int heads, float scale, void* dqkv, void* work, long long work_bytes,
                                 void* stream) {
    AttnParams p;
    if (int e = af_setup_long("attn_bwd_long", &p, batch, n_pix, heads, scale)) return e;
    if (out_fwd == nullptr || lse == nullptr || work == nullptr ||
        work_bytes < adm_attn_long_workspace(batch, n_pix, heads, 1) ||
        ((reinterpret_cast<uintptr_t>(da) | reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(out_fwd) |
          reinterpret_cast<uintptr_t>(dqkv) | reinterpret_cast<uintptr_t>(work)) & 15) != 0) {
        set_error("attn_bwd_long: forward output, log-sum-exp and workspace are required; pointers must be 16 B aligned");
        return ADM_ERR_SHAPE;
    }
    const long long rows = 1LL * batch * n_pix;
    p.stages = 1;
    p.out = static_cast<__nv_bfloat16*>(work);
    p.out_stride = rows * 3 * p.c;
    p.lse = const_cast<float*>(lse);
    p.o_in = static_cast<const __nv_bfloat16*>(out_fwd);
    CUtensorMap mq, mdo;
    if (int e = af_map(&mq, qkv, 3LL * p.c, n_pix, batch, 256, 1)) return e;
    if (int e = af_map(&mdo, da, p.c, n_pix, batch, 256, 1)) return e;
    if (const cudaError_t e = set_smem_limit_once<attn_bwd_kernel>(AT_SMEM_TOTAL)) {
        set_error("attn_bwd_long launch: %s", cudaGetErrorString(e));
        return ADM_ERR_CUDA;
    }
    const int grid = p.units < num_sms() ? p.units : num_sms();
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    launch_k(attn_bwd_kernel, dim3(grid), dim3(AT_THREADS), AT_SMEM_TOTAL, st, 0, mq, mdo, p);
    ADM_CHECK_LAUNCH("attn_bwd_long");
    const long long nvec = p.out_stride / 8;
    const int rgrid = static_cast<int>(std::min<long long>((nvec + 255) / 256, 8LL * num_sms()));
    attn_reduce_kernel<<<rgrid, 256, 0, st>>>(p.out, p.nblk, nvec, static_cast<__nv_bfloat16*>(dqkv));
    ADM_CHECK_LAUNCH("attn_reduce");
    return 0;
}
