// tcgen05 / TMEM / TMA GEMM engine shared by conv3x3 (implicit GEMM fprop + dgrad), conv1x1, wgrad, Linear and the
// batched attention products.  Persistent warp-specialised kernels — tc_gemm_kernel<PLAIN|CONV|WGRAD> (general),
// tc_conv_halo_kernel (3x3 fprop/dgrad with halo re-use of the pixel operand), tc_wgrad_rows_kernel (3x3 wgrad, three
// taps per MMA), tc_conv_splitk_kernel (cluster split-K conv) — with the same roles:
//   warp 0      : TMA producer (one lane)        global -> 128B-swizzled smem ring
//   warp 1      : TMEM allocator + UMMA issuer   tcgen05.mma, fp32 accumulators in TMEM (2 x 256 columns)
//   warps 2..   : epilogue                       tcgen05.ld -> +bias, +residual, *alpha -> bf16 / fp32 / fp32 atomics
//                 (warp w drains TMEM lane quadrant w % 4; with GEMM_EPI_WARPS = 8 the two warps of a quadrant split
//                 the tile's columns)
// Tile = 128 (M) x BN (N, runtime, multiple of 16, <= 256) x 64 (K per stage, bf16 = one 128 B swizzle row).
#pragma once
#include "ptx.cuh"
#include "adm_internal.h"

namespace adm {

constexpr int GEMM_BLOCK_M = 128;
constexpr int GEMM_BLOCK_K = 64;
// Epilogue warps: 4 (one per TMEM lane quadrant) or 8 (two per quadrant, each draining half of the tile's columns).
// Measured on B200 (tools/gemm_accounting.py): 8 warps change nothing on the short-K 1x1 convs — they wait for operand
// bytes, not for the epilogue — and cost ~8 % on the small 8x8 / 4x4 tiles, so 4 it is.
constexpr int GEMM_EPI_WARPS = 4;
constexpr int EPI_HALVES = GEMM_EPI_WARPS / 4;
constexpr int GEMM_THREADS = 64 + 32 * GEMM_EPI_WARPS;   // TMA warp + MMA warp + epilogue warps
constexpr int GEMM_A_STAGE = GEMM_BLOCK_M * 128;  // 16 KB
constexpr int GEMM_SMEM_RING = 200 * 1024;        // operand ring budget
constexpr int GEMM_SMEM_AUX = 4096;               // barriers + tmem ptr (first 1 KB) + per-tile bias slices (2 x 1 KB) +
                                                  // 1 KB spare
constexpr int GEMM_SMEM_TOTAL = GEMM_SMEM_RING + GEMM_SMEM_AUX + 1024;  // + alignment slack
constexpr int GEMM_MAX_STAGES = 8;

enum GemmMode { GEMM_PLAIN = 0, GEMM_CONV = 1, GEMM_WGRAD = 2 };
enum GemmOut { OUT_BF16 = 0, OUT_F32 = 1, OUT_F32_ATOMIC = 2 };

struct GemmParams {
    // ---- tile space: tile = (((bt * splits + sp) * m_tiles + mt) * n_tiles + nt)
    int m_tiles, n_tiles, batches, splits;
    int k_iters;  // K iterations (of 64) per split
    int k_total;  // total K iterations (last split may be shorter)
    int ksplit;   // tc_conv_splitk_kernel: CTAs of a cluster that split the K range of one tile (reduced through DSMEM)
    int bn;       // N tile
    int a_mn, b_mn;
    int M, N;  // valid rows (per batch) / cols
    // ---- conv / wgrad geometry (NHWC tensors; box = bw x bh x bni pixels)
    int H, W, bw, bh, bni, tiles_w, tiles_h;
    int ntaps;     // kw * kw: 1, 9, 25 or 49 (odd square kernels, 'same' padding kw / 2)
    int kw;        // taps per kernel row (1, 3, 5, 7)
    int cchunks;   // 64-channel chunks per tap (both A sources)
    int cchunks1;  // chunks taken from A source 1; the rest come from A source 2 (fused channel concat)
    int n_split;   // wgrad: output columns (per tap) served by X source 1; the rest by X source 2
    int co_chunks; // tap-row wgrad: 64-channel chunks of dY (M chunks = 3 dy x co_chunks)
    // ---- plain / batched coordinates: bt -> (b_hi = bt / bdiv, b_lo = bt % bdiv)
    int bdiv;
    int a_c0, a_c0_lo, a_c1, a_c1_lo, a_bhi, a_blo;
    int b_c0, b_c0_lo, b_c1, b_c1_lo, b_bhi, b_blo;
    // ---- epilogue
    void* C;
    long long ldc, c_bhi, c_blo;  // element strides
    int c_col_lo;                 // extra column offset per b_lo
    const float* bias;            // [N] or null
    const __nv_bfloat16* residual;
    long long ldr;
    float alpha;
    int out_mode;
    const int* row_map;  // plain / wgrad tiles: GEMM row r is stored at output row row_map[r] (nullptr = identity)
};

__device__ __forceinline__ void decode_pix(const GemmParams& p, int idx, int& n0, int& h0, int& w0) {
    const int per = p.tiles_w * p.tiles_h;
    n0 = (idx / per) * p.bni;
    const int r = idx % per;
    h0 = (r / p.tiles_w) * p.bh;
    w0 = (r % p.tiles_w) * p.bw;
}

// Pixel-box coordinates of consecutive k-iterations without per-iteration divisions (the producer is ONE thread: a few
// runtime integer divisions per k-iteration are a measurable share of its budget).
struct PixWalker {
    int n0, h0, w0;
    __device__ __forceinline__ PixWalker(const GemmParams& p, int idx) { decode_pix(p, idx, n0, h0, w0); }
    __device__ __forceinline__ void advance(const GemmParams& p) {
        w0 += p.bw;
        if (w0 >= p.W) {
            w0 = 0;
            h0 += p.bh;
            if (h0 >= p.H) { h0 = 0; n0 += p.bni; }
        }
    }
};

// The epilogue warps stage the tile's bias slice (bn <= 256 floats, zero beyond N) in shared memory BEFORE waiting for the
// accumulator: per-chunk __ldg of the bias missed L1 behind the streaming stores and cost ~30 us on the epilogue-bound
// 1x1 convs.  `t` = epilogue thread index; named barrier 1 covers exactly the epilogue threads.
__device__ __forceinline__ void stage_bias(const GemmParams& p, float* sbias, int col_base, int t) {
    if (p.bias == nullptr) return;
    for (int c = t; c < p.bn; c += 32 * GEMM_EPI_WARPS)
        sbias[c] = (col_base + c < p.N) ? __ldg(p.bias + col_base + c) : 0.f;
    asm volatile("bar.sync 1, %0;" ::"n"(32 * GEMM_EPI_WARPS) : "memory");
}

// Epilogue of one accumulator tile for one thread (= one output row): TMEM -> registers in groups of up to 64 columns
// (four 32x32b.x16 loads in flight behind ONE wait, with the residual row segment prefetched behind the same wait),
// then alpha * acc + bias + residual -> bf16 / fp32 / fp32 atomics.  c_off / r_off: element offsets of this row in the
// output and the residual (before the column); col_shift: extra output column offset (batched GEMMs); the tile columns
// drained are [c_begin, ncols) (multiples of 16).
__device__ __forceinline__ void epilogue_row(const GemmParams& p, uint32_t taddr, int col_base, int col_shift,
                                             long long c_off, long long r_off, bool row_ok, const float* sbias,
                                             int c_begin, int ncols) {
    for (int c0 = c_begin; c0 < ncols; c0 += 64) {
        if (col_base + c0 >= p.N) break;  // warp-uniform
        uint32_t v[4][16];
        uint4 rr[4][2];
        const int nsub = min(4, (ncols - c0) >> 4);
        __syncwarp();
#pragma unroll
        for (int s = 0; s < 4; ++s)
            if (s < nsub) tmem_ld_x16(taddr + c0 + 16 * s, v[s]);
        // residual prefetch (aligned full chunks only; the ragged path re-reads below)
        const bool res_vec = p.residual != nullptr && row_ok &&
                             ((reinterpret_cast<uintptr_t>(p.residual + r_off + col_base + c0) & 15) == 0);
        if (res_vec) {
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const int col = col_base + c0 + 16 * s;
                if (s < nsub && col + 16 <= p.N) {
                    const uint4* rp = reinterpret_cast<const uint4*>(p.residual + r_off + col);
                    rr[s][0] = rp[0];
                    rr[s][1] = rp[1];
                }
            }
        }
        tmem_ld_wait();
        if (!row_ok) continue;
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            if (s >= nsub) break;
            const int col = col_base + c0 + 16 * s;
            if (col >= p.N) break;
            float f[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[s][j]) * p.alpha;
            const bool full = (col + 16 <= p.N);
            if (p.bias != nullptr) {  // this tile's bias slice was staged in shared memory (zero beyond N)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 b4 = *reinterpret_cast<const float4*>(sbias + c0 + 16 * s + 4 * j);
                    f[4 * j] += b4.x; f[4 * j + 1] += b4.y; f[4 * j + 2] += b4.z; f[4 * j + 3] += b4.w;
                }
            }
            if (p.residual != nullptr) {
                if (res_vec && full) {
                    const uint32_t w[8] = {rr[s][0].x, rr[s][0].y, rr[s][0].z, rr[s][0].w,
                                           rr[s][1].x, rr[s][1].y, rr[s][1].z, rr[s][1].w};
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        f[2 * j] += __uint_as_float(w[j] << 16);
                        f[2 * j + 1] += __uint_as_float(w[j] & 0xFFFF0000u);
                    }
                } else if (row_ok) {
                    const __nv_bfloat16* rp = p.residual + r_off + col;
                    for (int j = 0; j < 16; ++j)
                        if (col + j < p.N) f[j] += __bfloat162float(rp[j]);
                }
            }
            const long long off = c_off + col_shift + col;
            if (p.out_mode == OUT_BF16) {
                __nv_bfloat16* cp = reinterpret_cast<__nv_bfloat16*>(p.C) + off;
                if (full && ((reinterpret_cast<uintptr_t>(cp) & 15) == 0)) {
                    uint32_t w[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const __nv_bfloat162 b2 = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
                        w[j] = *reinterpret_cast<const uint32_t*>(&b2);
                    }
                    if ((reinterpret_cast<uintptr_t>(cp) & 31) == 0) {
                        // one 256-bit store = one full 32 B sector per thread (sm_100 st.global.v8): rows of a tile are
                        // scattered over 128 different lines, so two 16 B halves would each be a partial-sector write
                        asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(cp), "r"(w[0]),
                                     "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
                                     : "memory");
                    } else {
                        *reinterpret_cast<uint4*>(cp) = make_uint4(w[0], w[1], w[2], w[3]);
                        *reinterpret_cast<uint4*>(cp + 8) = make_uint4(w[4], w[5], w[6], w[7]);
                    }
                } else {
                    for (int j = 0; j < 16; ++j)
                        if (col + j < p.N) cp[j] = __float2bfloat16(f[j]);
                }
            } else if (p.out_mode == OUT_F32) {
                float* cp = reinterpret_cast<float*>(p.C) + off;
                if (full && ((reinterpret_cast<uintptr_t>(cp) & 15) == 0)) {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<float4*>(cp + 4 * j) =
                            make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
                } else {
                    for (int j = 0; j < 16; ++j)
                        if (col + j < p.N) cp[j] = f[j];
                }
            } else {
                float* cp = reinterpret_cast<float*>(p.C) + off;
                if (full && ((reinterpret_cast<uintptr_t>(cp) & 15) == 0)) {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        atomicAdd(reinterpret_cast<float4*>(cp + 4 * j),
                                  make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]));
                } else {
                    for (int j = 0; j < 16; ++j)
                        if (col + j < p.N) atomicAdd(cp + j, f[j]);
                }
            }
        }
    }
}

// The epilogue warps' persistent loop (4 warps, one TMEM lane quadrant each): per tile, stage the bias slice, wait for
// the accumulator, drain it through epilogue_row, release it.  Shared by tc_gemm_kernel and tc_conv_halo_kernel.
template <int MODE>
__device__ __forceinline__ void epilogue_warps(const GemmParams& p, uint8_t* smem, uint32_t tmem_base,
                                               uint64_t* tfull_bar, uint64_t* tempty_bar, int warp, int lane,
                                               int num_tiles) {
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;   // which half of the tile's columns this warp drains
    const int m = quad * 32 + lane;     // row inside the tile
    const int c_split = EPI_HALVES == 2 ? (((p.bn >> 1) + 15) & ~15) : p.bn;
    const int c_begin = half ? c_split : 0, c_end = half ? p.bn : c_split;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int nt = tile % p.n_tiles;
        int r = tile / p.n_tiles;
        const int mt = r % p.m_tiles;
        r /= p.m_tiles;
        const int bt = r / p.splits;
        const int b_hi = bt / p.bdiv, b_lo = bt % p.bdiv;

        long long row_off;  // element offset of this thread's output row (before column)
        bool row_ok;
        if (MODE == GEMM_CONV) {
            int n0, h0, w0;
            decode_pix(p, mt, n0, h0, w0);
            const int wi = m % p.bw, hi = (m / p.bw) % p.bh, ni = m / (p.bw * p.bh);
            const long long pix = (static_cast<long long>(n0 + ni) * p.H + (h0 + hi)) * p.W + (w0 + wi);
            row_ok = pix < p.M;
            row_off = pix;
        } else {
            const int row = mt * 128 + m;
            row_ok = row < p.M;
            row_off = (p.row_map != nullptr && row_ok) ? __ldg(p.row_map + row) : row;
        }
        const long long c_base = b_hi * p.c_bhi + b_lo * p.c_blo + row_off * p.ldc;
        const int col_base = nt * p.bn;           // column inside [0, N)
        const int col_shift = b_lo * p.c_col_lo;  // extra offset in the output row

        float* sbias = reinterpret_cast<float*>(smem + GEMM_SMEM_RING + 1024) + acc * 256;
        stage_bias(p, sbias, col_base, (warp - 2) * 32 + lane);
        mbar_wait(&tfull_bar[acc], acc_phase, 4);
        tc_fence_after();
        const uint32_t taddr = tmem_base + acc * 256 + (static_cast<uint32_t>(quad * 32) << 16);
        epilogue_row(p, taddr, col_base, col_shift, c_base, row_off * p.ldr, row_ok, sbias, c_begin, c_end);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
}

template <int MODE>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2,
               const __grid_constant__ CUtensorMap tmB, const __grid_constant__ GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int stage_bytes = GEMM_A_STAGE + p.bn * 128;
    int num_stages = GEMM_SMEM_RING / stage_bytes;
    if (num_stages > GEMM_MAX_STAGES) num_stages = GEMM_MAX_STAGES;

    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + GEMM_SMEM_RING);
    uint64_t* empty_bar = full_bar + GEMM_MAX_STAGES;
    uint64_t* tfull_bar = empty_bar + GEMM_MAX_STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmA2);
        tma_prefetch_desc(&tmB);
        for (int i = 0; i < num_stages; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull_bar[i], 1);
            mbar_init(&tempty_bar[i], GEMM_EPI_WARPS);
        }
        fence_barrier_init();
        fence_proxy_async_smem();
    }
    if (warp == 1) tmem_alloc(tmem_ptr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    const int num_tiles = p.batches * p.splits * p.m_tiles * p.n_tiles;

    if (warp == 0) {
        // =========================================================== TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int nt = tile % p.n_tiles;
                int r = tile / p.n_tiles;
                const int mt = r % p.m_tiles;
                r /= p.m_tiles;
                const int sp = r % p.splits;
                const int bt = r / p.splits;
                const int k_begin = sp * p.k_iters;
                const int k_end = min(p.k_total, k_begin + p.k_iters);
                int n0 = 0, h0 = 0, w0 = 0;
                if (MODE == GEMM_CONV) decode_pix(p, mt, n0, h0, w0);
                const int b_hi = bt / p.bdiv, b_lo = bt % p.bdiv;
                int tap = 0, kc = 0;  // conv: ki = tap * cchunks + kc, walked without divisions
                if (MODE == GEMM_CONV) { tap = k_begin / p.cchunks; kc = k_begin % p.cchunks; }
                PixWalker px(p, MODE == GEMM_WGRAD ? k_begin : 0);
                for (int ki = k_begin; ki < k_end; ++ki) {
                    mbar_wait(&empty_bar[stage], phase ^ 1, 1);
                    uint8_t* sa = smem + stage * stage_bytes;
                    uint8_t* sb = sa + GEMM_A_STAGE;
                    mbar_expect_tx(&full_bar[stage], stage_bytes);
                    if (MODE == GEMM_CONV) {
                        int dh = 0, dw = 0;
                        if (p.kw == 3) { dh = tap / 3 - 1; dw = tap % 3 - 1; }
                        else if (p.kw > 1) { dh = tap / p.kw - (p.kw >> 1); dw = tap % p.kw - (p.kw >> 1); }
                        if (kc < p.cchunks1)
                            tma_load_4d(sa, &tmA, &full_bar[stage], kc * 64, w0 + dw, h0 + dh, n0);
                        else
                            tma_load_4d(sa, &tmA2, &full_bar[stage], (kc - p.cchunks1) * 64, w0 + dw, h0 + dh, n0);
                        if (!p.b_mn) {
                            // weights [Nout][ntaps * Kpad], K-major
                            tma_load_2d(sb, &tmB, &full_bar[stage], ki * 64, nt * p.bn);
                        } else {
                            // dgrad on the fprop-packed weights viewed as (N_gemm = Cin, taps, K_gemm = Cout): the
                            // spatial flip is the tap reversal, the transpose is the MN-major operand mode.
                            for (int c = 0; c * 64 < p.bn; ++c)
                                tma_load_3d(sb + c * 8192, &tmB, &full_bar[stage], nt * p.bn + c * 64,
                                            p.ntaps - 1 - tap, kc * 64);
                        }
                        if (++kc == p.cchunks) { kc = 0; ++tap; }
                    } else if (MODE == GEMM_WGRAD) {
                        // K runs over pixel blocks of 64; bt = tap.  A = dY (MN-major), B = shifted X (MN-major).
                        n0 = px.n0; h0 = px.h0; w0 = px.w0;
                        px.advance(p);
                        int dh = 0, dw = 0;
                        if (p.kw == 3) { dh = bt / 3 - 1; dw = bt % 3 - 1; }
                        else if (p.kw > 1) { dh = bt / p.kw - (p.kw >> 1); dw = bt % p.kw - (p.kw >> 1); }
                        tma_load_4d(sa, &tmA, &full_bar[stage], mt * 128, w0, h0, n0);
                        tma_load_4d(sa + 8192, &tmA, &full_bar[stage], mt * 128 + 64, w0, h0, n0);
                        // fused channel concat on the X side: columns >= n_split come from the second source
                        const int ncol = nt * p.bn;
                        const bool src2 = ncol >= p.n_split;
                        const CUtensorMap* mb = src2 ? &tmA2 : &tmB;
                        const int nc = src2 ? ncol - p.n_split : ncol;
                        for (int c = 0; c * 64 < p.bn; ++c)
                            tma_load_4d(sb + c * 8192, mb, &full_bar[stage], nc + c * 64, w0 + dw, h0 + dh, n0);
                    } else {
                        const int a0 = p.a_c0 + b_lo * p.a_c0_lo, a1 = p.a_c1 + b_lo * p.a_c1_lo;
                        const int a2 = b_hi * p.a_bhi + b_lo * p.a_blo;
                        const int b0 = p.b_c0 + b_lo * p.b_c0_lo, b1 = p.b_c1 + b_lo * p.b_c1_lo;
                        const int b2 = b_hi * p.b_bhi + b_lo * p.b_blo;
                        if (!p.a_mn) {
                            tma_load_3d(sa, &tmA, &full_bar[stage], a0 + ki * 64, a1 + mt * 128, a2);
                        } else {
                            tma_load_3d(sa, &tmA, &full_bar[stage], a0 + mt * 128, a1 + ki * 64, a2);
                            tma_load_3d(sa + 8192, &tmA, &full_bar[stage], a0 + mt * 128 + 64, a1 + ki * 64, a2);
                        }
                        if (!p.b_mn) {
                            tma_load_3d(sb, &tmB, &full_bar[stage], b0 + ki * 64, b1 + nt * p.bn, b2);
                        } else {
                            for (int c = 0; c * 64 < p.bn; ++c)
                                tma_load_3d(sb + c * 8192, &tmB, &full_bar[stage], b0 + nt * p.bn + c * 64,
                                            b1 + ki * 64, b2);
                        }
                    }
                    if (++stage == num_stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // =========================================================== UMMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc_bf16(GEMM_BLOCK_M, p.bn, p.a_mn, p.b_mn);
            const uint32_t a_lbo = p.a_mn ? 8192u : 16u, b_lbo = p.b_mn ? 8192u : 16u;
            // descriptor constants and k-step strides (in 16 B units) are hoisted: this thread's instruction stream is
            // the critical path of the main loop
            const uint32_t a_kstep = (p.a_mn ? 2048u : 32u) >> 4, b_kstep = (p.b_mn ? 2048u : 32u) >> 4;
            const uint64_t da0 = make_smem_desc(0, a_lbo, 1024), db0 = make_smem_desc(0, b_lbo, 1024);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int sp = (tile / (p.n_tiles * p.m_tiles)) % p.splits;
                const int k_begin = sp * p.k_iters;
                const int k_end = min(p.k_total, k_begin + p.k_iters);
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1, 2);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * 256;
                for (int ki = k_begin; ki < k_end; ++ki) {
                    mbar_wait(&full_bar[stage], phase, 3);
                    tc_fence_after();
                    const uint32_t sa16 = (smem_u32(smem + stage * stage_bytes) & 0x3FFFFu) >> 4;
                    const uint64_t da = da0 + sa16, db = db0 + (sa16 + (GEMM_A_STAGE >> 4));
#pragma unroll
                    for (int k = 0; k < GEMM_BLOCK_K / 16; ++k)
                        umma_bf16(tmem_d, da + k * a_kstep, db + k * b_kstep, idesc, (ki > k_begin || k > 0) ? 1u : 0u);
                    umma_commit(&empty_bar[stage]);
                    if (++stage == num_stages) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tfull_bar[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // =========================================================== epilogue (4 warps, one TMEM lane quadrant each)
        epilogue_warps<MODE>(p, smem, tmem_base, tfull_bar, tempty_bar, warp, lane, num_tiles);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------------------------------ cluster split-K conv
// Implicit-GEMM conv (fprop / dgrad, 3x3 or 1x1) for problems with too few 128 x bn output tiles to fill the GPU (the 4x4
// level: 2048 pixels x 384 channels = 48 tiles of 128 x 128, each with a K loop of 54-108 iterations).  A thread-block
// cluster of ksplit CTAs shares ONE output tile: CTA r multiplies K iterations [r * k_iters, (r + 1) * k_iters) into its own
// TMEM accumulator; the non-leaders then park their fp32 partial tiles in their (now idle) operand ring, signal the leader's
// mbarrier across the cluster, and the leader adds them through distributed shared memory (ld.shared::cluster) into its
// accumulator before the ordinary epilogue.  One tile per CTA (grid = tiles x ksplit); roles as in tc_gemm_kernel.
__device__ __forceinline__ uint32_t mapa_shared(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ float4 ld_dsmem_f4(uint32_t caddr) {
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(caddr));
    return v;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t caddr) {  // release at cluster scope
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(caddr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity, int code) {  // acquire at cluster scope
    const long long t0 = clock64();
    uint32_t ok = 0;
    while (!ok) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (!ok && clock64() - t0 > 8000000000LL) {
            g_device_error = code;
            __threadfence_system();
            asm volatile("trap;");
        }
    }
}

__global__ void __launch_bounds__(GEMM_THREADS, 1)
tc_conv_splitk_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2,
                      const __grid_constant__ CUtensorMap tmB, const __grid_constant__ GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int stage_bytes = GEMM_A_STAGE + p.bn * 128;
    int num_stages = GEMM_SMEM_RING / stage_bytes;
    if (num_stages > GEMM_MAX_STAGES) num_stages = GEMM_MAX_STAGES;

    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + GEMM_SMEM_RING);
    uint64_t* empty_bar = full_bar + GEMM_MAX_STAGES;
    uint64_t* tfull_bar = empty_bar + GEMM_MAX_STAGES;
    uint64_t* peers_bar = tfull_bar + 1;  // leader: the non-leaders' partial tiles are parked
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(peers_bar + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int rank = static_cast<int>(cluster_ctarank());
    const int tile = blockIdx.x / p.ksplit;
    const int nt = tile % p.n_tiles, mt = tile / p.n_tiles;
    const int k_begin = rank * p.k_iters;
    const int k_end = min(p.k_total, k_begin + p.k_iters);

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmA2);
        tma_prefetch_desc(&tmB);
        for (int i = 0; i < num_stages; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        mbar_init(tfull_bar, 1);
        mbar_init(peers_bar, (p.ksplit - 1) * GEMM_EPI_WARPS);
        fence_barrier_init();
        fence_proxy_async_smem();
    }
    if (warp == 1) tmem_alloc(tmem_ptr, 256);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // the leader's peers_bar is initialised before any remote arrive
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    int n0, h0, w0;
    decode_pix(p, mt, n0, h0, w0);
    if (warp == 0) {
        // =========================================================== TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int tap = k_begin / p.cchunks, kc = k_begin % p.cchunks;
            for (int ki = k_begin; ki < k_end; ++ki) {
                mbar_wait(&empty_bar[stage], phase ^ 1, 41);
                uint8_t* sa = smem + stage * stage_bytes;
                uint8_t* sb = sa + GEMM_A_STAGE;
                mbar_expect_tx(&full_bar[stage], stage_bytes);
                int dh = 0, dw = 0;
                if (p.kw == 3) { dh = tap / 3 - 1; dw = tap % 3 - 1; }
                        else if (p.kw > 1) { dh = tap / p.kw - (p.kw >> 1); dw = tap % p.kw - (p.kw >> 1); }
                if (kc < p.cchunks1)
                    tma_load_4d(sa, &tmA, &full_bar[stage], kc * 64, w0 + dw, h0 + dh, n0);
                else
                    tma_load_4d(sa, &tmA2, &full_bar[stage], (kc - p.cchunks1) * 64, w0 + dw, h0 + dh, n0);
                if (!p.b_mn) {
                    tma_load_2d(sb, &tmB, &full_bar[stage], ki * 64, nt * p.bn);
                } else {
                    for (int c = 0; c * 64 < p.bn; ++c)
                        tma_load_3d(sb + c * 8192, &tmB, &full_bar[stage], nt * p.bn + c * 64, p.ntaps - 1 - tap, kc * 64);
                }
                if (++kc == p.cchunks) { kc = 0; ++tap; }
                if (++stage == num_stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // =========================================================== UMMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc_bf16(GEMM_BLOCK_M, p.bn, 0, p.b_mn);
            const uint32_t b_lbo = p.b_mn ? 8192u : 16u;
            const uint32_t b_kstep = (p.b_mn ? 2048u : 32u) >> 4;
            const uint64_t da0 = make_smem_desc(0, 16u, 1024), db0 = make_smem_desc(0, b_lbo, 1024);
            int stage = 0;
            uint32_t phase = 0;
            for (int ki = k_begin; ki < k_end; ++ki) {
                mbar_wait(&full_bar[stage], phase, 43);
                tc_fence_after();
                // In a non-leader CTA of a cluster the shared-window address carries bits above the 14-bit descriptor field:
                // unmasked they spill into the leading-byte-offset field (which only MN-major multi-chunk B reads).
                const uint32_t sa16 = (smem_u32(smem + stage * stage_bytes) & 0x3FFFFu) >> 4;
                const uint64_t da = da0 + sa16, db = db0 + (sa16 + (GEMM_A_STAGE >> 4));
#pragma unroll
                for (int k = 0; k < GEMM_BLOCK_K / 16; ++k)
                    umma_bf16(tmem_base, da + 2 * k, db + k * b_kstep, idesc, (ki > k_begin || k > 0) ? 1u : 0u);
                umma_commit(&empty_bar[stage]);
                if (++stage == num_stages) { stage = 0; phase ^= 1; }
            }
            umma_commit(tfull_bar);
        }
    } else {
        // =========================================================== epilogue (4 warps, one TMEM lane quadrant each)
        const int quad = warp & 3;
        const int m = quad * 32 + lane;
        const int wi = m % p.bw, hi = (m / p.bw) % p.bh, ni = m / (p.bw * p.bh);
        const long long pix = (static_cast<long long>(n0 + ni) * p.H + (h0 + hi)) * p.W + (w0 + wi);
        const bool row_ok = pix < p.M;
        const int col_base = nt * p.bn;
        float* sbias = reinterpret_cast<float*>(smem + GEMM_SMEM_RING + 1024);
        if (rank == 0) stage_bias(p, sbias, col_base, (warp - 2) * 32 + lane);
        mbar_wait(tfull_bar, 0, 44);  // this CTA's K range is in its accumulator; its operand ring is idle from here on
        tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
        float4* park = reinterpret_cast<float4*>(smem);  // [bn / 4][128 rows] float4: lanes write consecutive 16 B
        if (rank != 0) {
            for (int c0 = 0; c0 < p.bn; c0 += 16) {
                uint32_t v[16];
                __syncwarp();
                tmem_ld_x16(taddr + c0, v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    park[((c0 >> 2) + j) * 128 + m] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                                                   __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
            }
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(mapa_shared(smem_u32(peers_bar), 0));
        } else {
            if (p.ksplit > 1) {
                mbar_wait_cluster(peers_bar, 0, 45);
                for (int c0 = 0; c0 < p.bn; c0 += 16) {
                    uint32_t v[16];
                    __syncwarp();
                    tmem_ld_x16(taddr + c0, v);
                    tmem_ld_wait();
                    for (int r = 1; r < p.ksplit; ++r) {
                        const uint32_t peer = mapa_shared(smem_u32(park), static_cast<uint32_t>(r));
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const float4 t = ld_dsmem_f4(peer + (((c0 >> 2) + j) * 128 + m) * 16);
                            v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) + t.x);
                            v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + t.y);
                            v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + t.z);
                            v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + t.w);
                        }
                    }
                    __syncwarp();
                    tmem_st_x16(taddr + c0, v);  // the total goes back into the accumulator: the epilogue below is unchanged
                }
                tmem_st_wait();
            }
            epilogue_row(p, taddr, col_base, 0, pix * p.ldc, pix * p.ldr, row_ok, sbias, 0, p.bn);
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // no CTA exits (or frees TMEM) while the leader may still read its shared memory
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 256);
    }
}

// ------------------------------------------------------------------------------------------------ halo conv kernel
// 3x3 implicit-GEMM conv whose pixel operand is loaded ONCE per 64-channel chunk instead of once per tap.  The pixel
// tile is 8 (w) x 16 (h); its 10 x 18 halo (zero-filled outside the image by TMA) lands in shared memory as 180 rows of
// 128 B.  A tap (dy, dx) is then just a shifted window of that halo: the UMMA A descriptor starts at row dy*10 + dx and
// walks its sixteen 8-row groups (= pixel rows of the tile) SBO = 10 rows apart.  The 128B-swizzle XOR is a function of
// the absolute shared-memory address on both the TMA and the UMMA side, so an unaligned start and a group stride that
// is not a multiple of 1024 B read back exactly what TMA wrote (tools/exp/umma_row_offset.cu, measured on B200).
// Per k-iteration (one tap x 64 channels) the SM ingests bn*128 B of weights + 23 KB / 9 of pixels instead of
// bn*128 B + 16 KB: -34 % for bn = 192.  K order is chunk-major (chunk, tap) — the weight TMA coordinates follow.
// Roles, accumulators and the epilogue are those of tc_gemm_kernel; two rings replace the single one:
//   halo ring  : HALO_BUFS buffers, filled one chunk step AHEAD (across tiles), released by a commit after the 9th tap
//   weight ring: as many bn*128 B stages as fit beside it
constexpr int HALO_W = 10, HALO_H = 18;
constexpr int HALO_TX_BYTES = HALO_W * HALO_H * 128;  // 23040
constexpr int HALO_BYTES = 23 * 1024;                 // buffer pitch, 1024-aligned
constexpr int HALO_BUFS = 3;

__global__ void __launch_bounds__(GEMM_THREADS, 1)
tc_conv_halo_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2,
                    const __grid_constant__ CUtensorMap tmB, const __grid_constant__ GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int b_bytes = p.bn * 128;
    int nb = (GEMM_SMEM_RING - HALO_BUFS * HALO_BYTES) / b_bytes;
    if (nb > GEMM_MAX_STAGES) nb = GEMM_MAX_STAGES;
    uint8_t* b_ring = smem + HALO_BUFS * HALO_BYTES;

    uint64_t* bfull = reinterpret_cast<uint64_t*>(smem + GEMM_SMEM_RING);
    uint64_t* bempty = bfull + GEMM_MAX_STAGES;
    uint64_t* tfull_bar = bempty + GEMM_MAX_STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint64_t* hfull = tempty_bar + 2;  // halo buffer landed
    uint64_t* hempty = hfull + HALO_BUFS;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(hempty + HALO_BUFS);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmA2);
        tma_prefetch_desc(&tmB);
        for (int i = 0; i < nb; ++i) {
            mbar_init(&bfull[i], 1);
            mbar_init(&bempty[i], 1);
        }
        for (int i = 0; i < HALO_BUFS; ++i) {
            mbar_init(&hfull[i], 1);
            mbar_init(&hempty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull_bar[i], 1);
            mbar_init(&tempty_bar[i], GEMM_EPI_WARPS);
        }
        fence_barrier_init();
        fence_proxy_async_smem();
    }
    if (warp == 1) tmem_alloc(tmem_ptr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    const int num_tiles = p.m_tiles * p.n_tiles;

    if (warp == 0) {
        // =========================================================== TMA producer
        if (lane == 0) {
            int hs = 0, bs = 0;
            uint32_t hphase = 0, bphase = 0;
            auto load_halo = [&](int tile, int kc) {
                int n0, h0, w0;
                decode_pix(p, (tile / p.n_tiles) % p.m_tiles, n0, h0, w0);
                mbar_wait(&hempty[hs], hphase ^ 1, 5);
                mbar_expect_tx(&hfull[hs], HALO_TX_BYTES);
                uint8_t* dst = smem + hs * HALO_BYTES;
                if (kc < p.cchunks1)
                    tma_load_4d(dst, &tmA, &hfull[hs], kc * 64, w0 - 1, h0 - 1, n0);
                else
                    tma_load_4d(dst, &tmA2, &hfull[hs], (kc - p.cchunks1) * 64, w0 - 1, h0 - 1, n0);
                if (++hs == HALO_BUFS) { hs = 0; hphase ^= 1; }
            };
            // Halo loads run AHEAD of the weight tiles by `ahead` chunk steps (a cursor over (tile, chunk) that only this
            // thread advances): 1 step hides the TMA latency under the nine MMAs of the current chunk; three buffers:
            // loading, multiplying, draining.
            int cur_tile = blockIdx.x, cur_kc = 0;
            auto next_halo = [&]() {
                if (cur_tile >= num_tiles) return;
                load_halo(cur_tile, cur_kc);
                if (++cur_kc == p.cchunks) { cur_kc = 0; cur_tile += gridDim.x; }
            };
            const int ahead = 1;  // (2 makes this thread wait for the buffer still being multiplied before it issues weights)
            for (int i = 0; i < ahead; ++i) next_halo();
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int nt = tile % p.n_tiles;
                for (int kc = 0; kc < p.cchunks; ++kc) {
                    next_halo();  // the halo `ahead` steps from now goes out before this step's nine weight tiles
                    for (int tap = 0; tap < 9; ++tap) {
                        mbar_wait(&bempty[bs], bphase ^ 1, 1);
                        uint8_t* sb = b_ring + bs * b_bytes;
                        mbar_expect_tx(&bfull[bs], b_bytes);
                        if (!p.b_mn) {
                            tma_load_2d(sb, &tmB, &bfull[bs], (tap * p.cchunks + kc) * 64, nt * p.bn);
                        } else {
                            for (int c = 0; c * 64 < p.bn; ++c)
                                tma_load_3d(sb + c * 8192, &tmB, &bfull[bs], nt * p.bn + c * 64, 8 - tap, kc * 64);
                        }
                        if (++bs == nb) { bs = 0; bphase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // =========================================================== UMMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc_bf16(GEMM_BLOCK_M, p.bn, 0, p.b_mn);
            const uint32_t b_lbo = p.b_mn ? 8192u : 16u;
            const uint32_t b_kstep = (p.b_mn ? 2048u : 32u) >> 4;
            const uint64_t da0 = make_smem_desc(0, 16, HALO_W * 128), db0 = make_smem_desc(0, b_lbo, 1024);
            int hs = 0, bs = 0;
            uint32_t hphase = 0, bphase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1, 2);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * 256;
                for (int kc = 0; kc < p.cchunks; ++kc) {
                    mbar_wait(&hfull[hs], hphase, 6);
                    tc_fence_after();
                    const uint64_t da_halo = da0 + (smem_u32(smem + hs * HALO_BYTES) >> 4);
#pragma unroll
                    for (int tap = 0; tap < 9; ++tap) {
                        mbar_wait(&bfull[bs], bphase, 3);
                        tc_fence_after();
                        const uint64_t da = da_halo + ((tap / 3) * HALO_W + tap % 3) * 8;  // (128 B rows) >> 4
                        const uint64_t db = db0 + (smem_u32(b_ring + bs * b_bytes) >> 4);
#pragma unroll
                        for (int k = 0; k < GEMM_BLOCK_K / 16; ++k)
                            umma_bf16(tmem_d, da + 2 * k, db + k * b_kstep, idesc, (kc > 0 || tap > 0 || k > 0) ? 1u : 0u);
                        umma_commit(&bempty[bs]);
                        if (++bs == nb) { bs = 0; bphase ^= 1; }
                    }
                    umma_commit(&hempty[hs]);
                    if (++hs == HALO_BUFS) { hs = 0; hphase ^= 1; }
                }
                umma_commit(&tfull_bar[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        epilogue_warps<GEMM_CONV>(p, smem, tmem_base, tfull_bar, tempty_bar, warp, lane, num_tiles);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------------------------------ tap-row wgrad kernel
// 3x3 weight gradient  dW[co][dy][dx][ci] = sum_q dY[q - (dy-1, 0)][co] * X[q + (0, dx-1)][ci]  with the vertical shift
// on the dY side and the horizontal shift on the X side, so that
//   * N = 192 = the THREE dx taps of one 64-channel X chunk, read as three windows of ONE w-halo tile (bw+2 pixels per
//     row): the MN-major B descriptor's chunk stride (LBO) is a single 128 B row — one MMA covers three taps;
//   * M = 128 = two (dy, 64-channel dY chunk) pairs, each an ordinary 64-pixel box loaded with its own vertical offset
//     (zero outside the image): Cout = 192 gives 9 M chunks = 4.5 tiles instead of 9 x 2 half-empty ones.
// Per k-iteration (64 pixels) an SM ingests 16 KB + ~9 KB for 128 x 192 x 64 MACs, against 16 KB + 24 KB per tap before.
// K = pixels (split across CTAs, fp32 atomics into the gradient arena), roles as in tc_gemm_kernel.
// K = pixels (split across CTAs, fp32 atomics into the gradient arena), roles as in tc_gemm_kernel.
__global__ void __launch_bounds__(GEMM_THREADS, 1)
tc_wgrad_rows_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                     const __grid_constant__ CUtensorMap tmB2, const __grid_constant__ GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int halo_w = p.bw + 2;
    const int b_tx = p.bh * halo_w * 128;
    const int stage_bytes = GEMM_A_STAGE + ((b_tx + 1023) & ~1023);
    int num_stages = GEMM_SMEM_RING / stage_bytes;
    if (num_stages > GEMM_MAX_STAGES) num_stages = GEMM_MAX_STAGES;

    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + GEMM_SMEM_RING);
    uint64_t* empty_bar = full_bar + GEMM_MAX_STAGES;
    uint64_t* tfull_bar = empty_bar + GEMM_MAX_STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        tma_prefetch_desc(&tmB2);
        for (int i = 0; i < num_stages; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull_bar[i], 1);
            mbar_init(&tempty_bar[i], GEMM_EPI_WARPS);
        }
        fence_barrier_init();
        fence_proxy_async_smem();
    }
    if (warp == 1) tmem_alloc(tmem_ptr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    // tile = (sp * m_tiles + mt) * n_tiles + nt : CTAs running together share a pixel range (split) — its dY / X boxes
    // stay L2-resident.  (A stream-K division of the (tile, k) space balanced the SMs but was 10 % slower: neighbouring
    // CTAs then stream different pixel ranges and the operand re-reads miss L2.)
    const int num_tiles = p.splits * p.m_tiles * p.n_tiles;
    const int m_chunks = 3 * p.co_chunks;

    if (warp == 0) {
        // =========================================================== TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int nt = tile % p.n_tiles;
                const int mt = (tile / p.n_tiles) % p.m_tiles;
                const int sp = tile / (p.n_tiles * p.m_tiles);
                const int k_begin = sp * p.k_iters;
                const int k_end = min(p.k_total, k_begin + p.k_iters);
                const int mc0 = 2 * mt, mc1 = min(2 * mt + 1, m_chunks - 1);  // an odd tail repeats a chunk (masked)
                const int dy0 = mc0 / p.co_chunks, cc0 = mc0 % p.co_chunks;
                const int dy1 = mc1 / p.co_chunks, cc1 = mc1 % p.co_chunks;
                const bool src2 = nt >= p.cchunks1;
                const CUtensorMap* mb = src2 ? &tmB2 : &tmB;
                const int nc = (src2 ? nt - p.cchunks1 : nt) * 64;
                PixWalker px(p, k_begin);
                for (int ki = k_begin; ki < k_end; ++ki) {
                    const int n0 = px.n0, h0 = px.h0, w0 = px.w0;
                    px.advance(p);
                    mbar_wait(&empty_bar[stage], phase ^ 1, 1);
                    uint8_t* sa = smem + stage * stage_bytes;
                    mbar_expect_tx(&full_bar[stage], GEMM_A_STAGE + b_tx);
                    tma_load_4d(sa, &tmA, &full_bar[stage], cc0 * 64, w0, h0 + 1 - dy0, n0);
                    tma_load_4d(sa + 8192, &tmA, &full_bar[stage], cc1 * 64, w0, h0 + 1 - dy1, n0);
                    tma_load_4d(sa + GEMM_A_STAGE, mb, &full_bar[stage], nc, w0 - 1, h0, n0);
                    if (++stage == num_stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // =========================================================== UMMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc_bf16(GEMM_BLOCK_M, 192, 1, 1);
            // a 16-pixel k-step is two 8-pixel runs of the halo tile: adjacent (one image row, bw >= 16) or one halo
            // row apart (bw == 8: two image rows)
            const uint32_t b_sbo = p.bw >= 16 ? 1024u : static_cast<uint32_t>(halo_w) * 128u;
            // everything that does not depend on the stage is hoisted: this one thread's issue loop is the critical
            // path (two runtime integer divisions per k-step cost 25 % of the kernel when they sat inside it)
            const uint64_t da0 = make_smem_desc(0, 8192, 1024), db0 = make_smem_desc(0, 128, b_sbo);
            uint32_t a_off[GEMM_BLOCK_K / 16], b_off[GEMM_BLOCK_K / 16];
#pragma unroll
            for (int k = 0; k < GEMM_BLOCK_K / 16; ++k) {
                const int px = k * 16;  // halo row of this k-step's first pixel at dx = 0
                a_off[k] = (k * 2048) >> 4;
                b_off[k] = (GEMM_A_STAGE + ((px / p.bw) * halo_w + px % p.bw) * 128) >> 4;
            }
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int sp = tile / (p.n_tiles * p.m_tiles);
                const int k_begin = sp * p.k_iters;
                const int k_end = min(p.k_total, k_begin + p.k_iters);
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1, 2);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * 256;
                for (int ki = k_begin; ki < k_end; ++ki) {
                    mbar_wait(&full_bar[stage], phase, 3);
                    tc_fence_after();
                    const uint32_t sa16 = smem_u32(smem + stage * stage_bytes) >> 4;
#pragma unroll
                    for (int k = 0; k < GEMM_BLOCK_K / 16; ++k)
                        umma_bf16(tmem_d, da0 + (sa16 + a_off[k]), db0 + (sa16 + b_off[k]), idesc,
                                  (ki > k_begin || k > 0) ? 1u : 0u);
                    umma_commit(&empty_bar[stage]);
                    if (++stage == num_stages) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tfull_bar[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // =========================================================== epilogue: rows = (dy, co), three 64-column taps
        const int quad = warp & 3;
        const int half = (warp - 2) >> 2;
        const int m = quad * 32 + lane;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int nt = tile % p.n_tiles;
            const int mt = (tile / p.n_tiles) % p.m_tiles;
            const int mc = 2 * mt + (m >> 6);
            const int dy = mc / p.co_chunks, co = (mc % p.co_chunks) * 64 + (m & 63);
            const bool row_ok = mc < m_chunks && co < p.M;
            const long long c_base = static_cast<long long>(co) * p.ldc;
            mbar_wait(&tfull_bar[acc], acc_phase, 4);
            tc_fence_after();
            const uint32_t taddr = tmem_base + acc * 256 + (static_cast<uint32_t>(quad * 32) << 16);
            // 3 taps x 64 columns (with two warps per quadrant: 96 columns each, taps {0, 1 lower half} / {1 upper, 2})
#pragma unroll 1
            for (int i = 0; i < (EPI_HALVES == 2 ? 2 : 3); ++i) {
                const int dx = half + i;
                const int cb = (half == 1 && i == 0) ? 32 : 0, ce = (EPI_HALVES == 2 && half == 0 && i == 1) ? 32 : 64;
                epilogue_row(p, taddr + dx * 64, nt * 64, (dy * 3 + dx) * p.c_col_lo, c_base, 0, row_ok, nullptr, cb, ce);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

}  // namespace adm
