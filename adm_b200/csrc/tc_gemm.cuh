// tcgen05 / TMEM / TMA GEMM engine shared by conv3x3 (implicit GEMM fprop + dgrad), conv1x1, wgrad, Linear and the
// batched attention products.  Persistent warp-specialised kernels — tc_gemm_kernel<PLAIN|CONV|WGRAD> (general),
// tc_conv_halo_kernel (3x3 fprop/dgrad with halo re-use of the pixel operand), tc_wgrad_rows_kernel (3x3 wgrad, three
// taps per MMA), tc_conv_splitk_kernel (cluster split-K conv) — with the same roles:
//   warp 0      : TMA producer (one lane)        global -> 128B-swizzled smem ring
//   warp 1      : TMEM allocator + UMMA issuer   tcgen05.mma, fp32 accumulators in TMEM (2 x 256 columns)
//   warps 2..5  : epilogue                       tcgen05.ld -> +bias, +residual, *alpha -> bf16 / fp32 / fp32 atomics
//                 (warp w drains TMEM lane quadrant w % 4)
// Tile = 128 (M) x BN (N, runtime, multiple of 16, <= 256) x 64 (K per stage, bf16 = one 128 B swizzle row).
#pragma once
#include "ptx.cuh"
#include "adm_internal.h"

namespace adm {

constexpr int GEMM_BLOCK_M = 128;
constexpr int GEMM_BLOCK_K = 64;
// Epilogue warps: one per TMEM lane quadrant.  Eight (two per quadrant, each draining half of the tile's columns) were
// tried and removed: measured on B200 (tools/gemm_accounting.py) they changed nothing on the short-K 1x1 convs — they
// wait for operand bytes, not for the epilogue — and cost ~8 % on the small 8x8 / 4x4 tiles.
constexpr int GEMM_EPI_WARPS = 4;
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

// Coordinates of a tile of the persistent tile space: tile = ((plane * m_tiles + mt) * n_tiles + nt), plane = bt * splits
// + sp (see GemmParams).
struct TileCoord {
    int nt, mt, sp, bt;
    __device__ __forceinline__ TileCoord(const GemmParams& p, int tile) {
        nt = tile % p.n_tiles;
        int r = tile / p.n_tiles;
        mt = r % p.m_tiles;
        r /= p.m_tiles;
        sp = r % p.splits;
        bt = r / p.splits;
    }
    __device__ __forceinline__ int b_hi(const GemmParams& p) const { return bt / p.bdiv; }
    __device__ __forceinline__ int b_lo(const GemmParams& p) const { return bt % p.bdiv; }
    // The plane alone, in one division: the issuers need nothing but the split.
    static __device__ __forceinline__ int plane(const GemmParams& p, int tile) { return tile / (p.n_tiles * p.m_tiles); }
};

// Pixel shift (dh, dw) of conv tap `tap` (row-major over the kw x kw kernel, 'same' padding).
__device__ __forceinline__ void tap_shift(const GemmParams& p, int tap, int& dh, int& dw) {
    dh = 0;
    dw = 0;
    if (p.kw == 3) { dh = tap / 3 - 1; dw = tap % 3 - 1; }
    else if (p.kw > 1) { dh = tap / p.kw - (p.kw >> 1); dw = tap % p.kw - (p.kw >> 1); }
}

// Shared memory and TMEM every kernel of the engine starts from: the 1024-aligned operand ring (GEMM_SMEM_RING bytes),
// then the barriers, the TMEM address and the kernel's own barriers.
struct GemmPipeline {
    uint8_t* smem;
    int num_stages;        // stages of the stage ring
    uint64_t* full_bar;    // [GEMM_MAX_STAGES] stage landed (TMA transaction bytes)
    uint64_t* empty_bar;   // [GEMM_MAX_STAGES] stage consumed (UMMA commit)
    uint64_t* tfull_bar;   // [2] accumulator complete (UMMA commit)
    uint64_t* tempty_bar;  // [2] accumulator drained (one arrive per epilogue warp)
    uint64_t* own_bar;     // the kernel's own barriers
    uint32_t tmem_base;
};

// Sets a kernel up: thread 0 prefetches the three tensor maps and initialises as many stage_bytes stages as ring_bytes
// hold (at most GEMM_MAX_STAGES), `naccs` accumulator barrier pairs and, through init_own(own_bar), the kernel's own
// barriers; warp 1 allocates `tmem_cols` TMEM columns.
template <typename InitOwn>
__device__ __forceinline__ GemmPipeline pipeline_setup(uint8_t* smem_raw, const CUtensorMap* m0, const CUtensorMap* m1,
                                                       const CUtensorMap* m2, int ring_bytes, int stage_bytes, int naccs,
                                                       uint32_t tmem_cols, InitOwn init_own) {
    GemmPipeline pl;
    pl.smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    pl.num_stages = min(ring_bytes / stage_bytes, GEMM_MAX_STAGES);
    pl.full_bar = reinterpret_cast<uint64_t*>(pl.smem + GEMM_SMEM_RING);
    pl.empty_bar = pl.full_bar + GEMM_MAX_STAGES;
    pl.tfull_bar = pl.empty_bar + GEMM_MAX_STAGES;
    pl.tempty_bar = pl.tfull_bar + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(pl.tempty_bar + 2);
    pl.own_bar = pl.tempty_bar + 3;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(m0);
        tma_prefetch_desc(m1);
        tma_prefetch_desc(m2);
        for (int i = 0; i < pl.num_stages; ++i) {
            mbar_init(&pl.full_bar[i], 1);
            mbar_init(&pl.empty_bar[i], 1);
        }
        for (int i = 0; i < naccs; ++i) {
            mbar_init(&pl.tfull_bar[i], 1);
            mbar_init(&pl.tempty_bar[i], GEMM_EPI_WARPS);
        }
        init_own(pl.own_bar);
        fence_barrier_init();
        fence_proxy_async_smem();
    }
    if ((threadIdx.x >> 5) == 1) tmem_alloc(tmem_ptr, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pl.tmem_base = *tmem_ptr;
    return pl;
}

// All roles are done: warp 1 frees the TMEM columns pipeline_setup allocated.
__device__ __forceinline__ void pipeline_teardown(const GemmPipeline& pl, uint32_t tmem_cols) {
    tc_fence_before();
    __syncthreads();
    if ((threadIdx.x >> 5) == 1) {
        tc_fence_after();
        tmem_dealloc(pl.tmem_base, tmem_cols);
    }
}

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
// drained are [0, ncols) (a multiple of 16).
__device__ __forceinline__ void epilogue_row(const GemmParams& p, uint32_t taddr, int col_base, int col_shift,
                                             long long c_off, long long r_off, bool row_ok, const float* sbias,
                                             int ncols) {
    for (int c0 = 0; c0 < ncols; c0 += 64) {
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
__device__ __forceinline__ void epilogue_warps(const GemmParams& p, const GemmPipeline& pl, int warp, int lane,
                                               int num_tiles) {
    const int quad = warp & 3;
    const int m = quad * 32 + lane;  // row inside the tile
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const TileCoord tc(p, tile);
        const int b_hi = tc.b_hi(p), b_lo = tc.b_lo(p);

        long long row_off;  // element offset of this thread's output row (before column)
        bool row_ok;
        if (MODE == GEMM_CONV) {
            int n0, h0, w0;
            decode_pix(p, tc.mt, n0, h0, w0);
            const int wi = m % p.bw, hi = (m / p.bw) % p.bh, ni = m / (p.bw * p.bh);
            const long long pix = (static_cast<long long>(n0 + ni) * p.H + (h0 + hi)) * p.W + (w0 + wi);
            row_ok = pix < p.M;
            row_off = pix;
        } else {
            const int row = tc.mt * 128 + m;
            row_ok = row < p.M;
            row_off = (p.row_map != nullptr && row_ok) ? __ldg(p.row_map + row) : row;
        }
        const long long c_base = b_hi * p.c_bhi + b_lo * p.c_blo + row_off * p.ldc;
        const int col_base = tc.nt * p.bn;        // column inside [0, N)
        const int col_shift = b_lo * p.c_col_lo;  // extra offset in the output row

        float* sbias = reinterpret_cast<float*>(pl.smem + GEMM_SMEM_RING + 1024) + acc * 256;
        stage_bias(p, sbias, col_base, (warp - 2) * 32 + lane);
        mbar_wait(&pl.tfull_bar[acc], acc_phase, 4);
        tc_fence_after();
        const uint32_t taddr = pl.tmem_base + acc * 256 + (static_cast<uint32_t>(quad * 32) << 16);
        epilogue_row(p, taddr, col_base, col_shift, c_base, row_off * p.ldr, row_ok, sbias, p.bn);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&pl.tempty_bar[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
}

// One stage of the implicit-GEMM conv, k-iteration ki = tap * cchunks + kc: the pixel box at tap `tap`'s shift, channel
// chunk kc (past cchunks1 from A source 2: the fused channel concat), and the weight tile.
__device__ __forceinline__ void load_conv_stage(const GemmParams& p, const CUtensorMap* tmA, const CUtensorMap* tmA2,
                                                const CUtensorMap* tmB, uint8_t* sa, uint64_t* bar, int ki, int tap,
                                                int kc, int nt, int n0, int h0, int w0) {
    uint8_t* sb = sa + GEMM_A_STAGE;
    int dh, dw;
    tap_shift(p, tap, dh, dw);
    if (kc < p.cchunks1)
        tma_load_4d(sa, tmA, bar, kc * 64, w0 + dw, h0 + dh, n0);
    else
        tma_load_4d(sa, tmA2, bar, (kc - p.cchunks1) * 64, w0 + dw, h0 + dh, n0);
    if (!p.b_mn) {
        // weights [Nout][ntaps * Kpad], K-major
        tma_load_2d(sb, tmB, bar, ki * 64, nt * p.bn);
    } else {
        // dgrad on the fprop-packed weights viewed as (N_gemm = Cin, taps, K_gemm = Cout): the spatial flip is the tap
        // reversal, the transpose is the MN-major operand mode.
        for (int c = 0; c * 64 < p.bn; ++c)
            tma_load_3d(sb + c * 8192, tmB, bar, nt * p.bn + c * 64, p.ntaps - 1 - tap, kc * 64);
    }
}

// UMMA descriptors of a 128 x bn x 64 ring stage (A at the stage start, B GEMM_A_STAGE bytes behind it).  Built once, out
// of the issue loop: this thread's instruction stream is the critical path of the main loop.
struct StageDescs {
    uint32_t idesc;
    uint32_t a_kstep, b_kstep;  // 16-deep k-step strides, in 16 B units
    uint64_t da0, db0;
    __device__ __forceinline__ StageDescs(int bn, int a_mn, int b_mn)
        : idesc(make_idesc_bf16(GEMM_BLOCK_M, bn, a_mn, b_mn)),
          a_kstep((a_mn ? 2048u : 32u) >> 4),
          b_kstep((b_mn ? 2048u : 32u) >> 4),
          da0(make_smem_desc(0, a_mn ? 8192u : 16u, 1024)),
          db0(make_smem_desc(0, b_mn ? 8192u : 16u, 1024)) {}
};

// Issues k-iterations [k_begin, k_end) of one tile into the accumulator at tmem_d: per ring stage, wait for it to land,
// four UMMA k-steps, release it.  `code` names the full-barrier wait site.
__device__ __forceinline__ void issue_k_range(const GemmPipeline& pl, const StageDescs& d, int stage_bytes, int& stage,
                                              uint32_t& phase, uint32_t tmem_d, int k_begin, int k_end, int code) {
    for (int ki = k_begin; ki < k_end; ++ki) {
        mbar_wait(&pl.full_bar[stage], phase, code);
        tc_fence_after();
        // In a non-leader CTA of a cluster the shared-window address carries bits above the 14-bit descriptor field:
        // unmasked they spill into the leading-byte-offset field (which only MN-major multi-chunk B reads).
        const uint32_t sa16 = (smem_u32(pl.smem + stage * stage_bytes) & 0x3FFFFu) >> 4;
        const uint64_t da = d.da0 + sa16, db = d.db0 + (sa16 + (GEMM_A_STAGE >> 4));
#pragma unroll
        for (int k = 0; k < GEMM_BLOCK_K / 16; ++k)
            umma_bf16(tmem_d, da + k * d.a_kstep, db + k * d.b_kstep, d.idesc, (ki > k_begin || k > 0) ? 1u : 0u);
        umma_commit(&pl.empty_bar[stage]);
        if (++stage == pl.num_stages) { stage = 0; phase ^= 1; }
    }
}

template <int MODE>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2,
               const __grid_constant__ CUtensorMap tmB, const __grid_constant__ GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    const int stage_bytes = GEMM_A_STAGE + p.bn * 128;
    const GemmPipeline pl = pipeline_setup(smem_raw, &tmA, &tmA2, &tmB, GEMM_SMEM_RING, stage_bytes, 2, 512,
                                           [](uint64_t*) {});
    uint8_t* smem = pl.smem;
    uint64_t* full_bar = pl.full_bar;
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_tiles = p.batches * p.splits * p.m_tiles * p.n_tiles;

    if (warp == 0) {
        // =========================================================== TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const TileCoord tc(p, tile);
                const int nt = tc.nt, mt = tc.mt, bt = tc.bt;
                const int k_begin = tc.sp * p.k_iters;
                const int k_end = min(p.k_total, k_begin + p.k_iters);
                int n0 = 0, h0 = 0, w0 = 0;
                if (MODE == GEMM_CONV) decode_pix(p, mt, n0, h0, w0);
                const int b_hi = tc.b_hi(p), b_lo = tc.b_lo(p);
                int tap = 0, kc = 0;  // conv: ki = tap * cchunks + kc, walked without divisions
                if (MODE == GEMM_CONV) { tap = k_begin / p.cchunks; kc = k_begin % p.cchunks; }
                PixWalker px(p, MODE == GEMM_WGRAD ? k_begin : 0);
                for (int ki = k_begin; ki < k_end; ++ki) {
                    mbar_wait(&pl.empty_bar[stage], phase ^ 1, 1);
                    uint8_t* sa = smem + stage * stage_bytes;
                    uint8_t* sb = sa + GEMM_A_STAGE;
                    mbar_expect_tx(&full_bar[stage], stage_bytes);
                    if (MODE == GEMM_CONV) {
                        load_conv_stage(p, &tmA, &tmA2, &tmB, sa, &full_bar[stage], ki, tap, kc, nt, n0, h0, w0);
                        if (++kc == p.cchunks) { kc = 0; ++tap; }
                    } else if (MODE == GEMM_WGRAD) {
                        // K runs over pixel blocks of 64; bt = tap.  A = dY (MN-major), B = shifted X (MN-major).
                        n0 = px.n0; h0 = px.h0; w0 = px.w0;
                        px.advance(p);
                        int dh, dw;
                        tap_shift(p, bt, dh, dw);
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
                    if (++stage == pl.num_stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // =========================================================== UMMA issuer
        if (lane == 0) {
            const StageDescs d(p.bn, p.a_mn, p.b_mn);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int k_begin = TileCoord::plane(p, tile) % p.splits * p.k_iters;
                const int k_end = min(p.k_total, k_begin + p.k_iters);
                mbar_wait(&pl.tempty_bar[acc], acc_phase ^ 1, 2);
                tc_fence_after();
                issue_k_range(pl, d, stage_bytes, stage, phase, pl.tmem_base + acc * 256, k_begin, k_end, 3);
                umma_commit(&pl.tfull_bar[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // =========================================================== epilogue (4 warps, one TMEM lane quadrant each)
        epilogue_warps<MODE>(p, pl, warp, lane, num_tiles);
    }
    pipeline_teardown(pl, 512);
}

// ------------------------------------------------------------------------------------------------ cluster split-K conv
// Implicit-GEMM conv (fprop / dgrad, 3x3 or 1x1) for problems with too few 128 x bn output tiles to fill the GPU (the 4x4
// level: 2048 pixels x 384 channels = 48 tiles of 128 x 128, each with a K loop of 54-108 iterations).  A thread-block
// cluster of ksplit CTAs shares ONE output tile: CTA r multiplies K iterations [r * k_iters, (r + 1) * k_iters) into its own
// TMEM accumulator; the non-leaders then park their fp32 partial tiles in their (now idle) operand ring, signal the leader's
// mbarrier across the cluster, and the leader adds them through distributed shared memory (ld.shared::cluster) into its
// accumulator before the ordinary epilogue.  One tile per CTA (grid = tiles x ksplit); roles as in tc_gemm_kernel.
__global__ void __launch_bounds__(GEMM_THREADS, 1)
tc_conv_splitk_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2,
                      const __grid_constant__ CUtensorMap tmB, const __grid_constant__ GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    const int stage_bytes = GEMM_A_STAGE + p.bn * 128;
    // one accumulator; the leader's own barrier counts the non-leaders' parked partial tiles
    const GemmPipeline pl = pipeline_setup(smem_raw, &tmA, &tmA2, &tmB, GEMM_SMEM_RING, stage_bytes, 1, 256,
                                           [&](uint64_t* own) { mbar_init(own, (p.ksplit - 1) * GEMM_EPI_WARPS); });
    cluster_sync_all();  // the leader's peers_bar is initialised before any remote arrive
    uint8_t* smem = pl.smem;
    uint64_t* full_bar = pl.full_bar;
    uint64_t* peers_bar = pl.own_bar;
    const uint32_t tmem_base = pl.tmem_base;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int rank = static_cast<int>(cluster_ctarank());
    const int tile = blockIdx.x / p.ksplit;
    const int nt = tile % p.n_tiles, mt = tile / p.n_tiles;
    const int k_begin = rank * p.k_iters;
    const int k_end = min(p.k_total, k_begin + p.k_iters);

    int n0, h0, w0;
    decode_pix(p, mt, n0, h0, w0);
    if (warp == 0) {
        // =========================================================== TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int tap = k_begin / p.cchunks, kc = k_begin % p.cchunks;
            for (int ki = k_begin; ki < k_end; ++ki) {
                mbar_wait(&pl.empty_bar[stage], phase ^ 1, 41);
                uint8_t* sa = smem + stage * stage_bytes;
                mbar_expect_tx(&full_bar[stage], stage_bytes);
                load_conv_stage(p, &tmA, &tmA2, &tmB, sa, &full_bar[stage], ki, tap, kc, nt, n0, h0, w0);
                if (++kc == p.cchunks) { kc = 0; ++tap; }
                if (++stage == pl.num_stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // =========================================================== UMMA issuer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            issue_k_range(pl, StageDescs(p.bn, 0, p.b_mn), stage_bytes, stage, phase, tmem_base, k_begin, k_end, 43);
            umma_commit(pl.tfull_bar);
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
        mbar_wait(pl.tfull_bar, 0, 44);  // this CTA's K range is in its accumulator; its operand ring is idle from here on
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
            epilogue_row(p, taddr, col_base, 0, pix * p.ldc, pix * p.ldr, row_ok, sbias, p.bn);
        }
    }
    pipeline_teardown(pl, 256);
    cluster_sync_all();  // no CTA exits while the leader may still read its parked partial tile
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
    const int b_bytes = p.bn * 128;
    // the stage ring is the weight ring, behind the halo buffers; the kernel's own barriers are the halo ring's
    const auto init_halo_ring = [](uint64_t* own) {
        for (int i = 0; i < 2 * HALO_BUFS; ++i) mbar_init(&own[i], 1);
    };
    const GemmPipeline pl = pipeline_setup(smem_raw, &tmA, &tmA2, &tmB, GEMM_SMEM_RING - HALO_BUFS * HALO_BYTES, b_bytes,
                                           2, 512, init_halo_ring);
    uint8_t* smem = pl.smem;
    uint8_t* b_ring = smem + HALO_BUFS * HALO_BYTES;
    const int nb = pl.num_stages;
    uint64_t* bfull = pl.full_bar;
    uint64_t* bempty = pl.empty_bar;
    uint64_t* hfull = pl.own_bar;  // halo buffer landed
    uint64_t* hempty = hfull + HALO_BUFS;
    const uint32_t tmem_base = pl.tmem_base;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
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
            // Halo loads run one chunk step AHEAD of the weight tiles (a cursor over (tile, chunk) that only this thread
            // advances): one step hides the TMA latency under the nine MMAs of the current chunk; three buffers:
            // loading, multiplying, draining.  (Two steps make this thread wait for the buffer still being multiplied
            // before it issues weights.)
            int cur_tile = blockIdx.x, cur_kc = 0;
            auto next_halo = [&]() {
                if (cur_tile >= num_tiles) return;
                load_halo(cur_tile, cur_kc);
                if (++cur_kc == p.cchunks) { cur_kc = 0; cur_tile += gridDim.x; }
            };
            next_halo();
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int nt = tile % p.n_tiles;
                for (int kc = 0; kc < p.cchunks; ++kc) {
                    next_halo();  // the next step's halo goes out before this step's nine weight tiles
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
                mbar_wait(&pl.tempty_bar[acc], acc_phase ^ 1, 2);
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
                umma_commit(&pl.tfull_bar[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        epilogue_warps<GEMM_CONV>(p, pl, warp, lane, num_tiles);
    }

    pipeline_teardown(pl, 512);
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
__global__ void __launch_bounds__(GEMM_THREADS, 1)
tc_wgrad_rows_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                     const __grid_constant__ CUtensorMap tmB2, const __grid_constant__ GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    const int halo_w = p.bw + 2;
    const int b_tx = p.bh * halo_w * 128;
    const int stage_bytes = GEMM_A_STAGE + ((b_tx + 1023) & ~1023);
    const GemmPipeline pl = pipeline_setup(smem_raw, &tmA, &tmB, &tmB2, GEMM_SMEM_RING, stage_bytes, 2, 512,
                                           [](uint64_t*) {});
    uint8_t* smem = pl.smem;
    uint64_t* full_bar = pl.full_bar;
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

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
                const TileCoord tc(p, tile);
                const int k_begin = tc.sp * p.k_iters;
                const int k_end = min(p.k_total, k_begin + p.k_iters);
                const int mc0 = 2 * tc.mt, mc1 = min(2 * tc.mt + 1, m_chunks - 1);  // an odd tail repeats a chunk (masked)
                const int dy0 = mc0 / p.co_chunks, cc0 = mc0 % p.co_chunks;
                const int dy1 = mc1 / p.co_chunks, cc1 = mc1 % p.co_chunks;
                const bool src2 = tc.nt >= p.cchunks1;
                const CUtensorMap* mb = src2 ? &tmB2 : &tmB;
                const int nc = (src2 ? tc.nt - p.cchunks1 : tc.nt) * 64;
                PixWalker px(p, k_begin);
                for (int ki = k_begin; ki < k_end; ++ki) {
                    const int n0 = px.n0, h0 = px.h0, w0 = px.w0;
                    px.advance(p);
                    mbar_wait(&pl.empty_bar[stage], phase ^ 1, 1);
                    uint8_t* sa = smem + stage * stage_bytes;
                    mbar_expect_tx(&full_bar[stage], GEMM_A_STAGE + b_tx);
                    tma_load_4d(sa, &tmA, &full_bar[stage], cc0 * 64, w0, h0 + 1 - dy0, n0);
                    tma_load_4d(sa + 8192, &tmA, &full_bar[stage], cc1 * 64, w0, h0 + 1 - dy1, n0);
                    tma_load_4d(sa + GEMM_A_STAGE, mb, &full_bar[stage], nc, w0 - 1, h0, n0);
                    if (++stage == pl.num_stages) { stage = 0; phase ^= 1; }
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
                const int k_begin = TileCoord::plane(p, tile) * p.k_iters;  // no batches: the plane is the split
                const int k_end = min(p.k_total, k_begin + p.k_iters);
                mbar_wait(&pl.tempty_bar[acc], acc_phase ^ 1, 2);
                tc_fence_after();
                const uint32_t tmem_d = pl.tmem_base + acc * 256;
                for (int ki = k_begin; ki < k_end; ++ki) {
                    mbar_wait(&full_bar[stage], phase, 3);
                    tc_fence_after();
                    const uint32_t sa16 = smem_u32(smem + stage * stage_bytes) >> 4;
#pragma unroll
                    for (int k = 0; k < GEMM_BLOCK_K / 16; ++k)
                        umma_bf16(tmem_d, da0 + (sa16 + a_off[k]), db0 + (sa16 + b_off[k]), idesc,
                                  (ki > k_begin || k > 0) ? 1u : 0u);
                    umma_commit(&pl.empty_bar[stage]);
                    if (++stage == pl.num_stages) { stage = 0; phase ^= 1; }
                }
                umma_commit(&pl.tfull_bar[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // =========================================================== epilogue: rows = (dy, co), three 64-column taps
        const int quad = warp & 3;
        const int m = quad * 32 + lane;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const TileCoord tc(p, tile);
            const int mc = 2 * tc.mt + (m >> 6);
            const int dy = mc / p.co_chunks, co = (mc % p.co_chunks) * 64 + (m & 63);
            const bool row_ok = mc < m_chunks && co < p.M;
            const long long c_base = static_cast<long long>(co) * p.ldc;
            mbar_wait(&pl.tfull_bar[acc], acc_phase, 4);
            tc_fence_after();
            const uint32_t taddr = pl.tmem_base + acc * 256 + (static_cast<uint32_t>(quad * 32) << 16);
#pragma unroll 1
            for (int dx = 0; dx < 3; ++dx)
                epilogue_row(p, taddr + dx * 64, tc.nt * 64, (dy * 3 + dx) * p.c_col_lo, c_base, 0, row_ok, nullptr, 64);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&pl.tempty_bar[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    pipeline_teardown(pl, 512);
}

}  // namespace adm
