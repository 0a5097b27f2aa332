// Host side of the tcgen05 GEMM engine: tensor-map construction, tile-shape selection, launches, and the C-ABI entry
// points declared in include/adm_b200.h.  No torch types; raw device pointers + sizes + a cudaStream_t.
#include "tc_gemm.cuh"
#include "adm_internal.h"
#include <cudaTypedefs.h>
#include <limits.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace adm {

static PFN_cuTensorMapEncodeTiled g_encode = nullptr;
static int g_num_sms = 0;
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char* get_error() { return g_err; }

int num_sms() {
    if (g_num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (g_num_sms <= 0) g_num_sms = 148;
    }
    return g_num_sms;
}

static int init_driver() {
    if (g_encode) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || fn == nullptr) {
        set_error("cuTensorMapEncodeTiled unavailable: %s", cudaGetErrorString(e));
        return ADM_ERR_CUDA;
    }
    g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(fn);
    return 0;
}

int encode_map(CUtensorMap* m, const void* ptr, int rank, const long long* dims, const long long* strides,
               const int* box) {
    if (int e = init_driver()) return e;
    cuuint64_t gd[5];
    cuuint64_t gs[4];
    cuuint32_t bx[5];
    cuuint32_t es[5];
    for (int i = 0; i < rank; ++i) {
        gd[i] = static_cast<cuuint64_t>(dims[i]);
        bx[i] = static_cast<cuuint32_t>(box[i]);
        es[i] = 1;
        if (i > 0) gs[i - 1] = static_cast<cuuint64_t>(strides[i - 1]) * 2;
        if (dims[i] <= 0 || box[i] <= 0 || box[i] > 256) {
            set_error("tensor map: bad dim/box at %d (dim %lld box %d)", i, dims[i], box[i]);
            return ADM_ERR_SHAPE;
        }
    }
    for (int i = 0; i + 1 < rank; ++i)
        if (gs[i] % 16 != 0) {
            set_error("tensor map: stride %d = %llu B not a multiple of 16", i, (unsigned long long)gs[i]);
            return ADM_ERR_SHAPE;
        }
    if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0) {
        set_error("tensor map: base pointer not 16 B aligned");
        return ADM_ERR_SHAPE;
    }
    CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(ptr), gd, gs, bx, es,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d", static_cast<int>(r));
        return ADM_ERR_CUDA;
    }
    return 0;
}

// Launches a GEMM-engine kernel over the tiles of p: GEMM_THREADS threads and GEMM_SMEM_TOTAL bytes of shared memory
// per CTA.  Without a cluster the kernel is persistent: min(tiles, SMs) CTAs stride over the tiles.  With one (the
// split-K conv) every tile gets its own cluster of `cluster` CTAs.
template <auto Kern>
static int launch_gemm(const char* name, int cluster, const CUtensorMap& a, const CUtensorMap& a2, const CUtensorMap& b,
                       const GemmParams& p, cudaStream_t stream) {
    const long long tiles = 1LL * p.batches * p.splits * p.m_tiles * p.n_tiles;
    if (tiles <= 0 || tiles > INT_MAX) {
        set_error("%s: bad tile count %lld", name, tiles);
        return ADM_ERR_SHAPE;
    }
    const long long grid = cluster > 0 ? tiles * cluster : (tiles < num_sms() ? tiles : num_sms());
    cudaError_t e = set_smem_limit_once<Kern>(GEMM_SMEM_TOTAL);
    if (e == cudaSuccess)
        e = launch_k(Kern, dim3(static_cast<unsigned>(grid)), dim3(GEMM_THREADS), GEMM_SMEM_TOTAL, stream, cluster, a, a2, b, p);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s launch: %s", name, cudaGetErrorString(e));
        return ADM_ERR_CUDA;
    }
    count_launch();
    return 0;
}

// Under-filled convs (few pixel tiles, long K): pick (N tile, K split) minimising the critical path
// ceil(k_total / ks) x (128 + bn) operand rows + reduction, subject to tiles x ks <= SMs.  Returns ks (1 = plain kernel).
static int pick_splitk(int n, int multiple, int m_tiles, int k_total, int* bn_out) {
    const int n_pad = (n + multiple - 1) / multiple * multiple;
    // Test hook, read per call: ADM_SPLITK_FORCE="bn,ks" forces a tile width and split when they fit the problem, so the
    // tests can cover (bn, ks) pairs of the split-K kernel that the cost model below does not pick.
    if (const char* f = getenv("ADM_SPLITK_FORCE")) {
        int fb = 0, fk = 0;
        if (sscanf(f, "%d,%d", &fb, &fk) == 2 && fb >= multiple && fb % multiple == 0 && n_pad % fb == 0 && fk >= 1 && fk <= 8 &&
            m_tiles * (n_pad / fb) * fk <= num_sms() && (fk - 1) * ((k_total + fk - 1) / fk) < k_total) {
            if (fk > 1) *bn_out = fb;
            return fk;
        }
    }
    const int sms = num_sms();
    long long best = -1;
    int best_bn = 0, best_ks = 1;
    for (int bn = 256 / multiple * multiple; bn >= multiple; bn -= multiple) {
        if (n_pad % bn) continue;
        const int tiles = m_tiles * (n_pad / bn);
        for (int ks = 1; ks <= 4; ++ks) {
            if (tiles * ks > sms || ks * 6 > k_total) continue;
            const int k_per = (k_total + ks - 1) / ks;
            if ((ks - 1) * k_per >= k_total) continue;  // an empty last split
            const long long cost = 1LL * k_per * 8 * (128 + bn) / 3 + 8LL * bn + 500 + (ks > 1 ? 1500 + 12LL * bn * (ks - 1) : 0);
            if (best < 0 || cost < best) { best = cost; best_bn = bn; best_ks = ks; }
        }
    }
    if (best_ks > 1) *bn_out = best_bn;
    return best_ks;
}

// split K (pixels) for the wgrad kernels: the split that minimises waves x (k-iterations per tile + epilogue cost) on
// the persistent grid — fewer, fuller waves beat "more tiles" (wave quantisation), fewer splits mean fewer atomics.
static void pick_wgrad_split(GemmParams* p, int base_tiles, int epi) {
    const int sms = num_sms();
    long long best_cost = -1;
    int best_s = 1;
    for (int s = 1; s <= p->k_total && s <= 64; ++s) {
        const int k_per = (p->k_total + s - 1) / s;
        const int s_eff = (p->k_total + k_per - 1) / k_per;
        const long long waves = (1LL * base_tiles * s_eff + sms - 1) / sms;
        const long long cost = waves * (k_per + epi);
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_s = s_eff; }
    }
    p->k_iters = (p->k_total + best_s - 1) / best_s;
    p->splits = (p->k_total + p->k_iters - 1) / p->k_iters;
}

// The halo kernel serves 3x3 convs whose images tile into 8 x 16 pixel boxes (the 32x32 and 16x16 levels).
static bool halo_ok(int ntaps, int h, int w) { return ntaps == 9 && w % 8 == 0 && h % 16 == 0; }

// Largest multiple of 16 that is <= cap and divides ceil16(n); falls back to the smallest cover.
static int pick_bn(int n, int cap, int multiple) {
    const int n16 = (n + multiple - 1) / multiple * multiple;
    for (int bn = cap / multiple * multiple; bn >= multiple; bn -= multiple)
        if (n16 % bn == 0) return bn;
    return multiple;
}

// N tile for the conv kernels from a small cost model (clocks): waves x (k_iters x mma + epilogue), with the MMA time of
// a 128 x bn x 64 step proportional to the operand rows it reads from shared memory (128 + bn; measured ~0.43 us for
// bn = 192, tools/bench_floor.py) and ~500 clocks of epilogue per 64 columns.  It only departs from "largest divisor"
// when there are too few pixel tiles to fill the SMs (4x4 / 8x8 levels), where narrower tiles cut the critical path.
static int pick_bn_cost(int n, int multiple, int m_tiles, int k_total) {
    const int n_pad = (n + multiple - 1) / multiple * multiple;
    const int sms = num_sms();
    long long best = -1;
    int best_bn = multiple;
    for (int bn = 256 / multiple * multiple; bn >= multiple; bn -= multiple) {
        if (n_pad % bn) continue;
        const long long tiles = 1LL * m_tiles * (n_pad / bn);
        const long long waves = (tiles + sms - 1) / sms;
        const long long cost = waves * (1LL * k_total * 8 * (128 + bn) / 3 + 8LL * bn + 500);
        if (best < 0 || cost < best) { best = cost; best_bn = bn; }
    }
    return best_bn;
}

// Pixel box (bw, bh, bni) covering `pixels` output pixels of an H x W image batch.
static int pick_box(int n, int h, int w, int pixels, int* bw, int* bh, int* bni) {
    if (w >= pixels) {
        if (w % pixels != 0) return -1;
        *bw = pixels; *bh = 1; *bni = 1;
        return 0;
    }
    if (pixels % w != 0) return -1;
    *bw = w;
    const int rows = pixels / w;
    if (h >= rows) {
        if (h % rows != 0) return -1;
        *bh = rows; *bni = 1;
        return 0;
    }
    if (rows % h != 0) return -1;
    *bh = h;
    *bni = rows / h;
    (void)n;
    return 0;
}

static inline int pad64(int c) { return (c + 63) / 64 * 64; }

// taps per kernel row of a square odd kernel ('same' padding): 1 -> 1, 9 -> 3, 25 -> 5, 49 -> 7; 0 = unsupported
static inline int taps_per_row(int ntaps) { return ntaps == 1 ? 1 : ntaps == 9 ? 3 : ntaps == 25 ? 5 : ntaps == 49 ? 7 : 0; }

static void init_params(GemmParams* p) {
    memset(p, 0, sizeof(*p));
    p->batches = 1; p->splits = 1; p->bdiv = 1; p->ntaps = 1; p->kw = 1; p->alpha = 1.f;
    p->tiles_w = 1; p->tiles_h = 1; p->bni = 1; p->bw = 1; p->bh = 1;
    p->n_split = INT_MAX;
}

static int nhwc_map(CUtensorMap* m, const void* ptr, int c, long long ld, int n, int h, int w, int bw, int bh,
                    int bni) {
    const long long dims[4] = {c, w, h, n};
    const long long strides[3] = {ld, ld * w, ld * w * h};
    const int box[4] = {64, bw, bh, bni};
    return encode_map(m, ptr, 4, dims, strides, box);
}

}  // namespace adm

using namespace adm;

extern "C" {

int adm_conv_fprop(const void* x1, int c1, long long ld1, const void* x2, int c2, long long ld2, int n, int h, int w,
                   const void* wpk, int nout, int ntaps, void* out, int out_mode, long long ldc, const float* bias,
                   const void* residual, long long ldr, float alpha, void* stream) {
    if (taps_per_row(ntaps) == 0) { set_error("conv_fprop: ntaps must be 1, 9, 25 or 49"); return ADM_ERR_SHAPE; }
    if (c1 <= 0 || c1 % 8 || (x2 && (c2 <= 0 || c2 % 8))) { set_error("conv_fprop: channels must be multiples of 8"); return ADM_ERR_SHAPE; }
    GemmParams p;
    init_params(&p);
    const bool halo = halo_ok(ntaps, h, w);
    if (halo) { p.bw = 8; p.bh = 16; p.bni = 1; }
    else if (pick_box(n, h, w, 128, &p.bw, &p.bh, &p.bni)) { set_error("conv_fprop: unsupported H x W = %d x %d", h, w); return ADM_ERR_SHAPE; }
    p.H = h; p.W = w;
    p.tiles_w = w / p.bw; p.tiles_h = h / p.bh;
    p.m_tiles = p.tiles_w * p.tiles_h * ((n + p.bni - 1) / p.bni);
    p.ntaps = ntaps; p.kw = taps_per_row(ntaps);
    p.cchunks1 = pad64(c1) / 64;
    p.cchunks = p.cchunks1 + (x2 ? pad64(c2) / 64 : 0);
    p.k_total = p.k_iters = ntaps * p.cchunks;
    p.bn = pick_bn_cost(nout, 16, p.m_tiles, p.k_total);
    p.ksplit = 1;
    if (!halo && out_mode != OUT_F32_ATOMIC) {
        int bn_s = p.bn;
        const int ks = pick_splitk(nout, 16, p.m_tiles, p.k_total, &bn_s);
        if (ks > 1) { p.ksplit = ks; p.bn = bn_s; p.k_iters = (p.k_total + ks - 1) / ks; }
    }
    p.n_tiles = (nout + p.bn - 1) / p.bn;
    p.M = n * h * w; p.N = nout;
    p.C = out; p.ldc = ldc; p.bias = bias; p.residual = static_cast<const __nv_bfloat16*>(residual); p.ldr = ldr;
    p.alpha = alpha; p.out_mode = out_mode;
    CUtensorMap ma, ma2, mb;
    const int abw = halo ? HALO_W : p.bw, abh = halo ? HALO_H : p.bh;  // A box: the tile, or the tile + its 3x3 halo
    if (int e = nhwc_map(&ma, x1, c1, ld1, n, h, w, abw, abh, p.bni)) return e;
    if (x2) { if (int e = nhwc_map(&ma2, x2, c2, ld2, n, h, w, abw, abh, p.bni)) return e; } else ma2 = ma;
    const long long kpad = 1LL * ntaps * p.cchunks * 64;
    const long long bd[2] = {kpad, nout};
    const long long bs[1] = {kpad};
    const int bb[2] = {64, p.bn};
    if (int e = encode_map(&mb, wpk, 2, bd, bs, bb)) return e;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (halo) return launch_gemm<tc_conv_halo_kernel>("tc_conv_halo", 0, ma, ma2, mb, p, s);
    if (p.ksplit > 1) return launch_gemm<tc_conv_splitk_kernel>("tc_conv_splitk", p.ksplit, ma, ma2, mb, p, s);
    return launch_gemm<tc_gemm_kernel<GEMM_CONV>>("tc_gemm", 0, ma, ma2, mb, p, s);
}

int adm_conv_dgrad(const void* dy, int cout, long long ld_dy, int n, int h, int w, const void* wpk, int kpad,
                   int ntaps, void* dx, int n_valid, long long ldc, const void* residual, long long ldr, float alpha,
                   void* stream) {
    if (taps_per_row(ntaps) == 0) { set_error("conv_dgrad: ntaps must be 1, 9, 25 or 49"); return ADM_ERR_SHAPE; }
    if (kpad % 64) { set_error("conv_dgrad: kpad must be a multiple of 64"); return ADM_ERR_SHAPE; }
    GemmParams p;
    init_params(&p);
    const bool halo = halo_ok(ntaps, h, w);
    if (halo) { p.bw = 8; p.bh = 16; p.bni = 1; }
    else if (pick_box(n, h, w, 128, &p.bw, &p.bh, &p.bni)) { set_error("conv_dgrad: unsupported H x W = %d x %d", h, w); return ADM_ERR_SHAPE; }
    p.H = h; p.W = w;
    p.tiles_w = w / p.bw; p.tiles_h = h / p.bh;
    p.m_tiles = p.tiles_w * p.tiles_h * ((n + p.bni - 1) / p.bni);
    p.ntaps = ntaps; p.kw = taps_per_row(ntaps);
    p.cchunks1 = p.cchunks = pad64(cout) / 64;
    p.k_total = p.k_iters = ntaps * p.cchunks;
    p.bn = pick_bn_cost(kpad, 64, p.m_tiles, p.k_total);
    p.ksplit = 1;
    if (!halo) {
        int bn_s = p.bn;
        const int ks = pick_splitk(kpad, 64, p.m_tiles, p.k_total, &bn_s);
        if (ks > 1) { p.ksplit = ks; p.bn = bn_s; p.k_iters = (p.k_total + ks - 1) / ks; }
    }
    p.n_tiles = kpad / p.bn;
    p.b_mn = 1;
    p.M = n * h * w; p.N = n_valid;
    p.C = dx; p.ldc = ldc; p.residual = static_cast<const __nv_bfloat16*>(residual); p.ldr = ldr;
    p.alpha = alpha; p.out_mode = OUT_BF16;
    CUtensorMap ma, mb;
    if (int e = nhwc_map(&ma, dy, cout, ld_dy, n, h, w, halo ? HALO_W : p.bw, halo ? HALO_H : p.bh, p.bni)) return e;
    const long long bd[3] = {kpad, ntaps, cout};
    const long long bs[2] = {kpad, 1LL * kpad * ntaps};
    const int bb[3] = {64, 1, 64};
    if (int e = encode_map(&mb, wpk, 3, bd, bs, bb)) return e;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (halo) return launch_gemm<tc_conv_halo_kernel>("tc_conv_halo", 0, ma, ma, mb, p, s);
    if (p.ksplit > 1) return launch_gemm<tc_conv_splitk_kernel>("tc_conv_splitk", p.ksplit, ma, ma, mb, p, s);
    return launch_gemm<tc_gemm_kernel<GEMM_CONV>>("tc_gemm", 0, ma, ma, mb, p, s);
}

int adm_conv_wgrad(const void* dy, int cout, long long ld_dy, const void* x1, int c1, long long ld1, const void* x2,
                   int c2, long long ld2, int n, int h, int w, int ntaps, float* dw, void* stream) {
    return adm_conv_wgrad_mapped(dy, cout, ld_dy, x1, c1, ld1, x2, c2, ld2, n, h, w, ntaps, nullptr, dw, stream);
}

int adm_conv_wgrad_mapped(const void* dy, int cout, long long ld_dy, const void* x1, int c1, long long ld1,
                          const void* x2, int c2, long long ld2, int n, int h, int w, int ntaps, const int* row_map,
                          float* dw, void* stream) {
    if (row_map != nullptr && ntaps != 1) { set_error("conv_wgrad: a row map is supported for 1x1 convs only"); return ADM_ERR_SHAPE; }
    if (taps_per_row(ntaps) == 0) { set_error("conv_wgrad: ntaps must be 1, 9, 25 or 49"); return ADM_ERR_SHAPE; }
    GemmParams p;
    init_params(&p);
    const long long pixels = 1LL * n * h * w;
    // K box of 64 pixels; tiny tensors (e.g. Linear with batch < 64) use a short box and rely on zero OOB fill.
    if (pick_box(n, h, w, 64, &p.bw, &p.bh, &p.bni)) { set_error("conv_wgrad: unsupported H x W = %d x %d", h, w); return ADM_ERR_SHAPE; }
    p.H = h; p.W = w;
    p.tiles_w = w / p.bw; p.tiles_h = h / p.bh;
    p.k_total = p.tiles_w * p.tiles_h * ((n + p.bni - 1) / p.bni);
    const int kpad = pad64(c1) + (x2 ? pad64(c2) : 0);
    p.M = cout; p.N = kpad;
    if (ntaps == 9 && p.bni == 1 && (p.bw == 8 || p.bw % 16 == 0)) {
        // tap-row kernel: M chunks = (dy, 64-channel dY chunk), N = the three dx taps of one 64-channel X chunk
        p.co_chunks = pad64(cout) / 64;
        p.m_tiles = (3 * p.co_chunks + 1) / 2;
        p.n_tiles = kpad / 64;
        p.cchunks1 = pad64(c1) / 64;
        p.bn = 192;
        p.ntaps = 9; p.kw = 3;
        p.a_mn = 1; p.b_mn = 1;
        p.c_col_lo = kpad;
        pick_wgrad_split(&p, p.m_tiles * p.n_tiles, 8);
        p.C = dw; p.ldc = 9LL * kpad; p.out_mode = OUT_F32_ATOMIC;
        CUtensorMap ma, mb, mb2;
        if (int e = nhwc_map(&ma, dy, cout, ld_dy, n, h, w, p.bw, p.bh, 1)) return e;
        if (int e = nhwc_map(&mb, x1, c1, ld1, n, h, w, p.bw + 2, p.bh, 1)) return e;
        if (x2) { if (int e = nhwc_map(&mb2, x2, c2, ld2, n, h, w, p.bw + 2, p.bh, 1)) return e; } else mb2 = mb;
        return launch_gemm<tc_wgrad_rows_kernel>("tc_wgrad_rows", 0, ma, mb, mb2, p, static_cast<cudaStream_t>(stream));
    }
    p.m_tiles = (cout + 127) / 128;
    p.bn = x2 ? pick_bn(pad64(c1), 256, 64) : pick_bn(kpad, 256, 64);
    if (x2 && pad64(c2) % p.bn) p.bn = 64;
    p.n_tiles = kpad / p.bn;
    p.n_split = x2 ? pad64(c1) : INT_MAX;
    p.ntaps = ntaps; p.kw = taps_per_row(ntaps);
    p.batches = ntaps; p.bdiv = ntaps; p.c_col_lo = kpad;
    p.a_mn = 1; p.b_mn = 1;
    pick_wgrad_split(&p, ntaps * p.m_tiles * p.n_tiles, 6);  // epilogue ~ 6 k-iterations (fp32 vector atomics)
    p.C = dw; p.ldc = 1LL * ntaps * kpad; p.out_mode = OUT_F32_ATOMIC;
    p.row_map = row_map;
    (void)pixels;
    CUtensorMap ma, mb, mb2;
    if (int e = nhwc_map(&ma, dy, cout, ld_dy, n, h, w, p.bw, p.bh, p.bni)) return e;
    if (int e = nhwc_map(&mb, x1, c1, ld1, n, h, w, p.bw, p.bh, p.bni)) return e;
    if (x2) { if (int e = nhwc_map(&mb2, x2, c2, ld2, n, h, w, p.bw, p.bh, p.bni)) return e; } else mb2 = mb;
    return launch_gemm<tc_gemm_kernel<GEMM_WGRAD>>("tc_gemm", 0, ma, mb2, mb, p, static_cast<cudaStream_t>(stream));
}

int adm_device_error(void) {
    int v = 0;
    if (cudaMemcpyFromSymbol(&v, g_device_error, sizeof(int)) != cudaSuccess) return -1;
    return v;
}

int adm_gemm_batched(const adm_gemm_desc* d, void* stream) {
    GemmParams p;
    init_params(&p);
    p.M = d->m; p.N = d->n;
    p.m_tiles = (d->m + 127) / 128;
    p.bn = d->b.mn_major ? pick_bn(d->n, 256, 64) : pick_bn(d->n, 256, 16);
    p.n_tiles = (d->n + p.bn - 1) / p.bn;
    p.k_total = (d->k + 63) / 64;
    p.batches = d->batches; p.bdiv = d->bdiv > 0 ? d->bdiv : 1;
    p.a_mn = d->a.mn_major; p.b_mn = d->b.mn_major;
    p.a_c0 = d->a.c0; p.a_c0_lo = d->a.c0_lo; p.a_c1 = d->a.c1; p.a_c1_lo = d->a.c1_lo; p.a_bhi = d->a.bhi; p.a_blo = d->a.blo;
    p.b_c0 = d->b.c0; p.b_c0_lo = d->b.c0_lo; p.b_c1 = d->b.c1; p.b_c1_lo = d->b.c1_lo; p.b_bhi = d->b.bhi; p.b_blo = d->b.blo;
    int splits = d->splits > 0 ? d->splits : 1;
    if (splits > p.k_total) splits = p.k_total;
    p.k_iters = (p.k_total + splits - 1) / splits;
    p.splits = (p.k_total + p.k_iters - 1) / p.k_iters;
    if (p.splits > 1 && d->out_mode != OUT_F32_ATOMIC) { set_error("gemm_batched: split-K needs the atomic fp32 output mode"); return ADM_ERR_SHAPE; }
    p.C = d->c; p.ldc = d->ldc; p.c_bhi = d->c_bhi; p.c_blo = d->c_blo; p.c_col_lo = d->c_col_lo;
    p.bias = d->bias; p.residual = static_cast<const __nv_bfloat16*>(d->residual); p.ldr = d->ldr;
    p.alpha = d->alpha; p.out_mode = d->out_mode;
    CUtensorMap ma, mb;
    {
        const long long dims[3] = {d->a.dim0, d->a.dim1, d->a.dim2};
        const long long str[2] = {d->a.stride1, d->a.stride2};
        const int box[3] = {64, d->a.mn_major ? 64 : 128, 1};
        if (int e = encode_map(&ma, d->a.ptr, 3, dims, str, box)) return e;
    }
    {
        const long long dims[3] = {d->b.dim0, d->b.dim1, d->b.dim2};
        const long long str[2] = {d->b.stride1, d->b.stride2};
        const int box[3] = {64, d->b.mn_major ? 64 : p.bn, 1};
        if (int e = encode_map(&mb, d->b.ptr, 3, dims, str, box)) return e;
    }
    return launch_gemm<tc_gemm_kernel<GEMM_PLAIN>>("tc_gemm", 0, ma, ma, mb, p, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
