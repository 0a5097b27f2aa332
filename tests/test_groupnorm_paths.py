"""GroupNorm path by path: adm_gn_forward / adm_gn_apply / adm_gn_bwd (norm.cu) at the batch sizes that route to each
kernel, and at the cluster, group and pixel edges where they go wrong.  Each row of CASES names the kernels its shape
must run, the cluster size K of the fused kernels and the edge it exists for; one checker runs every row:

  * path     the CUDA kernels (and the split paths' memset) recorded under torch.profiler are exactly the expected
             list, the fused kernels' grid is n K CTAs (so the cluster size is K), and adm_launch_count() grows by the
             number of kernels.  gn_cluster_size is restated for the 148 SMs of a B200.  The launches of all rows are
             recorded once per module in a fresh process (see `routes`).
  * inputs   x1, x2, dy, add, params, gamma, beta and the backward's coef are views into NaN-filled buffers (channels
             past C, one image or row before and after); the workspaces `work` and `bcoef` are NaN-filled.  A read
             outside the view, or a workspace that is not cleared before it is accumulated into, shows up as NaN.
  * outputs  y, dx1, dx2, coef and dparams are views into sentinel-filled buffers with extra channels and guard images;
             dgamma, dbeta, dbias1 and dbias1b accumulate onto finite random values with guard elements on either
             side.  Every element outside the views keeps its bits; with dy_scratch = 0, so does all of dy.
  * values   every element against an fp64 reference from the same bf16 / fp32 operands.  Forward: F.group_norm,
             addcmul(shift, ., 1 + scale), SiLU, dropout (the mask restated below), avg_pool2d / nearest-up.  coef is
             [N, C, 4] = {A, B, mean, rstd} with y = act(x A + B).  Backward: autograd of the same forward at the mean
             and rstd of the coef the forward kernel returned (checked first), plus the adjoint of `add` (add / 4
             spread for add_mode 1, 2x2 sum for add_mode 2).

The bound is first order in the unit roundoffs u = 2^-24 (fp32) and 2^-8 (bf16, as in the conv and attention files),
written through absolute-value shadows in fp64.  Its parts, from the kernels' arithmetic:

  statistics  s = sum x and q = sum x^2 are fp32 sums whose depth D is the kernel's serial chain plus its merges: P
              pixels per thread (ceil(HW / (chunks * lanes))), the sum over the `lanes` threads of a channel vector,
              the `chunks` atomics (split) or K cluster partials (fused), then the cpg channels of the group (split:
              +2 for the pairwise 4-pixel unroll).  With a = mean |x|, b = mean x^2 over the group (L = cpg HW):
                  |d mean| <= (D + 2) u a
                  |d var|  <= (3 D + 9) u b        one-pass q / L - mean^2: relative to var it grows as 1 + mean^2/var
                  eps_r    =  (1 - rho)^-1/2 - 1 + 4 u,   rho = (|d var| + u (var + eps)) / (var + eps)   (rsqrtf 2 ulp)
  coef        A = rstd gamma (1 + scale), B = (beta - mean rstd gamma)(1 + scale) + shift, each a few fp32 roundings
              (3 u |A|, 6 u of B's shadow S_B) on top of the statistics.
  forward     pre-activation v = x A + B:  e_v = |A| (|x - mean| eps_r + |d mean|) + 6 u (|x A| + S_B)
              SiLU by tanh.approx.f32 (max error 2^-10.987, PTX ISA) on v / 2:  e_y = 1.1 e_v + (2^-11.987 + 4 u) |v|
              (|silu'| <= 1.1); dropout multiply 2 u, the 2x2 average 3 u; bf16 store 2^-8 |y|.
  backward    dv = g mask silu'(v) with v = x A + B from the fp32 coef (7 u shadow, |silu''| <= 1/2) and the tanh
              error (|d silu' / dT| <= (1 + |v|) / 2): e_dv = G mask (7/2 u S_v + (1 + |v|)(2^-11.987 + 6 u)) + 4 u |dv|,
              G the shadow of the upstream gradient; reuse_dv stores dv as bf16 (+ 2^-8 |dv|) before pass 2.
              S1 = sum dv, S2 = rstd (sum dv x - mean sum dv) are sums of depth Db (P pixels, lanes, chunks / K):
                  |d S1| <= sum e_dv + Db u sum |dv|
                  |d S2| <= rstd (sum e_dv |x - mean| + (Db + 1) u sum |dv x| + (Db + 2) u |mean| sum |dv|) + 2 u |S2|
              M1, M2 = group means of gamma' S1, gamma' S2 (cpg + 3 roundings), dx = dv K1 + x K2 + K3:
                  e_dx = |K1| e_dv + rstd |d M1| + rstd^2 (|x| + |mean|) |d M2| + 8 u (shadow of the three terms)
                         + 4 u |add adjoint| + u |dx|, then 2^-8 |dx| for the bf16 store.
              dgamma, dbeta, dparams: the S1 / S2 errors times their factors, plus one rounding per atomic onto the
              prefill (n per channel).  dbias1: the dx1 bounds summed, plus a chain of (pixels per thread + lanes +
              atomics) roundings: the fused kernel's n K CTAs, or col_sums_kernel's grid.
The constants come from the roundings above and the documented accuracy of tanh.approx.f32 and rsqrtf, not from errors
measured on a GPU.  The |mean| / std = 16 row is where the one-pass variance term is largest (about 257 times its
value at zero mean); the test prints its share of the y bound there.

Dropout: the mask of vecmath.cuh is restated in numpy (uint32 / uint64 arithmetic) and compared exactly with what the
kernels draw: gn_apply over ones (as engine.export_dropout_masks does it) bit for bit, the zeros of y on the split and
K = 1, 2, 8 forward paths, the zeros the reuse_dv path leaves in dy, and, on the split and piped backward, the mask
read back from dx wherever keeping or dropping one element moves dx by more than four bounds.

The test_checker_* tests (CPU) show that the checker accepts an fp32 implementation of the chain and rejects subtly
wrong kernels; test_dropout_* check the restated mask itself.
"""
import json
import math
import os
import subprocess
import sys
from dataclasses import dataclass

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.test_conv_paths import _bits, _device_ready

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
B200_SMS = 148
SENTINEL = 1000.0
U = 2.0 ** -24  # fp32 unit roundoff
BF = 2.0 ** -8  # bf16 store, as in test_conv_paths / test_attention_paths
ET = 2.0 ** -10.987  # tanh.approx.f32: maximum error (PTX ISA)
RSQRT = 4 * U  # rsqrtf: 2 ulp
SEED = 0x243F6A8885A308D3
COUNTER = 7
GUARD_C = 24  # extra channels of every image buffer (a multiple of 8: rows stay 16-byte aligned)

# kernel names as torch.profiler reports them on the B200 (without "void adm::" and the parameter list)
MEMSET = "Memset"
STATS = "gn_stats_kernel"
APPLY = "gn_apply_kernel"
FWD = "gn_fwd_fused_kernel"
REDUCE = "gn_bwd_reduce_kernel"
BAPPLY = "gn_bwd_apply_kernel"
COLSUMS = "col_sums_kernel"
BWD = "gn_bwd_fused_kernel"


# ------------------------------------------------------------------------------------------------ host launch math
# restated from norm.cu for 148 SMs: the path and the summation chains the bound is written for
def cluster_size(n):
    """gn_cluster_size: the smallest K in {1, 2, 4, 8} with n K >= 60 % of the SMs; 0 = the split kernels."""
    want = (B200_SMS * 6 + 9) // 10
    k = 1
    while k < 8 and n * k < want:
        k *= 2
    return k if n * k >= want else 0


def threads_for(nvec):
    return 256 if nvec >= 256 else nvec * (256 // nvec)


def grid_for(work, threads, n_batch):
    cap = max(1, -(-8 * B200_SMS // n_batch))
    return max(1, min(-(-work // threads), cap))


def fused_lanes(v, hw, k):
    """Threads per channel vector of the fused kernels (gn_fused_threads / V)."""
    return max(1, min(512 // v, -(-hw // k)))


@dataclass(frozen=True)
class Case:
    name: str
    op: str  # "fwd" (adm_gn_forward), "apply" (adm_gn_apply) or "bwd" (adm_gn_bwd)
    n: int
    h: int
    w: int
    c1: int
    c2: int
    k: int  # cluster size the batch must pick; 0 = the split (multi-block) kernels
    edge: str
    groups: int = 0  # 0: min(32, C / 4), as the UNet engine picks
    eps: float = 1e-5
    act: bool = True
    params: bool = False  # adaptive (1 + scale), shift of UNetBlock
    drop: float = 0.0
    resample: int = 0  # 1: 2x2 average pool, 2: nearest-up
    shift: float = 0.0  # added to x1: its |mean| / std
    add_mode: int = -1  # bwd: -1 no skip-path gradient, else add_mode
    dparams: bool = False  # bwd
    dbias: int = 0  # bwd: 1 dbias1, 2 dbias1 and dbias1b
    scratch: bool = False  # bwd: dy_scratch
    need_dx: bool = True  # bwd

    @property
    def id(self):
        return f"{self.name}-{self.op}"

    @property
    def c(self):
        return self.c1 + self.c2

    @property
    def g(self):
        return self.groups or min(32, self.c // 4)

    @property
    def cpg(self):
        return self.c // self.g

    @property
    def hw(self):
        return self.h * self.w

    @property
    def out_hw(self):
        return {0: (self.h, self.w), 1: (self.h // 2, self.w // 2), 2: (2 * self.h, 2 * self.w)}[self.resample]

    @property
    def subpath(self):
        """Branch of gn_bwd_fused_kernel."""
        piped = self.resample == 0 and self.add_mode <= 0
        if piped and self.scratch and self.need_dx and (self.act or self.drop > 0):
            return "reuse_dv"
        return "piped" if piped else "non-piped"

    @property
    def kernels(self):
        if self.op == "apply":
            return [APPLY]
        if self.op == "fwd":
            return [FWD] if self.k else [MEMSET, STATS, APPLY]
        if self.k:
            return [BWD]
        return [MEMSET, REDUCE] + ([BAPPLY] + [COLSUMS] * self.dbias if self.need_dx else [])

    def lanes(self):
        v = self.c // 8
        return fused_lanes(v, self.hw, self.k) if self.k else threads_for(v) // v

    def stat_depth(self):
        """Depth of the forward's fp32 statistics sums (module docstring)."""
        t = self.lanes()
        if self.k:
            return -(-self.hw // (self.k * t)) + t + self.k + self.cpg
        chunks = grid_for(self.hw, t, self.n)
        return -(-self.hw // (chunks * t)) + 2 + t + chunks + self.cpg

    def bsum_depth(self):
        """Depth of the backward's S1 / S2 sums."""
        t = self.lanes()
        chunks = self.k if self.k else grid_for(self.hw, 2 * t, self.n)
        return -(-self.hw // (chunks * t)) + 1 + t + chunks

    def bias_depth(self):
        """Depth of the dbias1 column sums: fused, in the kernel's pass 2; split, col_sums_kernel over dx1."""
        if self.k:
            t = self.lanes()
            return -(-self.hw // (self.k * t)) + t + self.n * self.k
        v1 = self.c1 // 8
        t = threads_for(v1) // v1
        rows = self.n * self.hw
        chunks = grid_for(rows, t, 1)
        return -(-rows // (chunks * t)) + t + chunks


def _rows(name, n, h, w, c1, c2, k, edge, ops=("fwd", "bwd"), **kw):
    return [Case(name, op, n, h, w, c1, c2, k, edge, **kw) for op in ops]


NORM1 = dict(params=True, drop=0.1, dparams=True, dbias=1, scratch=True)  # engine.py block_bwd, norm1
CASES = [
    # path boundaries of gn_cluster_size on 148 SMs (n K >= 89)
    *_rows("split-n11", 11, 8, 8, 128, 0, 0, "largest batch of the split kernels", params=True, dparams=True, dbias=2),
    *_rows("k8-n12", 12, 8, 8, 128, 0, 8, "smallest fused batch, K = 8", params=True, dparams=True, dbias=1),
    *_rows("k8-n22", 22, 8, 8, 128, 0, 8, "largest K = 8 batch"),
    *_rows("k4-n23", 23, 8, 8, 128, 0, 4, "smallest K = 4 batch", add_mode=0),
    *_rows("k4-n44", 44, 8, 8, 128, 0, 4, "largest K = 4 batch", dbias=2),
    *_rows("k2-n45", 45, 8, 8, 128, 0, 2, "smallest K = 2 batch", params=True, dparams=True),
    *_rows("k2-n88", 88, 8, 8, 128, 0, 2, "largest K = 2 batch"),
    *_rows("k1-n89", 89, 8, 8, 128, 0, 1, "smallest K = 1 batch", add_mode=0, dbias=1),
    # the benchmark's shapes: CIFAR at batch 128, CelebAHQ-latent at batch 48
    *_rows("cifar-32x32", 128, 32, 32, 192, 0, 1, "CIFAR 32x32 level, C = 192"),
    *_rows("cifar-16x16-down", 128, 16, 16, 384, 0, 1, "CIFAR down block (norm0): avg-pool on the store",
           resample=1, add_mode=1, scratch=True, dbias=1),
    *_rows("cifar-8x8-up-concat", 128, 8, 8, 384, 384, 1, "CIFAR decoder (norm0): concat 384 + 384, nearest-up",
           resample=2, add_mode=2, scratch=True, dbias=2),
    *_rows("cifar-norm2", 128, 16, 16, 384, 0, 1, "norm2 before attention: no SiLU, skip gradient, two bias sinks",
           act=False, add_mode=0, dbias=2),
    *_rows("celeb-64x64", 48, 64, 64, 96, 0, 2, "CelebAHQ 64x64 level, group size 4"),
    *_rows("celeb-16x16-c288", 48, 16, 16, 288, 0, 2, "C = 288, group size 9: channel vectors span two groups",
           params=True, dparams=True),
    *_rows("celeb-concat-384+288", 48, 16, 16, 384, 288, 2, "decoder concat 384 + 288, group size 21",
           add_mode=0, scratch=True, dbias=1),
    # edges
    *_rows("k8-6x10", 12, 6, 10, 64, 0, 8, "60 pixels over 8 CTAs of 8 lanes: the last CTA gets 4"),
    *_rows("split-12x20", 4, 12, 20, 128, 64, 0, "split kernels: non-square, concat, avg-pool",
           resample=1, add_mode=1, dbias=2),
    *_rows("hw4-c768", 128, 2, 2, 768, 0, 1, "4 pixels, fewer than the 5 lanes per channel vector"),
    *_rows("c2048-k8", 16, 4, 4, 2048, 0, 8, "largest C: the largest shared-memory launch (184 KB)", dbias=1),
    *_rows("c2048-split", 2, 4, 4, 2048, 0, 0, "largest C on the split kernels", dbias=1),
    *_rows("eps1e-6", 24, 8, 8, 256, 0, 4, "eps = 1e-6, as SongUNet uses", eps=1e-6),
    *_rows("mean16", 128, 16, 16, 192, 0, 1, "|mean| / std = 16 (a conv output with a bias): one-pass variance",
           shift=16.0, params=True, dparams=True),
    # the engine's three backward calls (engine.py block_bwd) and dx1 = None
    Case("norm1", "bwd", 48, 32, 32, 192, 0, 2, "norm1: params, dropout, dparams, dy_scratch (reuse_dv)", **NORM1),
    Case("norm1-split", "bwd", 8, 16, 16, 128, 0, 0, "norm1 on the split kernels", **NORM1),
    Case("params-only", "bwd", 44, 8, 8, 256, 0, 4, "dx1 = None: only the parameter gradients", params=True,
         dparams=True, need_dx=False),
    Case("params-only-split", "bwd", 6, 8, 8, 256, 0, 0, "dx1 = None on the split kernels", params=True,
         dparams=True, need_dx=False),
    # dropout
    Case("drop-split", "fwd", 8, 16, 16, 128, 0, 0, "dropout, split forward", params=True, drop=0.1),
    Case("drop-k1", "fwd", 128, 8, 8, 192, 0, 1, "dropout, K = 1", params=True, drop=0.1),
    Case("drop-k2", "fwd", 48, 16, 16, 192, 0, 2, "dropout, K = 2", params=True, drop=0.13),
    Case("drop-k8", "fwd", 12, 16, 16, 128, 0, 8, "dropout, K = 8", params=True, drop=0.1),
    Case("drop-split", "bwd", 8, 16, 16, 128, 0, 0, "dropout, split backward", params=True, drop=0.1),
    Case("drop-k8-piped", "bwd", 12, 16, 16, 128, 0, 8, "dropout, fused piped backward (dy kept)", params=True,
         drop=0.1, dparams=True),
    Case("ones-mask", "apply", 128, 16, 16, 192, 0, 0, "engine.export_dropout_masks: gn_apply over ones",
         act=False, drop=0.1),
]


# ------------------------------------------------------------------------------------------------ dropout mask, restated
_M64 = (1 << 64) - 1
_LANE_MUL = np.array([0x9E3779B1, 0x85EBCA6B, 0xC2B2AE35, 0x27D4EB2F, 0x165667B1, 0xD3A2646D, 0xFD7046C5, 0xB55A4F09],
                     dtype=np.uint32)


def dropout_mask(seed, counter, p, n, hw, c, lanes=_LANE_MUL):
    """keep-scales [n, hw, c] (float32: 0 or 1 / (1 - p)) of vecmath.cuh: seed += counter * 0x9E3779B97F4A7C15, the
    drop_ctx avalanche, drop_base of the vector index (sample * HW + pixel) * (C / 8) + channel / 8 (uint32), one
    multiplicative hash per lane compared with floor(p 2^32)."""
    s = (seed + counter * 0x9E3779B97F4A7C15) & _M64
    z = (s * 0x9E3779B97F4A7C15) & _M64
    z ^= z >> 32
    z = (z * 0xD6E8FEB86659FD93) & _M64
    z ^= z >> 32
    s0, s1 = np.uint32(z & 0xFFFFFFFF), np.uint32(z >> 32)
    pf = np.float32(p)
    thr = 0xFFFFFFFF if pf >= 1 else int(float(pf) * 4294967296.0)
    keep = np.float32(1) / (np.float32(1) - pf)
    vec = (np.arange(n * hw * (c // 8), dtype=np.uint64) & 0xFFFFFFFF).astype(np.uint32)
    h = (vec ^ s0) * np.uint32(0x9E3779B1)
    h = h ^ (h >> np.uint32(15)) ^ s1
    h = h * np.uint32(0x85EBCA77)
    h ^= h >> np.uint32(13)
    kept = (h[:, None] * lanes[None, :]) >= np.uint32(thr)
    return np.where(kept, keep, np.float32(0)).astype(np.float32).reshape(n, hw, c)


# ------------------------------------------------------------------------------------------------ operands
def poisoned(t, before=1, after=1, extra=GUARD_C):
    """t [n, ..., c] as a view into a NaN-filled buffer with `extra` channels and before / after slabs of dim 0."""
    buf = torch.full((before + t.shape[0] + after, *t.shape[1:-1], t.shape[-1] + extra), float("nan"), dtype=t.dtype,
                     device=t.device)
    view = buf[before:before + t.shape[0], ..., :t.shape[-1]]
    view.copy_(t)
    return view


def operands(case, device, seed=0):
    """The case's inputs, each inside its NaN-filled buffer, and (dropout) the restated mask [n, H, W, C]."""
    c = case
    g = torch.Generator(device="cpu").manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, generator=g).to(device)
    t = {"x1": poisoned((rnd(c.n, c.h, c.w, c.c1) + c.shift).to(BF16)),
         "x2": poisoned(rnd(c.n, c.h, c.w, c.c2).to(BF16)) if c.c2 else None}
    for name, val in (("gamma", 1 + 0.2 * rnd(c.c)), ("beta", 0.2 * rnd(c.c))):
        buf = torch.full((c.c + 16,), float("nan"), device=device)
        t[name] = buf[8:8 + c.c]
        t[name].copy_(val)
    t["params"] = None
    if c.params:  # [n, 2C] = (scale | shift), 8 NaN columns on both sides and a NaN row before and after
        buf = torch.full((c.n + 2, 2 * c.c + 16), float("nan"), device=device)
        t["params"] = buf[1:1 + c.n, 8:8 + 2 * c.c]
        t["params"].copy_(0.3 * rnd(c.n, 2 * c.c))
    t["counter"] = torch.tensor([COUNTER], dtype=torch.int64, device=device)
    t["mask"] = None
    if c.drop:
        m = dropout_mask(SEED, COUNTER, c.drop, c.n, c.hw, c.c)
        t["mask"] = torch.from_numpy(m).reshape(c.n, c.h, c.w, c.c).to(device)
    if c.op == "bwd":
        ho, wo = c.out_hw
        t["dy0"] = rnd(c.n, ho, wo, c.c).to(BF16)  # dy as given: the kernel may overwrite t["dy"] (dy_scratch)
        t["dy"] = poisoned(t["dy0"])
        t["add"] = None
        if c.add_mode >= 0:
            ah, aw = {0: (c.h, c.w), 1: (c.h // 2, c.w // 2), 2: (2 * c.h, 2 * c.w)}[c.add_mode]
            t["add"] = poisoned(rnd(c.n, ah, aw, c.c).to(BF16))
        t["pre"] = {k: rnd(n_) for k, n_ in (("dgamma", c.c), ("dbeta", c.c), ("dbias1", c.c1), ("dbias1b", c.c1))}
    if c.op == "apply":  # export_dropout_masks: ones through A = 1, B = 0
        t["x1"] = poisoned(torch.ones(c.n, c.h, c.w, c.c1, dtype=BF16, device=device))
        coef = torch.zeros(c.n, c.c, 4, device=device)
        coef[..., 0] = 1
        t["coef"] = poisoned(coef, 1, 1, 0)
    return t


# ------------------------------------------------------------------------------------------------ reference and bound
def _nchw(x):
    return x.to(F64).permute(0, 3, 1, 2)


def _nhwc(x):
    return x.permute(0, 2, 3, 1)


def _x(t):
    return _nchw(t["x1"]) if t["x2"] is None else torch.cat([_nchw(t["x1"]), _nchw(t["x2"])], 1)


def _affine(case, t, dtype=F64):
    """gamma, beta [C] and scale, shift [n, C] (zeros without params)."""
    gam, bet = t["gamma"].to(dtype), t["beta"].to(dtype)
    if t["params"] is None:
        z = torch.zeros(case.n, case.c, dtype=dtype, device=gam.device)
        return gam, bet, z, z.clone()
    p = t["params"].to(dtype)
    return gam, bet, p[:, :case.c], p[:, case.c:]


def _e4(z):
    return z[..., None, None]


def _up(z):
    return F.interpolate(z, scale_factor=2, mode="nearest")


def _post(case, t, v):
    """pre-activation v [n, C, H, W] -> output: SiLU, dropout, resample."""
    y = F.silu(v) if case.act else v
    if t["mask"] is not None:
        y = y * _nchw(t["mask"]).to(v.dtype)
    if case.resample == 1:
        y = F.avg_pool2d(y, 2)
    elif case.resample == 2:
        y = _up(y)
    return y


def _group_mean(z, case):
    """[n, C, ...] -> mean over each group's channels and pixels, broadcast back to [n, C]."""
    n = z.shape[0]
    return z.reshape(n, case.g, -1).mean(-1).repeat_interleave(case.cpg, 1)


def forward_reference(case, t, dtype=F64, mean_c=None, rstd_c=None):
    """y [n, C, Ho, Wo]; with mean_c / rstd_c [n, C] the normalisation uses those statistics (mutants)."""
    gam, bet, sc, sh = _affine(case, t, dtype)
    x = _x(t).to(dtype)
    if mean_c is None:
        gn = F.group_norm(x, case.g, gam, bet, case.eps)
    else:
        gn = (x - _e4(mean_c)) * _e4(rstd_c) * _e4(gam) + _e4(bet)
    return _post(case, t, torch.addcmul(_e4(sh), gn, _e4(1 + sc)))


def forward_expected(case, t):
    """{"y": (ref, bound) [n, Ho, Wo, C], "coef": (ref, bound) [n, C, 4]} (module docstring)."""
    gam, bet, sc, sh = _affine(case, t)
    x = _x(t)
    sig = 1 + sc
    xg = x.reshape(case.n, case.g, -1)
    mean, var = xg.mean(-1), xg.var(-1, unbiased=False)
    a, b = xg.abs().mean(-1), (xg * xg).mean(-1)
    d = case.stat_depth()
    dm = (d + 2) * U * a
    rho = ((3 * d + 9) * U * b + U * (var + case.eps)) / (var + case.eps)
    eps_r = (1 - rho) ** -0.5 - 1 + RSQRT
    pc = lambda z: z.repeat_interleave(case.cpg, 1)
    m, r, dm, eps_r = pc(mean), pc((var + case.eps) ** -0.5), pc(dm), pc(eps_r)
    A = r * gam * sig
    B = (bet - m * r * gam) * sig + sh
    s_b = sig.abs() * ((m * r * gam).abs() + bet.abs()) + sh.abs()
    coef = torch.stack([A, B, m, r], -1)
    coef_bound = torch.stack([A.abs() * (eps_r + 3 * U), A.abs() * (m.abs() * eps_r + dm) + 6 * U * s_b, dm,
                              r * eps_r], -1)
    v = x * _e4(A) + _e4(B)
    e = _e4(A.abs()) * ((x - _e4(m)).abs() * _e4(eps_r) + _e4(dm)) + 6 * U * (x.abs() * _e4(A.abs()) + _e4(s_b))
    y0 = v
    if case.act:
        e = 1.1 * e + (ET / 2 + 4 * U) * v.abs()
        y0 = F.silu(v)
    if t["mask"] is not None:
        mk = _nchw(t["mask"])
        e, y0 = e * mk, y0 * mk
        e = e + 2 * U * y0.abs()
    if case.resample == 1:
        e = F.avg_pool2d(e, 2) + 3 * U * F.avg_pool2d(y0.abs(), 2)
    elif case.resample == 2:
        e = _up(e)
    y = forward_reference(case, t)
    return {"y": (_nhwc(y), _nhwc(e * (1 + BF) + BF * y.abs())), "coef": (coef, coef_bound)}


class _NormalizeAt(torch.autograd.Function):
    """xhat = (x - mean) rstd at given per-(n, c) statistics, with GroupNorm's adjoint at those statistics:
    dx = rstd (g - mean_g(g) - xhat mean_g(g xhat))."""

    @staticmethod
    def forward(ctx, x, mean, rstd, case):
        xhat = (x - _e4(mean)) * _e4(rstd)
        ctx.save_for_backward(xhat, rstd)
        ctx.case = case
        return xhat

    @staticmethod
    def backward(ctx, g):
        xhat, rstd = ctx.saved_tensors
        gm = lambda z: _e4(_group_mean(z, ctx.case))
        return _e4(rstd) * (g - gm(g) - xhat * gm(g * xhat)), None, None, None


def _add_adjoint(case, add):
    """Gradient the skip path adds to dx: add (mode 0), add / 4 spread (mode 1), 2x2 sum (mode 2)."""
    if case.add_mode == 1:
        return _up(add) / 4
    if case.add_mode == 2:
        return F.avg_pool2d(add, 2) * 4
    return add


def _upstream(case, dy):
    """The output gradient at the input resolution (the adjoint of the resample)."""
    if case.resample == 1:
        return _up(dy) / 4
    if case.resample == 2:
        return F.avg_pool2d(dy, 2) * 4
    return dy


def backward_reference(case, t, coef, dtype=F64):
    """{"dx" [n, C, H, W], "dgamma", "dbeta" [C], "dscale", "dshift" [n, C]} by autograd in `dtype` at the mean and rstd
    of `coef`; fp32 (CPU checker tests) uses F.group_norm's own statistics instead."""
    gam, bet, sc, sh = (z.detach().requires_grad_(True) for z in _affine(case, t, dtype))
    x = _x(t).to(dtype).requires_grad_(True)
    if dtype == F64:
        xhat = _NormalizeAt.apply(x, coef[..., 2].to(F64), coef[..., 3].to(F64), case)
        gn = xhat * _e4(gam) + _e4(bet)
    else:
        gn = F.group_norm(x, case.g, gam, bet, case.eps)
    y = _post(case, t, torch.addcmul(_e4(sh), gn, _e4(1 + sc)))
    dx, dgam, dbet, dsc, dsh = torch.autograd.grad(y, (x, gam, bet, sc, sh), _nchw(t["dy0"]).to(dtype))
    if t["add"] is not None:
        dx = dx + _add_adjoint(case, _nchw(t["add"]).to(dtype))
    return {"dx": dx, "dgamma": dgam, "dbeta": dbet, "dscale": dsc, "dshift": dsh}


def backward_expected(case, t, coef, ref=None):
    """{output: (ref, bound)} of the backward (module docstring), given the coef the forward kernel returned.  Also
    returns the pieces the dropout read-back needs."""
    c = case
    ref = ref or backward_reference(c, t, coef)
    gam, bet, sc, sh = _affine(c, t)
    sig = 1 + sc
    x = _x(t)
    ck = coef.to(F64)
    A, B, m, r = ck[..., 0], ck[..., 1], ck[..., 2], ck[..., 3]
    s_v = x.abs() * _e4(A.abs()) + _e4(sig.abs() * ((m * r * gam).abs() + bet.abs()) + sh.abs())
    v = (x - _e4(m)) * _e4(r * gam * sig) + _e4(bet * sig + sh)
    dy = _nchw(t["dy0"])
    g_in, g_abs = _upstream(c, dy), _upstream(c, dy.abs())
    mk = _nchw(t["mask"]) if t["mask"] is not None else torch.ones_like(x)
    if c.act:
        s = torch.sigmoid(v)
        sp = s * (1 + v * (1 - s))
        e_sp = 3.5 * U * s_v + (1 + v.abs()) * (ET / 2 + 6 * U)
    else:
        sp, e_sp = torch.ones_like(v), torch.zeros_like(v)
    dv = g_in * mk * sp
    e_dv = g_abs * mk * (e_sp + 4 * U * sp.abs())
    sum_p = lambda z: z.sum((2, 3))
    db = c.bsum_depth()
    xm = x - _e4(m)
    s1, s2 = sum_p(dv), r * sum_p(dv * xm)
    ds1 = sum_p(e_dv) + db * U * sum_p(dv.abs())
    ds2 = (r * (sum_p(e_dv * xm.abs()) + (db + 1) * U * sum_p((dv * x).abs()) + (db + 2) * U * m.abs() * sum_p(dv.abs()))
           + 2 * U * s2.abs())
    out, pre = {}, t["pre"]
    atom = (c.n + 1) * U
    out["dgamma"] = (pre["dgamma"].to(F64) + ref["dgamma"],
                     (sig.abs() * ds2 + 2 * U * (sig * s2).abs()).sum(0)
                     + atom * (pre["dgamma"].to(F64).abs() + (sig * s2).abs().sum(0)))
    out["dbeta"] = (pre["dbeta"].to(F64) + ref["dbeta"],
                    (sig.abs() * ds1 + 2 * U * (sig * s1).abs()).sum(0)
                    + atom * (pre["dbeta"].to(F64).abs() + (sig * s1).abs().sum(0)))
    if c.dparams:
        out["dparams"] = (torch.cat([ref["dscale"], ref["dshift"]], 1),
                          torch.cat([gam.abs() * ds2 + bet.abs() * ds1 + 2 * U * ((gam * s2).abs() + (bet * s1).abs()),
                                     ds1], 1))
    extra = {"dv": dv, "sp": sp, "g_in": g_in, "k1": r * gam * sig}
    if not c.need_dx:
        return out, extra
    gs = gam * sig
    gsum = lambda z: z.reshape(c.n, c.g, c.cpg).sum(-1).repeat_interleave(c.cpg, 1)
    L = c.cpg * c.hw
    m1, m2 = gsum(gs * s1) / L, gsum(gs * s2) / L
    dm1 = (gsum(gs.abs() * ds1) + (c.cpg + 3) * U * gsum((gs * s1).abs())) / L
    dm2 = (gsum(gs.abs() * ds2) + (c.cpg + 3) * U * gsum((gs * s2).abs())) / L
    k1 = _e4(r * gs)
    xa = x.abs() + _e4(m.abs())
    e_dv2 = e_dv + (BF * dv.abs() if c.k and c.subpath == "reuse_dv" else 0)
    e = (k1.abs() * e_dv2 + _e4(r * dm1) + _e4(r * r * dm2) * xa
         + 8 * U * ((k1 * dv).abs() + _e4(r * m1.abs()) + _e4(r * r * m2.abs()) * xa))
    if t["add"] is not None:
        e = e + 4 * U * _add_adjoint(c, _nchw(t["add"]).abs())
    dx = ref["dx"]
    e = e + U * dx.abs()
    bound = e * (1 + BF) + BF * dx.abs()
    out["dx1"] = (_nhwc(dx[:, :c.c1]), _nhwc(bound[:, :c.c1]))
    if c.c2:
        out["dx2"] = (_nhwc(dx[:, c.c1:]), _nhwc(bound[:, c.c1:]))
    for i, name in enumerate(("dbias1", "dbias1b")[:c.dbias]):
        p = pre[name].to(F64)
        col = dx[:, :c.c1].sum((0, 2, 3))
        out[name] = (p + col, bound[:, :c.c1].sum((0, 2, 3))
                     + c.bias_depth() * U * (p.abs() + dx[:, :c.c1].abs().sum((0, 2, 3))))
    extra["dx"], extra["bound"] = dx, bound
    return out, extra


# ------------------------------------------------------------------------------------------------ guarded outputs, checker
def _guarded(shape, dtype, device, before=1, after=1, extra=GUARD_C, fill=SENTINEL):
    """(buf, view, writable): a view of `shape` inside a `fill`-ed buffer with extra channels and guard slabs."""
    buf = torch.full((before + shape[0] + after, *shape[1:-1], shape[-1] + extra), fill, dtype=dtype, device=device)
    writable = torch.zeros(buf.shape, dtype=torch.bool, device=device)
    sl = (slice(before, before + shape[0]),) + (slice(None),) * (len(shape) - 2) + (slice(0, shape[-1]),)
    writable[sl] = True
    return buf, buf[sl], writable


def _accumulator(prefill, seed):
    """(buf, view, writable): `prefill` inside finite random values, 8 guard elements on either side."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    buf = torch.randn(prefill.numel() + 16, generator=g).to(prefill.device)
    buf[8:-8] = prefill
    writable = torch.zeros(buf.shape, dtype=torch.bool, device=buf.device)
    writable[8:-8] = True
    return buf, buf[8:-8], writable


def guarded_outputs(case, t, device):
    c = case
    outs = {}
    if c.op in ("fwd", "apply"):
        ho, wo = c.out_hw
        outs["y"] = _guarded((c.n, ho, wo, c.c), BF16, device)
    if c.op == "fwd":
        outs["coef"] = _guarded((c.n, c.c, 4), F32, device, extra=0)
    if c.op == "bwd":
        if c.need_dx:
            outs["dx1"] = _guarded((c.n, c.h, c.w, c.c1), BF16, device)
            if c.c2:
                outs["dx2"] = _guarded((c.n, c.h, c.w, c.c2), BF16, device)
        outs["dgamma"] = _accumulator(t["pre"]["dgamma"], 1)
        outs["dbeta"] = _accumulator(t["pre"]["dbeta"], 2)
        if c.dparams:
            buf, _, writable = _guarded((c.n, 2 * c.c + 8), F32, device, extra=8)
            writable[:, :8] = False  # the view starts 8 columns into its row: columns on both sides
            outs["dparams"] = (buf, buf[1:1 + c.n, 8:8 + 2 * c.c], writable)
        for i, name in enumerate(("dbias1", "dbias1b")[:c.dbias]):
            outs[name] = _accumulator(t["pre"][name], 3 + i)
        # dy is an input; with dy_scratch the kernel may overwrite its view (never anything around it)
        dyb = t["dy"]._base
        writable = torch.zeros(dyb.shape, dtype=torch.bool, device=device)
        if c.scratch:
            writable[1:1 + c.n, ..., :c.c] = True
        outs["dy"] = (dyb, t["dy"], writable)
    return outs


def verify(before, outs, expected):
    """Problems (strings) of one result and the largest |got - ref| / bound per output.  `before`: the buffers'
    contents before the call; `outs`: {name: (buf, view, writable)}; `expected`: {name: (ref, bound)}."""
    problems, worst = [], {}
    for name, (buf, view, writable) in outs.items():
        stray = (_bits(before[name]) != _bits(buf)) & ~writable
        if stray.any():
            idx = stray.nonzero()[:4].tolist()
            problems.append(f"{name}: {int(stray.sum())} elements outside the output changed, e.g. at {idx}")
        if name not in expected:
            continue
        got = view.to(F64)
        ref, bound = expected[name]
        if torch.isnan(got).any():
            problems.append(f"{name}: {int(torch.isnan(got).sum())} NaN outputs")
        err = (got - ref).abs()
        bad = ~(err <= bound)
        ratio = torch.where(bound > 0, err / bound, torch.where(err > 0, math.inf, 0.0))
        worst[name] = float(ratio.nan_to_num(math.inf).max())
        if bad.any():
            i = tuple(bad.nonzero()[0].tolist())
            problems.append(f"{name}: {int(bad.sum())} of {bad.numel()} elements outside the bound, first at {i}: got "
                            f"{float(got[i])}, ref {float(ref[i])}, bound {float(bound[i]):.3g}; "
                            f"max err/bound {worst[name]:.3g}")
    return problems, worst


# ------------------------------------------------------------------------------------------------ GPU: the table
def _src(x):
    return (None, 0, 0) if x is None else (x.data_ptr(), x.shape[-1], x.stride(2))


def _p(x):
    return None if x is None else x.data_ptr()


def _nan(*shape):
    return torch.full(shape, float("nan"), device="cuda")


def _forward_call(lib, case, t, coef, y):
    """adm_gn_forward into the views `coef` [n, C, 4] and `y`, with a NaN-filled workspace."""
    c = case
    p1, c1, ld1 = _src(t["x1"])
    p2, c2, ld2 = _src(t["x2"])
    work = _nan(2 * c.n * c.c + c.n)
    ldp = t["params"].stride(0) if t["params"] is not None else 0
    return lambda: lib.adm_gn_forward(p1, c1, ld1, p2, c2, ld2, c.n, c.h, c.w, c.g, c.eps, _p(t["gamma"]),
                                      _p(t["beta"]), _p(t["params"]), ldp, _p(work), _p(coef), int(c.act), c.drop,
                                      SEED, _p(t["counter"]), c.resample, _p(y), y.stride(2),
                                      torch.cuda.current_stream().cuda_stream)


def _call(lib, case, t, outs, coef):
    c = case
    stream = torch.cuda.current_stream().cuda_stream
    if c.op == "fwd":
        return _forward_call(lib, c, t, outs["coef"][1], outs["y"][1])
    y = outs.get("y", (None, None))[1]
    if c.op == "apply":
        p1, c1, ld1 = _src(t["x1"])
        return lambda: lib.adm_gn_apply(p1, c1, ld1, None, 0, 0, c.n, c.h, c.w, _p(coef), int(c.act), c.drop, SEED,
                                        _p(t["counter"]), c.resample, _p(y), y.stride(2), stream)
    p1, c1, ld1 = _src(t["x1"])
    p2, c2, ld2 = _src(t["x2"])
    work, bcoef = _nan(2 * c.n * c.c + c.n), _nan(c.n, c.c, 4)
    ldp = t["params"].stride(0) if t["params"] is not None else 0
    dp = outs.get("dparams", (None, None))[1]
    dx1 = outs.get("dx1", (None, None))[1]
    dx2 = outs.get("dx2", (None, None))[1]
    add = t["add"]
    o = lambda name: _p(outs[name][1]) if name in outs else None
    return lambda: lib.adm_gn_bwd(
        _p(t["dy"]), t["dy"].stride(2), p1, c1, ld1, p2, c2, ld2, c.n, c.h, c.w, c.g, _p(coef), _p(t["gamma"]),
        _p(t["beta"]), _p(t["params"]), ldp, int(c.act), c.drop, SEED, _p(t["counter"]), c.resample, _p(work),
        _p(bcoef), o("dgamma"), o("dbeta"), _p(dp), dp.stride(0) if dp is not None else 0, _p(add),
        add.stride(2) if add is not None else 0, max(c.add_mode, 0), _p(dx1), dx1.stride(2) if dx1 is not None else 0,
        _p(dx2), dx2.stride(2) if dx2 is not None else 0, o("dbias1"), o("dbias1b"), int(c.scratch), stream)


def _launches(fn, tmp_path):
    """(name, grid) of every kernel and memset fn runs, in start order, from torch.profiler's chrome trace; fn's
    return code."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        try:
            rc = fn()
        finally:
            torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    events = json.loads(path.read_text())["traceEvents"]
    ran = []
    for ev in events:
        name = ev.get("name", "")
        if ev.get("cat") == "kernel":
            name = name.split("(")[0].replace("void ", "").replace("adm::", "").strip()
        elif name.startswith("Memset") and ev.get("ph") == "X" and ev.get("cat") != "cuda_runtime":
            name = MEMSET
        else:
            continue
        ran.append((float(ev["ts"]), name, tuple(ev.get("args", {}).get("grid", ()))))
    return [(name, grid) for _, name, grid in sorted(ran)], rc


def _check_masks(case, t, outs, extra):
    """The dropout mask the kernels applied against the restated one (module docstring)."""
    keep = t["mask"] != 0
    if case.op in ("fwd", "apply"):
        drawn = outs["y"][1] != 0
        assert torch.equal(drawn, keep), f"{int((drawn != keep).sum())} mask elements differ from the restatement"
        return "y"
    if case.subpath == "reuse_dv" and case.k:
        drawn = outs["dy"][1] != 0  # pass 1 left dv (0 where dropped) in dy's place
        assert torch.equal(drawn, keep), f"{int((drawn != keep).sum())} mask elements of dv differ"
        return "dv"
    # dx moves by K1 * g * silu'(v) / (1 - p) when one element is kept instead of dropped
    dx_got = torch.cat([_nchw(outs["dx1"][1])] + ([_nchw(outs["dx2"][1])] if case.c2 else []), 1)
    k1, mk = _e4(extra["k1"]), _nchw(t["mask"])
    step = k1 * extra["g_in"] * extra["sp"] * float(np.float32(1) / (np.float32(1) - np.float32(case.drop)))
    base = extra["dx"] - k1 * extra["dv"]
    drawn = (dx_got - base - step).abs() < (dx_got - base).abs()
    sep = step.abs() > 4 * extra["bound"]
    assert float(sep.double().mean()) > 0.9, "too few elements where the mask is observable"
    assert torch.equal(drawn[sep], (mk != 0)[sep]), f"{int((drawn != (mk != 0))[sep].sum())} mask elements differ"
    return f"dx ({float(sep.double().mean()):.3f} observable)"


def _prepare(lib, case, forward=True):
    """Operands, the coef input (bwd: the forward kernel's, in a guarded buffer; sentinels without `forward`) and the
    guarded outputs."""
    t = operands(case, "cuda")
    coef = t.get("coef")
    if case.op == "bwd":
        cbuf, coef, cw = _guarded((case.n, case.c, 4), F32, "cuda", extra=0)
        t["coef_guard"] = (cbuf.clone(), cbuf, coef, cw)
        if forward:
            y = torch.empty(case.n, *case.out_hw, case.c, dtype=BF16, device="cuda")
            assert _forward_call(lib, case, t, coef, y)() == 0
    return t, coef, guarded_outputs(case, t, "cuda")


def _rejected_case(name, op, kw):
    return Case(**{**dict(name=name, op=op, n=12, h=4, w=4, c1=64, c2=0, k=8, edge="rejected", dbias=1, dparams=True),
                   **kw})


def _record_routes(path):
    """Runs every row's call (and every rejected shape's) under torch.profiler and writes {id: [[name, grid], ...]}."""
    import pathlib
    lib, _ = _device_ready()
    out = pathlib.Path(path)
    calls = [(c.id, c, True) for c in CASES] + [(f"rejected-{n}-{op}", _rejected_case(n, op, kw), False)
                                                  for n, op, kw, _ in REJECTED]
    routes = {}
    for key, case, forward in calls:
        t, coef, outs = _prepare(lib, case, forward)
        routes[key] = [[name, list(grid)] for name, grid in _launches(_call(lib, case, t, outs, coef), out)[0]]
    (out / "routes.json").write_text(json.dumps(routes))


@pytest.fixture(scope="module")
def routes(tmp_path_factory):
    """The (kernel, grid) list of every call, recorded in a fresh process.  In a process that profiled before it
    captured CUDA graphs (the path tests of other files run before the parity tests), later torch.profiler sessions
    lose kernel records, so the launches are not recorded in the test process itself."""
    out = tmp_path_factory.mktemp("routes")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = f"import sys; sys.path.insert(0, {root!r}); from tests.test_groupnorm_paths import _record_routes; " \
           f"_record_routes({str(out)!r})"
    subprocess.run([sys.executable, *(["-s"] if sys.flags.no_user_site else []), "-c", code], check=True, timeout=900)
    return {k: [(name, tuple(grid)) for name, grid in v] for k, v in json.loads((out / "routes.json").read_text()).items()}


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_groupnorm_path(case, routes):
    lib, _ = _device_ready()
    assert cluster_size(case.n) == case.k or case.op == "apply"
    t, coef, outs = _prepare(lib, case)
    torch.cuda.synchronize()
    inputs = {}
    if case.op == "bwd":  # the statistics the backward works at: the forward kernel's coef, checked first
        cbefore, cbuf, _, cw = t["coef_guard"]
        problems, _ = verify({"coef": cbefore}, {"coef": (cbuf, coef, cw)}, {"coef": forward_expected(case, t)["coef"]})
        assert not problems, f"{case.id} forward coef: " + "; ".join(problems)
        inputs["coef"] = cbuf
    elif coef is not None:
        inputs["coef"] = coef._base
    for name in ("x1", "x2", "params", "add", "gamma", "beta"):
        if t.get(name) is not None:
            inputs[name] = t[name]._base
    inputs_before = {k: v.clone() for k, v in inputs.items()}
    before = {k: buf.clone() for k, (buf, _, _) in outs.items()}
    launches = lib.adm_launch_count()
    rc = _call(lib, case, t, outs, coef)()
    torch.cuda.synchronize()
    assert rc == 0, lib.adm_last_error()
    ran = routes[case.id]
    names = [name for name, _ in ran]
    assert names == case.kernels, f"{case.id} ({case.edge}) ran {names}, expected {case.kernels}"
    for name, grid in ran:
        if name in (FWD, BWD):
            assert grid[0] == case.n * case.k, f"{name} grid {grid}: cluster size {grid[0] / case.n}, expected {case.k}"
    assert lib.adm_launch_count() == launches + len([k for k in case.kernels if k != MEMSET])
    assert lib.adm_device_error() == 0
    for k, v in inputs.items():
        assert torch.equal(_bits(v), _bits(inputs_before[k])), f"input {k} was written"
    extra = None
    if case.op == "fwd":
        expected = forward_expected(case, t)
    elif case.op == "apply":
        expected = {"y": (t["mask"].to(BF16).to(F64), torch.zeros_like(t["mask"], dtype=F64))}
    else:
        expected, extra = backward_expected(case, t, coef)
    problems, worst = verify(before, outs, expected)
    assert not problems, f"{case.id} ({case.edge}): " + "; ".join(problems)
    note = ""
    if case.drop:
        note = ", mask from " + _check_masks(case, t, outs, extra)
    if case.shift:
        note += f", one-pass variance share of the y bound {_variance_share(case, t):.3g}"
    path = f"K = {case.k}" if case.k else "split"
    sub = f" {case.subpath}" if case.op == "bwd" and case.k else ""
    print(f"{case.id}: {names} ({path}{sub}), max |err| / bound = "
          + ", ".join(f"{k} {v:.3g}" for k, v in worst.items()) + note)


def _variance_share(case, t):
    """Largest share of the y bound that the one-pass variance term takes: |A| |x - mean| (3 D + 9) u b / (2 (var +
    eps)), the rstd error it causes, carried to y (resample 0 rows)."""
    full = forward_expected(case, t)["y"][1]
    x = _x(t)
    xg = x.reshape(case.n, case.g, -1)
    var = xg.var(-1, unbiased=False)
    pc = lambda z: z.repeat_interleave(case.cpg, 1)
    rel = pc(0.5 * (3 * case.stat_depth() + 9) * U * (xg * xg).mean(-1) / (var + case.eps))
    gam, _, sc, _ = _affine(case, t)
    part = _e4((rel * pc(var + case.eps) ** -0.5 * gam * (1 + sc)).abs()) * (x - _e4(pc(xg.mean(-1)))).abs()
    if case.act:
        part = 1.1 * part
    return float((_nhwc(part) / full).max())


@pytest.mark.gpu
def test_seed_counter_changes_and_reproduces_the_mask():
    lib, _ = _device_ready()
    case = next(c for c in CASES if c.op == "apply")
    t = operands(case, "cuda")
    got = []
    for counter in (COUNTER, COUNTER + 1, COUNTER):
        t["counter"].fill_(counter)
        outs = guarded_outputs(case, t, "cuda")
        assert _call(lib, case, t, outs, t["coef"])() == 0
        got.append(outs["y"][1].clone())
    torch.cuda.synchronize()
    assert torch.equal(_bits(got[0]), _bits(got[2]))
    assert not torch.equal(got[0], got[1])
    nxt = dropout_mask(SEED, COUNTER + 1, case.drop, case.n, case.hw, case.c)
    assert torch.equal(_bits(got[1].cpu()), _bits(torch.from_numpy(nxt).reshape(got[1].shape).to(BF16)))


# shapes the entry points reject before launching anything: (name, op, case overrides, message)
REJECTED = [
    ("c2056", "fwd", dict(c1=2056, groups=8), "gn_forward: C too large"),
    ("c2056", "bwd", dict(c1=2056, groups=8), "gn_bwd: C too large"),
    ("c2056", "apply", dict(c1=2056, groups=8), "gn_apply: C too large"),
    ("groups", "fwd", dict(c1=96, groups=7), "gn_forward: channels must be multiples of 8 and divisible by groups"),
    ("groups", "bwd", dict(c1=96, groups=7), "gn_bwd: bad channels / groups"),
    ("odd-h", "fwd", dict(h=5, resample=1), "gn_forward: bad resample"),
    ("odd-h", "bwd", dict(h=5, resample=1), r"gn_bwd: bad resample / add_mode"),
    ("odd-h-add", "bwd", dict(h=5, add_mode=1), r"gn_bwd: bad resample / add_mode"),
    ("odd-h", "apply", dict(h=5, resample=1), "gn_apply: bad resample"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,op,kw,match", REJECTED, ids=[f"{r[0]}-{r[1]}" for r in REJECTED])
def test_rejected_shape_is_an_error(name, op, kw, match, routes):
    """A shape the kernels do not take is an AdmError: nothing launched, nothing written."""
    lib, _ = _device_ready()
    from adm_b200._lib import AdmError, check
    case = _rejected_case(name, op, kw)
    t, coef, outs = _prepare(lib, case, forward=False)
    before = {k: buf.clone() for k, (buf, _, _) in outs.items()}
    launches = lib.adm_launch_count()
    rc = _call(lib, case, t, outs, coef)()
    torch.cuda.synchronize()
    with pytest.raises(AdmError, match=match):
        check(rc, op)
    assert routes[f"rejected-{name}-{op}"] == [] and lib.adm_launch_count() == launches
    assert lib.adm_device_error() == 0
    for k, (buf, _, _) in outs.items():
        assert torch.equal(_bits(buf), _bits(before[k])), f"{k} was written"


# ------------------------------------------------------------------------------------------------ CPU: the checker's teeth
# Reduced versions of table geometries.  The "kernel" here is a candidate result written into the guarded outputs.
GS9 = Case("gs9", "fwd", 2, 4, 4, 72, 0, 0, "group size 9", groups=8, params=True)
CLUSTER = Case("cluster", "fwd", 12, 6, 10, 64, 0, 8, "K = 8, 8 lanes per vector: CTA r owns pixels 64 j + 8 r + l")
DROP = Case("drop", "fwd", 2, 4, 4, 64, 0, 0, "dropout", params=True, drop=0.1)
DOWN = Case("down", "bwd", 2, 4, 4, 64, 0, 0, "avg-pool, add_mode 1", resample=1, add_mode=1, dbias=2)
NORM1_SMALL = Case("norm1", "bwd", 12, 4, 4, 72, 0, 8, "norm1, group size 9", groups=8, **NORM1)
CONCAT_UP = Case("concat-up", "bwd", 2, 4, 4, 64, 32, 0, "concat, nearest-up", resample=2, add_mode=2, dbias=1)


def _fwd32(case, t):
    """fp32 implementation of the forward chain and its coef (F.group_norm's own statistics)."""
    x = _x(t).to(F32)
    gam, bet, sc, sh = _affine(case, t, F32)
    var, mean = torch.var_mean(x.reshape(case.n, case.g, -1), -1, unbiased=False)
    r = torch.rsqrt(var + case.eps).repeat_interleave(case.cpg, 1)
    m = mean.repeat_interleave(case.cpg, 1)
    coef = torch.stack([r * gam * (1 + sc), (bet - m * r * gam) * (1 + sc) + sh, m, r], -1)
    gn = F.group_norm(x, case.g, gam, bet, case.eps)
    return _post(case, t, torch.addcmul(_e4(sh), gn, _e4(1 + sc))), coef


def _judge(case, t, write, coef=None):
    """Problems of the result that `write(outs)` leaves in fresh guarded outputs."""
    outs = guarded_outputs(case, t, "cpu")
    before = {k: buf.clone() for k, (buf, _, _) in outs.items()}
    write(outs)
    expected = forward_expected(case, t) if case.op == "fwd" else backward_expected(case, t, coef)[0]
    return verify(before, outs, expected)[0]


def _fwd_writer(y, coef):
    def write(outs):
        outs["y"][1].copy_(_nhwc(y))
        outs["coef"][1].copy_(coef)
    return write


def _bwd_writer(case, ref):
    """Writes a candidate {"dx", "dgamma", "dbeta", "dscale", "dshift"} as the kernels would (accumulating)."""
    def write(outs):
        dx = ref["dx"]
        if "dx1" in outs:
            outs["dx1"][1].copy_(_nhwc(dx[:, :case.c1]))
        if "dx2" in outs:
            outs["dx2"][1].copy_(_nhwc(dx[:, case.c1:]))
        outs["dgamma"][1].add_(ref["dgamma"].to(F32))
        outs["dbeta"][1].add_(ref["dbeta"].to(F32))
        if "dparams" in outs:
            outs["dparams"][1].copy_(torch.cat([ref["dscale"], ref["dshift"]], 1))
        for name in ("dbias1", "dbias1b"):
            if name in outs:
                outs[name][1].add_(dx[:, :case.c1].sum((0, 2, 3)).to(F32))
    return write


def _coef64(case, t):
    return forward_expected(case, t)["coef"][0].to(F32)


@pytest.mark.parametrize("case", [GS9, CLUSTER, DROP], ids=lambda c: c.id)
def test_checker_accepts_rounded_reference_and_fp32_forward(case):
    t = operands(case, "cpu")
    ref = forward_expected(case, t)
    assert _judge(case, t, _fwd_writer(_nchw(ref["y"][0]), ref["coef"][0])) == []
    assert _judge(case, t, _fwd_writer(*_fwd32(case, t))) == []


@pytest.mark.parametrize("case", [DOWN, NORM1_SMALL, CONCAT_UP], ids=lambda c: c.id)
def test_checker_accepts_rounded_reference_and_fp32_backward(case):
    t = operands(case, "cpu")
    coef = _coef64(case, t)
    assert _judge(case, t, _bwd_writer(case, backward_reference(case, t, coef)), coef) == []
    assert _judge(case, t, _bwd_writer(case, backward_reference(case, t, coef, dtype=F32)), coef) == []


def _stats_of(case, x, keep=None):
    """Per-(n, c) mean and rstd of each group, over the pixels where `keep` [H * W] is True (all by default); the
    pixel count stays cpg * H * W, as a kernel that loses a chunk would divide by."""
    n, c = case.n, case.c
    xs = x.reshape(n, c, -1)
    if keep is not None:
        xs = xs * keep.to(xs.dtype)
    s = xs.reshape(n, case.g, -1).sum(-1)
    q = (xs * xs).reshape(n, case.g, -1).sum(-1)
    L = case.cpg * case.hw
    mean = s / L
    var = q / L - mean * mean
    return mean.repeat_interleave(case.cpg, 1), ((var + case.eps) ** -0.5).repeat_interleave(case.cpg, 1)


def test_checker_rejects_statistics_grouped_by_channel_vector():
    """Group size 9: each 8-channel vector takes the group of its first channel."""
    c = GS9
    t = operands(c, "cpu")
    mean, rstd = _stats_of(c, _x(t))
    vec_group = torch.arange(c.c) // 8 * 8
    y = forward_reference(c, t, mean_c=mean[:, vec_group], rstd_c=rstd[:, vec_group])
    assert _judge(c, t, _fwd_writer(y, _coef64(c, t)))


def _cta_pixels(case, r):
    """Pixels CTA r of a fused cluster streams: p0 = r * lanes + lane, step = K * lanes."""
    lanes = case.lanes()
    p = torch.arange(case.hw)
    return (p % (case.k * lanes)) // lanes == r


def test_checker_rejects_cluster_missing_one_cta_chunk():
    c = CLUSTER
    t = operands(c, "cpu")
    mean, rstd = _stats_of(c, _x(t), keep=~_cta_pixels(c, c.k - 1))
    y = forward_reference(c, t, mean_c=mean, rstd_c=rstd)
    assert _judge(c, t, _fwd_writer(y, _coef64(c, t)))


def test_checker_rejects_coef_of_previous_sample_on_one_chunk():
    """Sample 5's pixels of CTA 3 normalised with the statistics of sample 4."""
    c = CLUSTER
    t = operands(c, "cpu")
    mean, rstd = _stats_of(c, _x(t))
    y = forward_reference(c, t)
    mean[5], rstd[5] = mean[4], rstd[4]
    y_mut = forward_reference(c, t, mean_c=mean, rstd_c=rstd)
    chunk = _cta_pixels(c, 3).reshape(c.h, c.w)
    y[5][:, chunk] = y_mut[5][:, chunk]
    assert _judge(c, t, _fwd_writer(y, _coef64(c, t)))


def test_checker_rejects_add_mode_1_without_quarter():
    c = DOWN
    t = operands(c, "cpu")
    coef = _coef64(c, t)
    ref = backward_reference(c, t, coef)
    ref["dx"] = ref["dx"] + 3 * _add_adjoint(c, _nchw(t["add"]))
    assert _judge(c, t, _bwd_writer(c, ref), coef)


def test_checker_rejects_dx_missing_mean_g_term_in_one_group():
    """dx = rstd (g - xhat mean(g xhat)) for group 3 of sample 1: the mean(g) term dropped."""
    c = NORM1_SMALL
    t = operands(c, "cpu")
    coef = _coef64(c, t)
    ref = backward_reference(c, t, coef)
    _, extra = backward_expected(c, t, coef, ref)
    gam, _, sc, _ = _affine(c, t)
    gx = extra["dv"] * _e4(gam * (1 + sc))  # gradient at xhat
    m1 = _group_mean(gx, c)
    chans = slice(3 * c.cpg, 4 * c.cpg)
    ref["dx"][1, chans] += (coef[1, chans, 3].to(F64) * m1[1, chans])[:, None, None]
    assert _judge(c, t, _bwd_writer(c, ref), coef)


def test_checker_rejects_mask_with_two_lanes_swapped():
    c = DROP
    t = operands(c, "cpu")
    swapped = _LANE_MUL[[1, 0, 2, 3, 4, 5, 6, 7]]
    t_mut = {**t, "mask": torch.from_numpy(dropout_mask(SEED, COUNTER, c.drop, c.n, c.hw, c.c, swapped)).reshape(
        c.n, c.h, c.w, c.c)}
    assert not torch.equal(t_mut["mask"], t["mask"])
    y = forward_reference(c, t_mut)
    assert _judge(c, t, _fwd_writer(y, _coef64(c, t)))


# ------------------------------------------------------------------------------------------------ CPU: mask and table
def test_dropout_mask_values_and_counter():
    p = 0.1
    m = dropout_mask(SEED, COUNTER, p, 4, 64, 128)
    keep = np.float32(1) / (np.float32(1) - np.float32(p))
    assert set(np.unique(m).tolist()) == {0.0, float(keep)}
    assert np.array_equal(m, dropout_mask(SEED, COUNTER, p, 4, 64, 128))
    assert not np.array_equal(m, dropout_mask(SEED, COUNTER + 1, p, 4, 64, 128))


def test_dropout_mask_per_lane_keep_rate():
    """4 M elements at p = 0.1: every lane keeps 1 - p of its 512 K draws, within 5 binomial standard deviations."""
    p, vectors = 0.1, 1 << 19
    m = dropout_mask(SEED, COUNTER, p, 1, vectors, 8).reshape(vectors, 8)
    rate = (m != 0).mean(0)
    q = 1 - math.floor(np.float32(p) * 2.0 ** 32) / 2.0 ** 32
    sd = math.sqrt(q * (1 - q) / vectors)
    assert np.all(np.abs(rate - q) <= 5 * sd), (rate, q, sd)


def test_cases_cover_every_path():
    for c in CASES:
        if c.op != "apply":
            assert cluster_size(c.n) == c.k, c.id
        if c.drop:
            assert c.resample == 0, c.id  # the only combination callers use (engine.py block_fwd)
    fwd = {c.k for c in CASES if c.op == "fwd"}
    bwd = {c.k for c in CASES if c.op == "bwd"}
    assert fwd == {0, 1, 2, 4, 8} and bwd == {0, 1, 2, 4, 8}
    assert {c.subpath for c in CASES if c.op == "bwd" and c.k} == {"piped", "reuse_dv", "non-piped"}
    assert any(c.op == "apply" for c in CASES)
    assert {(c.op, c.k) for c in CASES if c.drop} >= {("fwd", 0), ("fwd", 1), ("fwd", 2), ("fwd", 8), ("bwd", 0)}
    assert any(c.op == "bwd" and c.drop and c.k and c.subpath == "piped" for c in CASES)
    for n, k in ((11, 0), (12, 8), (22, 8), (23, 4), (44, 4), (45, 2), (88, 2), (89, 1)):
        assert cluster_size(n) == k and any(c.n == n for c in CASES)
    assert len({c.id for c in CASES}) == len(CASES)
