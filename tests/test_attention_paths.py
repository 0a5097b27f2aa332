"""Attention path by path: ops.attention_fwd / ops.attention_bwd at the packing and blocking edges where the fused
tcgen05 kernels (attn_fused.cu) and the unfused batched-GEMM + softmax path (attn_optim.cu) go wrong.  Each row of CASES
names the kernels its shape must be routed to and the edge it exists for; one checker runs every row:

  * path     the CUDA kernels recorded under torch.profiler are exactly the expected list, and adm_launch_count() grows
             by its length.  The units per CTA depend on the SM count: the table is worked out for the 148 SMs of a B200.
  * inputs   qkv, dO, the forward output O, the log-sum-exp and the saved probabilities are views into NaN-filled
             buffers with whole images (a packed tile's worth) before and after them; the blocked kernels get a
             NaN-filled workspace.  A TMA box that reaches past the batch, or a partial buffer that is read but never
             written, turns into NaN in the output.
  * outputs  a, lse and dqkv are written through views of sentinel-filled buffers with the same guard images (for lse:
             guard rows).  Every element outside the view keeps its bits, so do the rows of a partial packed tile that
             lie past the batch.
  * values   every element against an fp64 reference computed from the same bf16 operands and scale: P = softmax(scale
             q k^T), a = P v, lse = log2 sum_k 2^(scale log2(e) s_k) and dQ / dK / dV from autograd.  The bound is written
             through absolute-value shadows (fp64, same operands), A_qd = sum_k P_qk |V_kd| and G_qk = sum_d |dO_qd| |V_kd|,
             and is first order in the unit roundoffs: 2^-8 for bf16 (8 significant bits), 2^-24 for fp32.
             eps_q bounds the relative error of the probabilities of row q as the kernel forms them, before any bf16
             rounding:
                 eps_q = (ceil(d / 16) + 2) 2^-23 max_k scale sum_d |q_d k_d|   the fp32 score (one rounding per 16-deep
                                                                                MMA step, a factor of 2 for its inside)
                       + 2^-20 (1 + max_k |scale s_qk| + ln N)                  ex2.approx (<= 2^-22 relative), and the
                                                                                fp32 scale, c1 = scale log2(e), exponent
                                                                                and row max / lse (each <= 2^-24 of a
                                                                                value <= log2(e) (|s| + ln N)), twice
                                                                                for the blocked merge
                       + (ceil(N / 16) + 2) 2^-23 + N 2^-24                     the fp32 P V and row-sum accumulations
             forward   |a - ref| <= A (r 2^-8 + 2 eps_q) + 2^-8 |ref|
                       r: 1 for the bf16 P before P V, plus 1 for the bf16 partial outputs of the blocked mode.  A relative
                       error e of every P_k moves the normalised output by <= 2 e A; 2^-8 |ref| is the bf16 output.
                       |lse - ref| <= 3 eps_q + 2^-21 (|ref| + 1)   (log2(1 + e) <= 1.5 e; the blocked merge again)
             backward  D_q = sum_d dO_qd O_qd comes from the bf16 O (fused) or, as sum_k P~_qk dP_qk, from the bf16
                       probabilities (unfused): |dD_q| <= dD_q = (2^-8 + e_dp + N 2^-24) sum_d |dO_qd| A_qd, where
                       e_dp = (ceil(d / 16) + 2) 2^-23 bounds the fp32 dP relative to G.  dS is rounded to bf16 before dQ
                       and dK; P carries eps_q (fused: recomputed from the lse) or 2^-8 (unfused: the bf16 saved
                       probabilities); the blocked mode rounds its nblk partial dqkv buffers to bf16:
                 c     = 2^-8 + (eps_q fused | 2^-8 unfused) + 2^-8 [blocked] + (ceil(N / 16) + 2) 2^-23
                 T_qk  = P_qk (dD_q + e_dp G_qk + c |dP_qk - D_q|)
                 |dQ - ref| <= scale T |K| + 2^-8 |ref|,   |dK - ref| <= scale T^T |Q| + 2^-8 |ref|,
                 |dV - ref| <= c P^T |dO| + 2^-8 |ref|
             The constants come from the roundings above, not from errors measured on a GPU.

Every case also has adversarial rows in each (sample, head): query 0 scaled by 10 (logits over about +-30, so the max
subtraction matters), query 1 a multiple of key 3 (a near one-hot row), query 2 zero (all-equal logits); in packed
cases the keys of sample 1 are scaled by 4, so a row that leaks across the packing mask picks up logits far above its
own.

The test_checker_* tests (CPU) show that the checker accepts an fp32 attention and rejects subtly wrong kernels.
"""
import math
from dataclasses import dataclass

import pytest
import torch

from tests.test_conv_paths import _bits, _device_ready, _kernels_of

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
SENTINEL = 1000.0
LOG2E = 1.4426950408889634

# kernel names as torch.profiler reports them on the B200 (without "void adm::" and the parameter list)
FWD = "attn_fwd_kernel"
BWD = "attn_bwd_kernel"
COMBINE = "attn_combine_kernel"
REDUCE = "attn_reduce_kernel"
GEMM = "tc_gemm_kernel<0>"
SOFTMAX = "softmax_fwd_kernel"
SOFTMAX_LONG = "softmax_fwd_long_kernel"
SOFTMAX_BWD = "softmax_bwd_kernel"
# expected launch lists: fused, blocked, unfused (QK^T, softmax, PV / dV, dP, softmax backward, dQ, dK)
PATHS = {
    ("fwd", "fused"): [FWD], ("fwd", "blocked"): [FWD, COMBINE], ("fwd", "unfused"): [GEMM, SOFTMAX, GEMM],
    ("fwd", "unfused-long"): [GEMM, SOFTMAX_LONG, GEMM],
    ("bwd", "fused"): [BWD], ("bwd", "blocked"): [BWD, REDUCE], ("bwd", "unfused"): [GEMM, GEMM, SOFTMAX_BWD, GEMM, GEMM],
}


@dataclass(frozen=True)
class Case:
    name: str
    op: str  # "fwd" or "bwd"
    n: int
    h: int
    w: int
    heads: int
    dpad: int  # head width as stored in qkv (zero-padded)
    d: int  # true head width: the scale is d^-0.5
    path: str  # key of PATHS
    edge: str

    @property
    def id(self):
        return f"{self.name}-{self.op}"

    @property
    def npix(self):
        return self.h * self.w

    @property
    def c(self):
        return self.heads * self.dpad

    @property
    def scale(self):
        return self.d ** -0.5

    @property
    def kernels(self):
        return PATHS[(self.op, self.path)]

    @property
    def pack(self):
        """Samples per 128-row tile of the fused kernels (1 elsewhere)."""
        return 128 // self.npix if self.path == "fused" and self.npix < 256 else 1

    @property
    def guard(self):
        """Guard / poison images on either side of every view: one packed tile."""
        return self.pack

    @property
    def blocked(self):
        return self.path == "blocked"


def _rows(name, n, h, w, heads, dpad, d, path, edge, ops=("fwd", "bwd")):
    return [Case(name, op, n, h, w, heads, dpad, d, path, edge) for op in ops]


CASES = [
    *_rows("pack8-partial", 13, 4, 4, 2, 64, 64, "fused", "N = 16, 8 samples per tile: 13 leaves the last tile 5/8 full"),
    *_rows("pack8-ring", 1589, 4, 4, 6, 64, 64, "fused",
           "1194 units on 148 CTAs: 8-9 units each, the operand ring wraps its parity more than once; partial tile"),
    *_rows("pack2-odd", 127, 8, 8, 6, 64, 64, "fused", "N = 64, 2 samples per tile, odd batch (CIFAR 8x8 level)"),
    *_rows("cifar-16x16", 128, 16, 16, 6, 64, 64, "fused",
           "N = 256, two query tiles per unit: the CIFAR benchmark's 16x16 attention (C = 384, batch 128)"),
    *_rows("blk-512", 3, 16, 32, 2, 64, 64, "blocked", "blocked, nblk = 2"),
    *_rows("blk-768", 5, 24, 32, 1, 64, 64, "blocked", "blocked, nblk = 3 (odd)"),
    *_rows("blk-1024-celebahq", 48, 32, 32, 3, 64, 64, "blocked",
           "CelebAHQ-latent 32x32 level (C = 192, batch 48): 2304 units, the last wave 84 of 148"),
    *_rows("blk-4096", 1, 64, 64, 2, 64, 64, "blocked", "blocked, nblk = 16: 512 units, the last wave 68 of 148"),
    *_rows("pad32-cond", 5, 8, 8, 4, 64, 32, "fused",
           "cond UNet heads: d = 32 stored as 64, scale 32^-0.5, packed with a partial tile"),
    *_rows("pad72-celebahq-16x16", 48, 16, 16, 4, 128, 72, "unfused",
           "CelebAHQ-latent 16x16 level (C = 288, 4 heads of 72 stored as 128, scale 72^-0.5, batch 48)"),
    *_rows("pad72-1024", 2, 32, 32, 4, 128, 72, "unfused", "d = 72 stored as 128 at N = 1024: the one-warp softmax's "
           "longest row"),
    *_rows("ae-mid", 1, 64, 64, 1, 512, 512, "unfused-long",
           "autoencoder mid attention: 1 head, d = 512, 4096 tokens (encoder_decoder.py AttnBlock)", ops=("fwd",)),
]


# ------------------------------------------------------------------------------------------------ operands and reference
def _to_layout(t):
    """[n, heads, N, dpad] -> [n, N, heads * dpad] (the NHWC channel layout of one of q / k / v)."""
    n, hh, npix, dp = t.shape
    return t.permute(0, 2, 1, 3).reshape(n, npix, hh * dp)


def _from_layout(t, heads):
    n, npix, c = t.shape
    return t.reshape(n, npix, heads, c // heads).permute(0, 2, 1, 3)


def poisoned(t, before, after):
    """t as a contiguous view into a NaN-filled buffer with `before` / `after` slabs of its leading dim around it."""
    buf = torch.full((before + t.shape[0] + after, *t.shape[1:]), float("nan"), dtype=t.dtype, device=t.device)
    view = buf[before:before + t.shape[0]]
    view.copy_(t)
    return view


def operands(case, device, seed=0):
    """q, k, v, dO as bf16 [n, heads, N, dpad] (zero past the true head width) with the adversarial rows of the module
    docstring, and qkv / dO in the kernels' layout, each inside its poisoned buffer."""
    c = case
    g = torch.Generator(device=device).manual_seed(seed)
    shape = (c.n, c.heads, c.npix, c.dpad)
    q, k, v, do = (torch.randn(*shape, generator=g, device=device) for _ in range(4))
    for x in (q, k, v, do):
        x[..., c.d:] = 0
    q[:, :, 0] *= 10
    q[:, :, 1] = k[:, :, 3] * (24 / c.d ** 0.5)
    q[:, :, 2] = 0
    if c.pack > 1 and c.n > 1:
        k[1] *= 4
    q, k, v, do = (x.to(BF16) for x in (q, k, v, do))
    qkv = torch.cat([_to_layout(q), _to_layout(k), _to_layout(v)], -1).reshape(c.n, c.h, c.w, 3 * c.c)
    return {"q": q, "k": k, "v": v, "do": do, "qkv": poisoned(qkv, c.guard, c.guard),
            "do_nhwc": poisoned(_to_layout(do).reshape(c.n, c.h, c.w, c.c), c.guard, c.guard)}


def forward_reference(case, t, scale=None, dtype=F64):
    """(P, O, lse [log2 units], s) in [n, heads, N, .] computed in `dtype` from the case's operands."""
    scale = case.scale if scale is None else scale
    q, k, v = (t[x].to(dtype) for x in "qkv")
    s = scale * q @ k.transpose(-1, -2)
    p = torch.softmax(s, -1)
    return p, p @ v, torch.logsumexp(s, -1) * LOG2E, s


def eps_rows(case, t, s):
    """eps_q of the module docstring, [n, heads, N]."""
    c = case
    q, k = t["q"].to(F64), t["k"].to(F64)
    sabs = c.scale * q.abs() @ k.abs().transpose(-1, -2)
    return ((math.ceil(c.dpad / 16) + 2) * 2.0 ** -23 * sabs.amax(-1)
            + 2.0 ** -20 * (1 + s.abs().amax(-1) + math.log(c.npix))
            + (math.ceil(c.npix / 16) + 2) * 2.0 ** -23 + c.npix * 2.0 ** -24)


def fwd_expected(case, t):
    """{output: (ref, bound)} in the kernels' layouts: a [n, H, W, C] and (fused / blocked) lse [n, heads, N]."""
    c = case
    p, o, lse, s = forward_reference(c, t)
    eps = eps_rows(c, t, s)
    shadow = p @ t["v"].to(F64).abs()
    r = 2 if c.blocked else 1
    bound = shadow * (r * 2.0 ** -8 + 2 * eps[..., None]) + 2.0 ** -8 * o.abs()
    nhwc = lambda x: _to_layout(x).reshape(c.n, c.h, c.w, c.c)
    out = {"a": (nhwc(o), nhwc(bound))}
    if c.path in ("fused", "blocked"):
        out["lse"] = (lse, 3 * eps + 2.0 ** -21 * (lse.abs() + 1))
    return out


def bwd_inputs(case, t):
    """What the backward reads besides qkv and dO: the forward output (fp64 reference rounded to bf16) and, fused, the
    log-sum-exp (fp32) or, unfused, the probabilities (bf16), each inside its poisoned buffer."""
    c = case
    p, o, lse, _ = forward_reference(c, t)
    a = poisoned(_to_layout(o).reshape(c.n, c.h, c.w, c.c).to(BF16), c.guard, c.guard)
    if c.path == "unfused":
        aux = poisoned(p.reshape(c.n * c.heads, c.npix, c.npix).to(BF16), c.guard * c.heads, c.guard * c.heads)
    else:
        aux = poisoned(lse.to(F32), c.guard, c.guard)
    return a, aux


def backward_reference(case, t, dtype=F64, scale=None):
    """(dq, dk, dv) [n, heads, N, dpad] by autograd in `dtype`."""
    scale = case.scale if scale is None else scale
    q, k, v = (t[x].to(dtype).requires_grad_(True) for x in "qkv")
    o = torch.softmax(scale * q @ k.transpose(-1, -2), -1) @ v
    return torch.autograd.grad(o, (q, k, v), t["do"].to(dtype))


def bwd_expected(case, t):
    """{"dqkv": (ref, bound)} in the kernels' layout [n, H, W, 3C]."""
    c = case
    p, o, _, s = forward_reference(c, t)
    q, k, v, do = (t[x].to(F64) for x in ("q", "k", "v", "do"))
    eps = eps_rows(c, t, s)
    dq, dk, dv = backward_reference(c, t)
    dp = do @ v.transpose(-1, -2)
    dd = (do * o).sum(-1, keepdim=True)
    g = do.abs() @ v.abs().transpose(-1, -2)
    e_dp = (math.ceil(c.dpad / 16) + 2) * 2.0 ** -23
    d_err = (2.0 ** -8 + e_dp + c.npix * 2.0 ** -24) * (do.abs() * (p @ v.abs())).sum(-1, keepdim=True)
    eps_p = 2.0 ** -8 if c.path == "unfused" else eps[..., None]
    coef = 2.0 ** -8 + eps_p + (2.0 ** -8 if c.blocked else 0.0) + (math.ceil(c.npix / 16) + 2) * 2.0 ** -23
    tt = p * (d_err + e_dp * g + coef * (dp - dd).abs())
    bq = c.scale * tt @ k.abs() + 2.0 ** -8 * dq.abs()
    bk = c.scale * tt.transpose(-1, -2) @ q.abs() + 2.0 ** -8 * dk.abs()
    bv = coef * p.transpose(-1, -2) @ do.abs() + 2.0 ** -8 * dv.abs()
    nhwc = lambda a, b_, c_: torch.cat([_to_layout(a), _to_layout(b_), _to_layout(c_)], -1).reshape(
        c.n, c.h, c.w, 3 * c.c)
    return {"dqkv": (nhwc(dq, dk, dv), nhwc(bq, bk, bv))}


# ------------------------------------------------------------------------------------------------ guarded outputs, checker
def guarded_outputs(case, device):
    """{output: (buf, view)}: each output view inside a sentinel-filled buffer with case.guard images (lse: guard rows)
    on either side."""
    c, gd = case, case.guard

    def guarded(*shape, dtype):
        buf = torch.full((gd + shape[0] + gd, *shape[1:]), SENTINEL, dtype=dtype, device=device)
        return buf, buf[gd:gd + shape[0]]

    if c.op == "bwd":
        return {"dqkv": guarded(c.n, c.h, c.w, 3 * c.c, dtype=BF16)}
    out = {"a": guarded(c.n, c.h, c.w, c.c, dtype=BF16)}
    if c.path in ("fused", "blocked"):
        out["lse"] = guarded(c.n, c.heads, c.npix, dtype=F32)
    return out


def verify(case, before, outs, expected):
    """Problems (strings) of one result, and the largest |got - ref| / bound per output.  `before`: the buffers'
    contents before the call; `outs`: {output: (buf, view)}; `expected`: {output: (ref, bound)}."""
    problems, worst = [], {}
    for name, (buf, view) in outs.items():
        gd = case.guard
        stray = _bits(before[name]) != _bits(buf)
        stray[gd:gd + case.n] = False
        if stray.any():
            idx = stray.nonzero()[:4].tolist()
            problems.append(f"{name}: {int(stray.sum())} elements outside the output changed, e.g. at {idx}")
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
def _workspace(lib, case):
    """NaN-filled (all bits set) scratch for the blocked kernels, or None."""
    if not case.blocked:
        return None
    nbytes = lib.adm_attn_long_workspace(case.n, case.npix, case.heads, int(case.op == "bwd"))
    return torch.full((nbytes,), 255, dtype=torch.uint8, device="cuda")


def _call(case, t, ops, outs, work, bwd_in=None):
    c = case
    if c.op == "fwd":
        lse = outs["lse"][1] if "lse" in outs else None
        return lambda: ops.attention_fwd(t["qkv"], c.heads, scale=c.scale, out=outs["a"][1], lse=lse, work=work)
    a, aux = bwd_in
    return lambda: ops.attention_bwd(t["do_nhwc"], t["qkv"], aux, c.heads, scale=c.scale, a=a, out=outs["dqkv"][1],
                                     work=work)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_attention_path(case):
    lib, ops = _device_ready()
    t = operands(case, "cuda")
    bwd_in = bwd_inputs(case, t) if case.op == "bwd" else None
    outs = guarded_outputs(case, "cuda")
    before = {k: buf.clone() for k, (buf, _) in outs.items()}
    work = _workspace(lib, case)
    launches = lib.adm_launch_count()
    ran = _kernels_of(_call(case, t, ops, outs, work, bwd_in))
    assert ran == case.kernels, f"{case.id} ({case.edge}) ran {ran}, expected {case.kernels}"
    assert lib.adm_launch_count() == launches + len(case.kernels)
    assert lib.adm_device_error() == 0
    expected = fwd_expected(case, t) if case.op == "fwd" else bwd_expected(case, t)
    problems, worst = verify(case, before, outs, expected)
    print(f"{case.id}: {ran}, max |err| / bound = " + ", ".join(f"{k} {v:.3g}" for k, v in worst.items()))
    assert not problems, f"{case.id} ({case.edge}): " + "; ".join(problems)


# shapes the kernels reject: (case, forced routing, message)
REJECTED = [
    (Case("fused-n32", "fwd", 2, 4, 8, 2, 64, 64, "fused", "32 pixels: not a fused tile"), True,
     r"n_pix must be 16, 64 or 256 \(got 32\)"),
    (Case("fused-n32", "bwd", 2, 4, 8, 2, 64, 64, "fused", "32 pixels: not a fused tile"), True,
     r"n_pix must be 16, 64 or 256 \(got 32\)"),
    (Case("blk-640", "fwd", 1, 20, 32, 2, 64, 64, "blocked", "640 pixels: not whole 256-pixel blocks"), True,
     r"n_pix must be a multiple of 256 in \[512, 4096\] \(got 640\)"),
    (Case("blk-640", "bwd", 1, 20, 32, 2, 64, 64, "blocked", "640 pixels: not whole 256-pixel blocks"), True,
     r"n_pix must be a multiple of 256 in \[512, 4096\] \(got 640\)"),
    (Case("unfused-4096", "bwd", 1, 64, 64, 1, 128, 72, "unfused", "rows of 4096 keys: past the softmax backward"),
     False, r"at most 1024 keys \(got 4096\)"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case,fused,match", REJECTED, ids=[c.id for c, _, _ in REJECTED])
def test_unsupported_shape_is_an_error(case, fused, match):
    """A shape the routed kernels do not take is an AdmError before anything is launched or written."""
    lib, ops = _device_ready()
    from adm_b200._lib import AdmError
    t = operands(case, "cuda")
    outs = guarded_outputs(case, "cuda")
    if case.op == "bwd":
        # inputs of the right shapes: the forward output and the lse (fused) or the probabilities (unfused)
        a = poisoned(torch.zeros(case.n, case.h, case.w, case.c, dtype=BF16, device="cuda"), 1, 1)
        aux = (poisoned(torch.zeros(case.n * case.heads, case.npix, case.npix, dtype=BF16, device="cuda"), 1, 1)
               if not fused else poisoned(torch.zeros(case.n, case.heads, case.npix, device="cuda"), 1, 1))
    before = {k: buf.clone() for k, (buf, _) in outs.items()}
    work = torch.full((1 << 20,), 255, dtype=torch.uint8, device="cuda")
    launches = lib.adm_launch_count()

    def attempt():
        with pytest.raises(AdmError, match=match):
            if case.op == "fwd":
                ops.attention_fwd(t["qkv"], case.heads, scale=case.scale, fused=fused, out=outs["a"][1],
                                  lse=outs["lse"][1], work=work)
            else:
                ops.attention_bwd(t["do_nhwc"], t["qkv"], aux, case.heads, scale=case.scale, fused=fused, a=a,
                                  out=outs["dqkv"][1], work=work)

    assert _kernels_of(attempt) == [] and lib.adm_launch_count() == launches
    assert lib.adm_device_error() == 0
    for k, (buf, _) in outs.items():
        assert torch.equal(_bits(buf), _bits(before[k])), f"{k} was written"


# ------------------------------------------------------------------------------------------------ CPU: the checker's teeth
# Reduced versions of table geometries.  The "kernel" here is a candidate result written into the guarded outputs.
PACKED = Case("packed", "fwd", 3, 4, 4, 2, 64, 64, "fused", "8 samples per tile, partial")
BLOCKED = Case("blocked", "fwd", 1, 16, 32, 1, 64, 64, "blocked", "nblk = 2")
PADDED = Case("padded", "fwd", 2, 8, 8, 2, 128, 72, "unfused", "d = 72 stored as 128")
PACKED_BWD = Case("packed", "bwd", 3, 8, 8, 2, 64, 64, "fused", "2 samples per tile, partial")
PADDED_BWD = Case("padded", "bwd", 2, 8, 8, 2, 128, 72, "unfused", "d = 72 stored as 128")


def _judge(case, t, write):
    """Problems of the result that `write(outs)` leaves in fresh guarded outputs."""
    outs = guarded_outputs(case, "cpu")
    before = {k: buf.clone() for k, (buf, _) in outs.items()}
    write(outs)
    expected = fwd_expected(case, t) if case.op == "fwd" else bwd_expected(case, t)
    return verify(case, before, outs, expected)[0]


def _fwd_writer(case, o, lse):
    """Writes a candidate O [n, heads, N, dpad] and lse [n, heads, N] into the outputs (lse where the path has one)."""
    def write(outs):
        outs["a"][1].copy_(_to_layout(o).reshape(case.n, case.h, case.w, case.c))
        if "lse" in outs:
            outs["lse"][1].copy_(lse)
    return write


def _bwd_writer(case, dq, dk, dv):
    def write(outs):
        outs["dqkv"][1].copy_(torch.cat([_to_layout(dq), _to_layout(dk), _to_layout(dv)], -1).reshape(
            case.n, case.h, case.w, 3 * case.c))
    return write


@pytest.mark.parametrize("case", [PACKED, BLOCKED, PADDED, PACKED_BWD, PADDED_BWD], ids=lambda c: c.id)
def test_checker_accepts_rounded_reference_and_fp32_attention(case):
    t = operands(case, "cpu")
    for dtype in (F64, F32):  # fp32: another summation order and fp32 exponentials of the same operands
        if case.op == "fwd":
            _, o, lse, _ = forward_reference(case, t, dtype=dtype)
            assert _judge(case, t, _fwd_writer(case, o, lse)) == [], dtype
        else:
            assert _judge(case, t, _bwd_writer(case, *backward_reference(case, t, dtype=dtype))) == [], dtype


def test_checker_rejects_packing_mask_leak():
    """Query 5 of sample 0 also sees the keys of sample 1, its neighbour in the packed tile."""
    c = PACKED
    t = operands(c, "cpu")
    _, o, lse, _ = forward_reference(c, t)
    q, k, v = (t[x].to(F64) for x in "qkv")
    keys, vals = torch.cat([k[0], k[1]], -2), torch.cat([v[0], v[1]], -2)
    s = c.scale * q[0, :, 5:6] @ keys.transpose(-1, -2)
    o[0, :, 5:6] = torch.softmax(s, -1) @ vals
    lse[0, :, 5:6] = torch.logsumexp(s, -1) * LOG2E
    assert _judge(c, t, _fwd_writer(c, o, lse))


def test_checker_rejects_missing_last_image_of_partial_tile():
    c = PACKED
    t = operands(c, "cpu")
    _, o, lse, _ = forward_reference(c, t)

    def write(outs):
        outs["a"][1][:-1].copy_(_to_layout(o[:-1]).reshape(c.n - 1, c.h, c.w, c.c))
        outs["lse"][1][:-1].copy_(lse[:-1])

    assert _judge(c, t, write)


def _block_partials(case, t):
    """Per 256-key block: the block-normalised O_kb and the block's lse (log2 units), as the blocked forward emits."""
    q, k, v = (t[x].to(F64) for x in "qkv")
    parts = []
    for kb in range(case.npix // 256):
        sl = slice(kb * 256, (kb + 1) * 256)
        s = case.scale * q @ k[..., sl, :].transpose(-1, -2)
        parts.append((torch.softmax(s, -1) @ v[..., sl, :], torch.logsumexp(s, -1) * LOG2E))
    return parts


def test_checker_rejects_combine_dropping_a_key_block():
    c = BLOCKED
    t = operands(c, "cpu")
    _, _, lse, _ = forward_reference(c, t)
    o0, _ = _block_partials(c, t)[0]  # the merge of block 0 alone
    assert _judge(c, t, _fwd_writer(c, o0, lse))


def test_checker_rejects_combine_weighted_by_natural_log_lse():
    """The partial lse in natural-log units fed to the base-2 merge: w_kb = 2^(ln2 L_kb - m) / sum."""
    c = BLOCKED
    t = operands(c, "cpu")
    _, _, lse, _ = forward_reference(c, t)
    parts = _block_partials(c, t)
    ls = torch.stack([l_ for _, l_ in parts]) * math.log(2)
    w = torch.softmax(ls * math.log(2), 0)  # 2^(l_kb - m) normalised
    o = sum(w[i][..., None] * parts[i][0] for i in range(len(parts)))
    assert _judge(c, t, _fwd_writer(c, o, lse))


def test_checker_rejects_lse_in_natural_log():
    c = PACKED
    t = operands(c, "cpu")
    _, o, lse, _ = forward_reference(c, t)
    assert _judge(c, t, _fwd_writer(c, o, lse * math.log(2)))


def test_checker_rejects_padded_head_scaled_by_stored_width():
    c = PADDED
    t = operands(c, "cpu")
    _, o, lse, _ = forward_reference(c, t, scale=c.dpad ** -0.5)
    assert _judge(c, t, _fwd_writer(c, o, lse))


def test_checker_rejects_dk_of_one_head_written_to_the_next():
    c = PACKED_BWD
    t = operands(c, "cpu")
    dq, dk, dv = backward_reference(c, t)
    dk = dk.clone()
    dk[:, 1] = dk[:, 0]
    assert _judge(c, t, _bwd_writer(c, dq, dk, dv))


def test_checker_rejects_write_one_column_past_the_view():
    c = PACKED
    t = operands(c, "cpu")
    _, o, lse, _ = forward_reference(c, t)

    def write(outs):
        _fwd_writer(c, o, lse)(outs)
        buf, view = outs["a"]
        buf[c.guard + c.n, 0, 0, 0] = view[-1, -1, -1, -1]  # the element after the view's last one

    assert _judge(c, t, write)


def test_cases_cover_every_kernel_of_every_direction():
    reached = {(c.op, k) for c in CASES for k in c.kernels}
    assert reached == {("fwd", k) for k in (FWD, COMBINE, GEMM, SOFTMAX, SOFTMAX_LONG)} | \
        {("bwd", k) for k in (BWD, REDUCE, GEMM, SOFTMAX_BWD)}
    assert {(c.op, c.path) for c in CASES} == set(PATHS)
    assert len({c.id for c in CASES}) == len(CASES)
