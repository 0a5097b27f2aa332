"""Tensor-level wrappers around the C-ABI kernels.  torch is used for device memory and streams only.

Conventions: activations are NHWC bf16 tensors of shape [N, H, W, C] whose last dim is contiguous and whose pixel
stride ``ld = x.stride(2)`` may exceed C (channel-slice views).  Every function enqueues on torch's current stream.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import GemmDesc, Operand, check

BF16 = torch.bfloat16
F32 = torch.float32


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("adm_b200 kernels need CUDA tensors (there is no CPU fallback)")


def _ptr(t):
    return None if t is None else t.data_ptr()


def pad64(c: int) -> int:
    return (c + 63) // 64 * 64


def _nhwc(x):
    """(ptr, C, ld, N, H, W) of an NHWC bf16 view."""
    assert x.dim() == 4 and x.dtype == BF16 and x.stride(3) == 1, (x.shape, x.dtype, x.stride())
    n, h, w, c = x.shape
    ld = x.stride(2)
    assert x.stride(1) == ld * w and x.stride(0) == ld * w * h, "NHWC view must be dense over pixels"
    return x.data_ptr(), c, ld, n, h, w


# ------------------------------------------------------------------------------------------------ DDM elementwise
def qsample(x0, noise, t):
    _need_cuda(x0, noise, t)
    x0, noise, t = x0.contiguous(), noise.contiguous(), t.contiguous().float()
    out = torch.empty_like(x0)
    b = x0.shape[0]
    check(_lib.load().adm_qsample(_ptr(x0), _ptr(noise), _ptr(t), _ptr(out), b, x0.numel() // b, _stream()), "qsample")
    return out


def ddm_loss(c_pred, eps_pred, x0, noise, t, eps, weighting, use_l1=False, grad_scale=1.0, need_grad=True):
    """Returns (loss_per_sample [B], dC_pred, dEps_pred); grads are d(mean_b loss_b * grad_scale)."""
    _need_cuda(c_pred, eps_pred, x0, noise, t)
    c_pred, eps_pred, x0, noise = (a.contiguous() for a in (c_pred, eps_pred, x0, noise))
    b = x0.shape[0]
    flags = int(use_l1) if not isinstance(use_l1, bool) else int(use_l1)  # bool -> 1 (mean |.|); ints are flag words
    loss = torch.empty(b * (2 if flags & 4 else 1), device=x0.device, dtype=F32)
    dc = torch.empty_like(c_pred) if need_grad else None
    de = torch.empty_like(eps_pred) if need_grad else None
    check(_lib.load().adm_ddm_loss(_ptr(c_pred), _ptr(eps_pred), _ptr(x0), _ptr(noise), _ptr(t.contiguous().float()),
                                   float(eps), int(bool(weighting)), flags, float(grad_scale), _ptr(loss),
                                   _ptr(dc), _ptr(de), b, x0.numel() // b, _stream()), "ddm_loss")
    return loss, dc, de


def sampler_step(x, c_pred, eps_pred, t_cur, t_next, clip=1.0, do_clip=True, last=False, scale_input=1.0):
    _need_cuda(x, c_pred, eps_pred)
    assert x.dtype in (torch.float64, torch.float32)
    x = x.contiguous()
    out = torch.empty_like(x)
    check(_lib.load().adm_sampler_step(_ptr(x), _ptr(c_pred.contiguous()), _ptr(eps_pred.contiguous()), _ptr(out),
                                       float(t_cur), float(t_next), float(clip), int(do_clip), int(last),
                                       float(scale_input), int(x.dtype == torch.float64), x.numel(), _stream()),
          "sampler_step")
    return out


def sampler_step_stochastic(x, c_pred, eps_pred, z, t_cur, s, clip=1.0, do_clip=True):
    _need_cuda(x, c_pred, eps_pred, z)
    x = x.contiguous().float()
    out = torch.empty_like(x)
    check(_lib.load().adm_sampler_step_stochastic(_ptr(x), _ptr(c_pred.contiguous()), _ptr(eps_pred.contiguous()),
                                                  _ptr(z.contiguous().float()), _ptr(out), float(t_cur), float(s),
                                                  float(clip), int(do_clip), x.numel(), _stream()),
          "sampler_step_stochastic")
    return out


# ------------------------------------------------------------------------------------------------ EDM edges
def unet_input(x_nchw, sigma, ld_out=8):
    _need_cuda(x_nchw, sigma)
    n, c, h, w = x_nchw.shape
    out = torch.empty(n, h, w, ld_out, device=x_nchw.device, dtype=BF16)
    sigma = sigma.reshape(-1).float().contiguous()
    check(_lib.load().adm_unet_input(_ptr(x_nchw.contiguous().float()), _ptr(sigma), int(sigma.numel() == 1),
                                     _ptr(out), n, c, h, w, ld_out, _stream()), "unet_input")
    return out


def unet_output(f1, f2, x_nchw, sigma):
    """f1, f2: fp32 NHWC [N,H,W,ldf]; returns (D1, D2) NCHW fp32."""
    n, c, h, w = x_nchw.shape
    ldf = f1.shape[-1]
    d1 = torch.empty(n, c, h, w, device=x_nchw.device, dtype=F32)
    d2 = torch.empty_like(d1)
    sigma = sigma.reshape(-1).float().contiguous()
    check(_lib.load().adm_unet_output(_ptr(f1), _ptr(f2), ldf, _ptr(x_nchw.contiguous().float()), _ptr(sigma),
                                      int(sigma.numel() == 1), _ptr(d1), _ptr(d2), n, c, h, w, _stream()),
          "unet_output")
    return d1, d2


def unet_output_bwd(dd1, dd2, sigma, ld_out=8):
    n, c, h, w = dd1.shape
    df1 = torch.empty(n, h, w, ld_out, device=dd1.device, dtype=BF16)
    df2 = torch.empty_like(df1)
    sigma = sigma.reshape(-1).float().contiguous()
    if sigma.numel() == 1:
        sigma = sigma.expand(n).contiguous()
    check(_lib.load().adm_unet_output_bwd(_ptr(dd1.contiguous()), _ptr(dd2.contiguous()), _ptr(sigma), _ptr(df1),
                                          _ptr(df2), n, c, h, w, ld_out, _stream()), "unet_output_bwd")
    return df1, df2


# ------------------------------------------------------------------------------------------------ GEMM engine
def pack_conv_weight(w, c1=None, c2=0, row_perm=None, out=None):
    """fp32 [cout, c1+c2, k, k] -> bf16 [cout, k*k, pad64(c1)+pad64(c2)]."""
    _need_cuda(w)
    cout, cin, k, _ = w.shape
    c1 = cin if c1 is None else c1
    assert c1 + c2 == cin
    kpad = pad64(c1) + (pad64(c2) if c2 else 0)
    if out is None:
        out = torch.empty(cout, k * k, kpad, device=w.device, dtype=BF16)
    assert w.is_contiguous() and w.dtype == F32
    check(_lib.load().adm_pack_conv_weight(_ptr(w), _ptr(out), cout, c1, c2, k, _ptr(row_perm), _stream()),
          "pack_conv_weight")
    return out


def unpack_conv_wgrad(dw_packed, c1, c2, k, out=None, accumulate=False, row_perm=None):
    cout = dw_packed.shape[0]
    if out is None:
        out = torch.empty(cout, c1 + c2, k, k, device=dw_packed.device, dtype=F32)
        accumulate = False
    check(_lib.load().adm_unpack_conv_wgrad(_ptr(dw_packed), _ptr(out), cout, c1, c2, k, int(accumulate),
                                            _ptr(row_perm), _stream()), "unpack_conv_wgrad")
    return out


def cast_bf16(x):
    _need_cuda(x)
    x = x.contiguous().float()
    out = torch.empty(x.shape, device=x.device, dtype=BF16)
    check(_lib.load().adm_cast_f32_bf16(_ptr(x), _ptr(out), x.numel(), _stream()), "cast_f32_bf16")
    return out


def cast_bf16_into(src, dst):
    """dst (bf16, contiguous) <- src (fp32, contiguous), same numel."""
    assert src.is_contiguous() and dst.is_contiguous() and src.numel() == dst.numel()
    check(_lib.load().adm_cast_f32_bf16(_ptr(src), _ptr(dst), src.numel(), _stream()), "cast_f32_bf16")
    return dst


def weight_transpose_tiles(offset, cout, ntaps, cin):
    """Tile table (host int64 [tiles, 4]) of adm_transpose_weight_tiles for ONE conv whose packed bf16 weights
    [cout][ntaps][cin] start `offset` elements into the source buffer; the transposed, tap-mirrored copy
    [cin][ntaps][cout] goes to the same offset of the destination buffer.  cout, cin multiples of 64."""
    assert cout % 64 == 0 and cin % 64 == 0
    cot, t, cit = torch.meshgrid(torch.arange(cout // 64), torch.arange(ntaps), torch.arange(cin // 64), indexing="ij")
    src = offset + (cot * 64 * ntaps + t) * cin + cit * 64
    dst = offset + (cit * 64 * ntaps + (ntaps - 1 - t)) * cout + cot * 64
    return torch.stack([src, dst, torch.full_like(src, ntaps * cin), torch.full_like(src, ntaps * cout)],
                       dim=-1).reshape(-1, 4).to(torch.int64)


def transpose_weight_tiles(src, dst, tiles):
    """dst <- per-conv transposed / tap-mirrored copy of the packed bf16 weights in src (see weight_transpose_tiles)."""
    _need_cuda(src, dst, tiles)
    assert src.dtype == BF16 and dst.dtype == BF16 and tiles.dtype == torch.int64 and tiles.is_contiguous()
    check(_lib.load().adm_transpose_weight_tiles(_ptr(src), _ptr(dst), _ptr(tiles), tiles.shape[0], _stream()),
          "transpose_weight_tiles")
    return dst


def conv_fprop(x1, wpk, x2=None, bias=None, residual=None, alpha=1.0, out_dtype=BF16, out=None, nout=None,
               keep_pad=False):
    """Implicit-GEMM conv (3x3 pad 1 or 1x1) on NHWC bf16.  wpk: [nout, taps, kpad] bf16."""
    _need_cuda(x1, wpk)
    p1, c1, ld1, n, h, w = _nhwc(x1)
    p2, c2, ld2 = None, 0, 0
    if x2 is not None:
        p2, c2, ld2, n2, h2, w2 = _nhwc(x2)
        assert (n2, h2, w2) == (n, h, w)
    nout_w, ntaps, kpad = wpk.shape
    nout = nout_w if nout is None else nout
    assert kpad == pad64(c1) + (pad64(c2) if x2 is not None else 0), (kpad, c1, c2)
    if out is None:
        ldc = (nout + 7) // 8 * 8 if out_dtype == BF16 else (nout + 3) // 4 * 4
        out = torch.empty(n, h, w, ldc, device=x1.device, dtype=out_dtype)
        if ldc != nout:
            out.zero_()
    ldc = out.stride(2)
    ldr = 0
    if residual is not None:
        assert residual.dtype == BF16 and residual.stride(3) == 1
        ldr = residual.stride(2)
    check(_lib.load().adm_conv_fprop(p1, c1, ld1, p2, c2, ld2, n, h, w, _ptr(wpk), nout, ntaps, _ptr(out),
                                     0 if out.dtype == BF16 else 1, ldc, _ptr(bias), _ptr(residual), ldr, float(alpha),
                                     _stream()), "conv_fprop")
    return out[..., :nout] if (out.shape[-1] != nout and not keep_pad) else out


def conv_dgrad(dy, wpk, n_valid=None, residual=None, alpha=1.0, out=None):
    """dx = conv^T(dy) using the fprop-packed weights.  Returns NHWC bf16 [N,H,W,n_valid]."""
    _need_cuda(dy, wpk)
    pd, cout, ldd, n, h, w = _nhwc(dy)
    nout_w, ntaps, kpad = wpk.shape
    assert cout <= nout_w
    n_valid = kpad if n_valid is None else n_valid
    if out is None:
        out = torch.empty(n, h, w, (n_valid + 7) // 8 * 8, device=dy.device, dtype=BF16)
    ldr = residual.stride(2) if residual is not None else 0
    check(_lib.load().adm_conv_dgrad(pd, cout, ldd, n, h, w, _ptr(wpk), kpad, ntaps, _ptr(out), n_valid,
                                     out.stride(2), _ptr(residual), ldr, float(alpha), _stream()), "conv_dgrad")
    return out[..., :n_valid] if out.shape[-1] != n_valid else out


def conv_wgrad(dy, x1, x2=None, ntaps=9, out=None, row_map=None):
    """Packed weight gradient fp32 [cout, taps, kpad] (accumulated into `out` when given).
    row_map (1x1 convs; device int32 [cout]): the gradient of executed output channel r goes to row row_map[r] of `out`."""
    _need_cuda(dy, x1)
    pd, cout, ldd, n, h, w = _nhwc(dy)
    p1, c1, ld1, n1, h1, w1 = _nhwc(x1)
    assert (n1, h1, w1) == (n, h, w)
    p2, c2, ld2 = None, 0, 0
    if x2 is not None:
        p2, c2, ld2, _, _, _ = _nhwc(x2)
    kpad = pad64(c1) + (pad64(c2) if x2 is not None else 0)
    if out is None:
        out = torch.zeros(cout, ntaps, kpad, device=dy.device, dtype=F32)
    if row_map is not None:
        assert row_map.dtype == torch.int32 and row_map.numel() == cout and row_map.is_cuda
        check(_lib.load().adm_conv_wgrad_mapped(pd, cout, ldd, p1, c1, ld1, p2, c2, ld2, n, h, w, ntaps, _ptr(row_map),
                                                _ptr(out), _stream()), "conv_wgrad_mapped")
        return out
    check(_lib.load().adm_conv_wgrad(pd, cout, ldd, p1, c1, ld1, p2, c2, ld2, n, h, w, ntaps, _ptr(out), _stream()),
          "conv_wgrad")
    return out


def _operand(t, mn_major, dims, strides, c0=0, c0_lo=0, c1=0, c1_lo=0, bhi=0, blo=0):
    return Operand(t.data_ptr(), int(mn_major), dims[0], dims[1], dims[2], strides[0], strides[1], c0, c0_lo, c1,
                   c1_lo, bhi, blo)


def gemm_nt(a, b, bias=None, out_dtype=F32, alpha=1.0, out=None):
    """C[M,N] = alpha * A[M,K] @ B[N,K]^T + bias.  a, b: bf16 row-major (last dim contiguous)."""
    _need_cuda(a, b)
    assert a.dtype == BF16 and b.dtype == BF16 and a.stride(1) == 1 and b.stride(1) == 1
    m, k = a.shape
    n, k2 = b.shape
    assert k == k2
    if out is None:
        out = torch.empty(m, n, device=a.device, dtype=out_dtype)
    d = GemmDesc()
    d.a = _operand(a, 0, (k, m, 1), (a.stride(0), a.stride(0) * m))
    d.b = _operand(b, 0, (k, n, 1), (b.stride(0), b.stride(0) * n))
    d.m, d.n, d.k, d.batches, d.bdiv, d.splits = m, n, k, 1, 1, 1
    d.c, d.out_mode, d.ldc = out.data_ptr(), 0 if out.dtype == BF16 else 1, out.stride(0)
    d.bias, d.residual, d.alpha = _ptr(bias), None, float(alpha)
    check(_lib.load().adm_gemm_batched(d, _stream()), "gemm_nt")
    return out


def gemm_nn(a, b, out_dtype=F32, alpha=1.0, out=None, splits=1):
    """C[M,N] = alpha * A[M,K] @ B[K,N]; B row-major (N contiguous) consumed as an MN-major operand.
    splits > 1: split K over that many tiles (fp32 atomics into a zeroed fp32 output) — for a long K with few output tiles."""
    _need_cuda(a, b)
    assert a.dtype == BF16 and b.dtype == BF16 and a.stride(1) == 1 and b.stride(1) == 1
    m, k = a.shape
    k2, n = b.shape
    assert k == k2
    if out is None:
        out = (torch.zeros if splits > 1 else torch.empty)(m, n, device=a.device, dtype=F32 if splits > 1 else out_dtype)
    assert splits == 1 or out.dtype == F32
    d = GemmDesc()
    d.a = _operand(a, 0, (k, m, 1), (a.stride(0), a.stride(0) * m))
    d.b = _operand(b, 1, (n, k, 1), (b.stride(0), b.stride(0) * k))
    d.m, d.n, d.k, d.batches, d.bdiv, d.splits = m, n, k, 1, 1, splits
    d.c, d.out_mode, d.ldc = out.data_ptr(), (2 if splits > 1 else (0 if out.dtype == BF16 else 1)), out.stride(0)
    d.alpha = float(alpha)
    check(_lib.load().adm_gemm_batched(d, _stream()), "gemm_nn")
    return out


def gemm_tn(a, b, out_dtype=F32, alpha=1.0, out=None, splits=1, accumulate=False):
    """C[M,N] = alpha * A[K,M]^T @ B[K,N]; both row-major, both consumed MN-major (the wgrad shape).
    accumulate: C += (fp32 atomics) into the given `out`."""
    _need_cuda(a, b)
    assert a.dtype == BF16 and b.dtype == BF16 and a.stride(1) == 1 and b.stride(1) == 1
    k, m = a.shape
    k2, n = b.shape
    assert k == k2
    if out is None:
        out = (torch.zeros if splits > 1 else torch.empty)(m, n, device=a.device, dtype=F32 if splits > 1 else out_dtype)
    d = GemmDesc()
    d.a = _operand(a, 1, (m, k, 1), (a.stride(0), a.stride(0) * k))
    d.b = _operand(b, 1, (n, k, 1), (b.stride(0), b.stride(0) * k))
    d.m, d.n, d.k, d.batches, d.bdiv, d.splits = m, n, k, 1, 1, splits
    atomic = splits > 1 or accumulate
    assert not atomic or out.dtype == F32
    d.c, d.out_mode, d.ldc = out.data_ptr(), (2 if atomic else (0 if out.dtype == BF16 else 1)), out.stride(0)
    d.alpha = float(alpha)
    check(_lib.load().adm_gemm_batched(d, _stream()), "gemm_tn")
    return out


# ------------------------------------------------------------------------------------------------ GroupNorm family
def _src(x):
    """(ptr, C, ld) of an NHWC / [rows, C] bf16 view (or (None, 0, 0))."""
    if x is None:
        return None, 0, 0
    assert x.dtype == BF16 and x.stride(-1) == 1
    return x.data_ptr(), x.shape[-1], x.stride(-2)


def gn_stats(x1, x2, gamma, beta, groups, eps=1e-5, params=None):
    """GroupNorm pass 1 over the (fused concat of) x1, x2: returns coef fp32 [N, C, 4] = {A, B, mean, rstd}."""
    _need_cuda(x1)
    n, h, w, _ = x1.shape
    p1, c1, ld1 = _src(x1)
    p2, c2, ld2 = _src(x2)
    c = c1 + c2
    work = torch.empty(2 * n * c + n, device=x1.device, dtype=F32)
    coef = torch.empty(n, c, 4, device=x1.device, dtype=F32)
    ldp = params.stride(0) if params is not None else 0
    check(_lib.load().adm_gn_stats(p1, c1, ld1, p2, c2, ld2, n, h * w, groups, float(eps), _ptr(gamma), _ptr(beta),
                                   _ptr(params), ldp, _ptr(work), _ptr(coef), _stream()), "gn_stats")
    return coef


def gn_apply(x1, x2, coef, act=True, drop_p=0.0, seed=0, resample=0, seed_counter=None):
    n, h, w, _ = x1.shape
    p1, c1, ld1 = _src(x1)
    p2, c2, ld2 = _src(x2)
    ho, wo = (h // 2, w // 2) if resample == 1 else ((2 * h, 2 * w) if resample == 2 else (h, w))
    out = torch.empty(n, ho, wo, c1 + c2, device=x1.device, dtype=BF16)
    check(_lib.load().adm_gn_apply(p1, c1, ld1, p2, c2, ld2, n, h, w, _ptr(coef), int(act), float(drop_p),
                                   int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(seed_counter), int(resample), _ptr(out),
                                   out.stride(2), _stream()), "gn_apply")
    return out


def gn_forward(x1, x2, gamma, beta, groups, eps=1e-5, params=None, act=True, drop_p=0.0, seed=0, resample=0,
               seed_counter=None):
    """GroupNorm statistics + apply in one call (one cluster-per-sample kernel when the batch fills the SMs).
    seed_counter: optional CUDA int64[1] step counter mixed into the dropout seed (read only when drop_p > 0).
    Returns (coef [N, C, 4], y)."""
    _need_cuda(x1)
    n, h, w, _ = x1.shape
    p1, c1, ld1 = _src(x1)
    p2, c2, ld2 = _src(x2)
    c = c1 + c2
    work = torch.empty(2 * n * c + n, device=x1.device, dtype=F32)
    coef = torch.empty(n, c, 4, device=x1.device, dtype=F32)
    ho, wo = (h // 2, w // 2) if resample == 1 else ((2 * h, 2 * w) if resample == 2 else (h, w))
    out = torch.empty(n, ho, wo, c, device=x1.device, dtype=BF16)
    ldp = params.stride(0) if params is not None else 0
    check(_lib.load().adm_gn_forward(p1, c1, ld1, p2, c2, ld2, n, h, w, groups, float(eps), _ptr(gamma), _ptr(beta),
                                     _ptr(params), ldp, _ptr(work), _ptr(coef), int(act), float(drop_p),
                                     int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(seed_counter), int(resample), _ptr(out),
                                     out.stride(2), _stream()), "gn_forward")
    return coef, out


def gn_bwd(dy, x1, x2, coef, gamma, beta, groups, params=None, act=True, drop_p=0.0, seed=0, resample=0,
           dgamma=None, dbeta=None, dparams=None, add=None, add_mode=0, need_dx=True, dbias1=None, dbias1b=None,
           seed_counter=None, dy_scratch=False):
    """Returns (dx1, dx2).  dgamma/dbeta are accumulated in place; dparams ([N, 2C] view) is overwritten;
    dbias1 (fp32 [c1]) += column sums of dx1.  dy_scratch=True lets the kernel overwrite dy (saves recomputation)."""
    n, h, w, _ = x1.shape
    p1, c1, ld1 = _src(x1)
    p2, c2, ld2 = _src(x2)
    c = c1 + c2
    assert dy.dtype == BF16 and dy.stride(-1) == 1
    work = torch.empty(2 * n * c + n, device=x1.device, dtype=F32)
    bcoef = torch.empty(n, c, 4, device=x1.device, dtype=F32)
    dx1 = torch.empty(n, h, w, c1, device=x1.device, dtype=BF16) if need_dx else None
    dx2 = torch.empty(n, h, w, c2, device=x1.device, dtype=BF16) if (need_dx and x2 is not None) else None
    ldp = params.stride(0) if params is not None else 0
    lddp = dparams.stride(0) if dparams is not None else 0
    check(_lib.load().adm_gn_bwd(_ptr(dy), dy.stride(-2), p1, c1, ld1, p2, c2, ld2, n, h, w, groups, _ptr(coef),
                                 _ptr(gamma), _ptr(beta), _ptr(params), ldp, int(act), float(drop_p),
                                 int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(seed_counter), int(resample), _ptr(work),
                                 _ptr(bcoef), _ptr(dgamma),
                                 _ptr(dbeta), _ptr(dparams), lddp, _ptr(add),
                                 add.stride(-2) if add is not None else 0, int(add_mode), _ptr(dx1),
                                 dx1.stride(2) if dx1 is not None else 0, _ptr(dx2),
                                 dx2.stride(2) if dx2 is not None else 0, _ptr(dbias1), _ptr(dbias1b), int(dy_scratch),
                                 _stream()), "gn_bwd")
    return dx1, dx2


def col_sums(x, out, out_map=None):
    """out[c] += sum over rows of x[..., c]; x bf16 with contiguous last dim and uniform row stride.
    out_map (device int32 [c]): column c is accumulated into out[out_map[c]] instead."""
    c = x.shape[-1]
    rows = x.numel() // c
    if out_map is not None:
        assert out_map.dtype == torch.int32 and out_map.numel() == c and out_map.is_cuda
        check(_lib.load().adm_col_sums_mapped(_ptr(x), x.stride(-2), rows, c, _ptr(out), _ptr(out_map), _stream()),
              "col_sums_mapped")
        return out
    check(_lib.load().adm_col_sums(_ptr(x), x.stride(-2), rows, c, _ptr(out), _stream()), "col_sums")
    return out


def gather_rows(src, dst, table, row_bytes):
    """For every row i of table (device int64 [rows, 2], BYTE offsets): dst[table[i,1] : +row_bytes] = src[table[i,0] : ...]."""
    _need_cuda(src, dst, table)
    assert table.dtype == torch.int64 and table.is_contiguous() and table.shape[1] == 2
    check(_lib.load().adm_gather_rows(_ptr(src), _ptr(dst), _ptr(table), table.shape[0], int(row_bytes), _stream()),
          "gather_rows")
    return dst


def resample(x, mode):
    n, h, w, c = x.shape
    ho, wo = (h // 2, w // 2) if mode == 1 else (2 * h, 2 * w)
    out = torch.empty(n, ho, wo, c, device=x.device, dtype=BF16)
    check(_lib.load().adm_resample(_ptr(x), x.stride(2), n, h, w, c, mode, _ptr(out), out.stride(2), _stream()),
          "resample")
    return out


def add_bf16(a, b, c=None):
    """a + b (+ c) on NHWC bf16 views (any pixel stride)."""
    out = torch.empty(a.shape, device=a.device, dtype=BF16)
    ch = a.shape[-1]
    rows = a.numel() // ch
    check(_lib.load().adm_add_bf16(_ptr(a), a.stride(-2), _ptr(b), b.stride(-2), _ptr(c),
                                   c.stride(-2) if c is not None else 0, _ptr(out), out.stride(-2), rows, ch,
                                   _stream()), "add_bf16")
    return out


def silu(x, want_f32=True, want_bf16=True):
    x = x.contiguous()
    y = torch.empty_like(x) if want_f32 else None
    yb = torch.empty(x.shape, device=x.device, dtype=BF16) if want_bf16 else None
    check(_lib.load().adm_silu(_ptr(x), _ptr(y), _ptr(yb), x.numel(), _stream()), "silu")
    return y, yb


def silu_bwd(x, dy, want_f32=True, want_bf16=True):
    x, dy = x.contiguous(), dy.contiguous()
    dx = torch.empty_like(x) if want_f32 else None
    dxb = torch.empty(x.shape, device=x.device, dtype=BF16) if want_bf16 else None
    check(_lib.load().adm_silu_bwd(_ptr(x), _ptr(dy), _ptr(dx), _ptr(dxb), x.numel(), _stream()), "silu_bwd")
    return dx, dxb


# ------------------------------------------------------------------------------------------------ attention
def softmax_fwd(s):
    rows, length = s.numel() // s.shape[-1], s.shape[-1]
    p = torch.empty(s.shape, device=s.device, dtype=BF16)
    check(_lib.load().adm_softmax_fwd(_ptr(s), _ptr(p), rows, length, _stream()), "softmax_fwd")
    return p


SOFTMAX_BWD_MAX_LEN = 1024  # one warp per row, 32 values per lane (adm_softmax_bwd)


def softmax_bwd(p, dp, scale):
    rows, length = p.numel() // p.shape[-1], p.shape[-1]
    ds = torch.empty(p.shape, device=p.device, dtype=BF16)
    check(_lib.load().adm_softmax_bwd(_ptr(p), _ptr(dp), _ptr(ds), float(scale), rows, length, _stream()),
          "softmax_bwd")
    return ds


def _gemm(desc_kw, a_op, b_op, what):
    d = GemmDesc()
    d.a, d.b = a_op, b_op
    for k, v in desc_kw.items():
        setattr(d, k, v)
    check(_lib.load().adm_gemm_batched(d, _stream()), what)


def attention_fused_ok(d, hw):
    """Shapes served by the fused K9 kernels (everything else runs as batched GEMMs + a softmax kernel): one unit per
    (sample, head) up to 256 pixels, 256 x 256 blocks with a log-sum-exp merge for 512..4096 pixels."""
    return d == 64 and (hw in (16, 64, 256) or (hw % 256 == 0 and 512 <= hw <= 4096))


def _attn_workspace(n, hw, heads, backward, device):
    nbytes = _lib.load().adm_attn_long_workspace(n, hw, heads, int(backward))
    return torch.empty(nbytes, device=device, dtype=torch.uint8), nbytes


def attention_fwd(qkv, heads, scale=None, need_p=True, fused=None, out=None, lse=None, work=None):
    """qkv: [N, H, W, 3C] bf16 laid out as (q | k | v), each [heads, d].  Returns (a [N,H,W,C], aux) where aux is what
    attention_bwd needs besides qkv and a: the per-row log-sum-exp [N, heads, HW] fp32 for the fused kernel (d == 64, HW in
    {16, 64, 256}: ONE kernel, probabilities only ever in TMEM), or the normalised probabilities [N*heads, HW, HW] bf16
    for the unfused path.  aux is None when need_p is False.
    scale defaults to 1/sqrt(d) (d = C / heads as stored, which may include zero padding of the head dim).
    out / lse: contiguous tensors to write a / the log-sum-exp into (allocated when None); work: a uint8 scratch buffer
    for the blocked kernels (HW > 256), at least adm_attn_long_workspace bytes."""
    n, h, w, c3 = qkv.shape
    c, hw = c3 // 3, h * w
    d = c // heads
    scale = 1.0 / d ** 0.5 if scale is None else float(scale)
    assert qkv.is_contiguous()
    if out is None:
        out = torch.empty(n, h, w, c, device=qkv.device, dtype=BF16)
    assert out.is_contiguous() and out.dtype == BF16 and tuple(out.shape) == (n, h, w, c)
    a = out
    if fused is None:
        fused = attention_fused_ok(d, hw)
    if fused:
        if lse is None and need_p:
            lse = torch.empty(n, heads, hw, device=qkv.device, dtype=F32)
        assert lse is None or (lse.is_contiguous() and lse.dtype == F32 and tuple(lse.shape) == (n, heads, hw))
        if hw > 256:
            if work is None:
                work, nbytes = _attn_workspace(n, hw, heads, False, qkv.device)
            else:
                nbytes = work.numel() * work.element_size()
            check(_lib.load().adm_attn_fwd_long(_ptr(qkv), n, hw, heads, scale, _ptr(a), _ptr(lse), _ptr(work), nbytes,
                                                _stream()), "attn_fwd_long")
            return a, lse
        check(_lib.load().adm_attn_fwd_fused(_ptr(qkv), n, hw, heads, scale, _ptr(a), _ptr(lse), _stream()),
              "attn_fwd_fused")
        return a, lse
    s = torch.empty(n * heads, hw, hw, device=qkv.device, dtype=F32)
    qk_dims, qk_str = (c3, hw, n), (c3, c3 * hw)
    _gemm(dict(m=hw, n=hw, k=d, batches=n * heads, bdiv=heads, splits=1, c=s.data_ptr(), out_mode=1, ldc=hw,
               c_bhi=heads * hw * hw, c_blo=hw * hw, c_col_lo=0, alpha=scale),
          _operand(qkv, 0, qk_dims, qk_str, c0=0, c0_lo=d, bhi=1),
          _operand(qkv, 0, qk_dims, qk_str, c0=c, c0_lo=d, bhi=1), "attn QK^T")
    p = softmax_fwd(s)
    _gemm(dict(m=hw, n=d, k=hw, batches=n * heads, bdiv=heads, splits=1, c=a.data_ptr(), out_mode=0, ldc=c,
               c_bhi=hw * c, c_blo=0, c_col_lo=d, alpha=1.0),
          _operand(p, 0, (hw, hw, n * heads), (hw, hw * hw), bhi=heads, blo=1),
          _operand(qkv, 1, qk_dims, qk_str, c0=2 * c, c0_lo=d, bhi=1), "attn PV")
    return a, p


def attention_bwd(da, qkv, aux, heads, scale=None, fused=None, a=None, out=None, work=None):
    """Returns dqkv [N,H,W,3C] bf16.  Fused (aux = log-sum-exp, `a` = the forward output): ONE kernel recomputes the
    probabilities and produces dQ, dK, dV.  Unfused (aux = the saved probabilities): five batched GEMMs + softmax_bwd.
    out: a contiguous tensor to write dqkv into (allocated when None); work: as in attention_fwd."""
    n, h, w, c3 = qkv.shape
    c, hw = c3 // 3, h * w
    d = c // heads
    scale = 1.0 / d ** 0.5 if scale is None else float(scale)
    assert da.is_contiguous() and qkv.is_contiguous()
    if out is None:
        out = torch.empty_like(qkv)
    assert out.is_contiguous() and out.dtype == BF16 and out.shape == qkv.shape
    dqkv = out
    if fused is None:
        fused = attention_fused_ok(d, hw)
    if fused:
        assert a is not None and a.is_contiguous() and aux is not None and aux.dtype == F32, \
            "fused attention backward needs the forward output and its log-sum-exp"
        if hw > 256:
            if work is None:
                work, nbytes = _attn_workspace(n, hw, heads, True, qkv.device)
            else:
                nbytes = work.numel() * work.element_size()
            check(_lib.load().adm_attn_bwd_long(_ptr(da), _ptr(qkv), _ptr(a), _ptr(aux), n, hw, heads, scale, _ptr(dqkv),
                                                _ptr(work), nbytes, _stream()), "attn_bwd_long")
            return dqkv
        check(_lib.load().adm_attn_bwd_fused(_ptr(da), _ptr(qkv), _ptr(a), _ptr(aux), n, hw, heads, scale, _ptr(dqkv),
                                             _stream()), "attn_bwd_fused")
        return dqkv
    if hw > SOFTMAX_BWD_MAX_LEN:  # before the first GEMM: a rejected shape launches nothing and leaves dqkv untouched
        raise _lib.AdmError(f"attention_bwd: the unfused backward takes rows of at most {SOFTMAX_BWD_MAX_LEN} keys "
                            f"(got {hw})")
    p = aux
    qk_dims, qk_str = (c3, hw, n), (c3, c3 * hw)
    a_dims, a_str = (c, hw, n), (c, c * hw)
    p_dims, p_str = (hw, hw, n * heads), (hw, hw * hw)
    nb = n * heads
    esz = 2
    # dV[k, d] = sum_q P[q, k] dA[q, d]
    _gemm(dict(m=hw, n=d, k=hw, batches=nb, bdiv=heads, splits=1, c=dqkv.data_ptr() + 2 * c * esz, out_mode=0,
               ldc=c3, c_bhi=hw * c3, c_blo=0, c_col_lo=d, alpha=1.0),
          _operand(p, 1, p_dims, p_str, bhi=heads, blo=1),
          _operand(da, 1, a_dims, a_str, c0=0, c0_lo=d, bhi=1), "attn dV")
    # dP[q, k] = sum_d dA[q, d] V[k, d]
    dp = torch.empty(nb, hw, hw, device=qkv.device, dtype=F32)
    _gemm(dict(m=hw, n=hw, k=d, batches=nb, bdiv=heads, splits=1, c=dp.data_ptr(), out_mode=1, ldc=hw,
               c_bhi=heads * hw * hw, c_blo=hw * hw, c_col_lo=0, alpha=1.0),
          _operand(da, 0, a_dims, a_str, c0=0, c0_lo=d, bhi=1),
          _operand(qkv, 0, qk_dims, qk_str, c0=2 * c, c0_lo=d, bhi=1), "attn dP")
    ds = softmax_bwd(p, dp, scale)
    # dQ[q, d] = sum_k dS[q, k] K[k, d]
    _gemm(dict(m=hw, n=d, k=hw, batches=nb, bdiv=heads, splits=1, c=dqkv.data_ptr(), out_mode=0, ldc=c3,
               c_bhi=hw * c3, c_blo=0, c_col_lo=d, alpha=1.0),
          _operand(ds, 0, p_dims, p_str, bhi=heads, blo=1),
          _operand(qkv, 1, qk_dims, qk_str, c0=c, c0_lo=d, bhi=1), "attn dQ")
    # dK[k, d] = sum_q dS[q, k] Q[q, d]
    _gemm(dict(m=hw, n=d, k=hw, batches=nb, bdiv=heads, splits=1, c=dqkv.data_ptr() + c * esz, out_mode=0, ldc=c3,
               c_bhi=hw * c3, c_blo=0, c_col_lo=d, alpha=1.0),
          _operand(ds, 1, p_dims, p_str, bhi=heads, blo=1),
          _operand(qkv, 1, qk_dims, qk_str, c0=0, c0_lo=d, bhi=1), "attn dK")
    return dqkv


def spatial_att_fwd(h, res, w_map, scalars):
    n, hh, ww, c = h.shape
    out = torch.empty(n, hh, ww, c, device=h.device, dtype=BF16)
    att = torch.empty(n, hh * ww, device=h.device, dtype=F32)
    o = torch.empty_like(att)
    check(_lib.load().adm_spatial_att_fwd(_ptr(h), h.stride(2), _ptr(res), res.stride(2), _ptr(w_map), _ptr(scalars),
                                          n, hh * ww, c, _ptr(out), out.stride(2), _ptr(att), _ptr(o), _stream()),
          "spatial_att_fwd")
    return out, att, o


def spatial_att_bwd(dy, h, w_map, scalars, att, o, dw_map, dscalars):
    n, hh, ww, c = h.shape
    dh = torch.empty(n, hh, ww, c, device=h.device, dtype=BF16)
    check(_lib.load().adm_spatial_att_bwd(_ptr(dy), dy.stride(2), _ptr(h), h.stride(2), _ptr(w_map), _ptr(scalars),
                                          _ptr(att), _ptr(o), n, hh * ww, c, _ptr(dh), dh.stride(2), _ptr(dw_map),
                                          _ptr(dscalars), _stream()), "spatial_att_bwd")
    return dh


# ------------------------------------------------------------------------------------------------ optimizer
def sq_norm(g, out):
    check(_lib.load().adm_sq_norm(_ptr(g), g.numel(), _ptr(out), _stream()), "sq_norm")
    return out


def adamw(p, g, m, v, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0, max_norm=0.0, sqnorm=None,
          hyper_dev=None, p_bf16=None):
    check(_lib.load().adm_adamw(_ptr(p), _ptr(g), _ptr(m), _ptr(v), p.numel(), float(lr), float(beta1), float(beta2),
                                float(eps), float(weight_decay), int(step), float(grad_scale), float(max_norm),
                                _ptr(sqnorm), _ptr(hyper_dev), _ptr(p_bf16), _stream()), "adamw")


def lerp_f32(dst, src, weight):
    """dst += weight * (src - dst) over two flat fp32 CUDA tensors of equal length (the EMA arena update)."""
    _need_cuda(dst, src)
    assert dst.dtype == F32 and src.dtype == F32 and dst.is_contiguous() and src.is_contiguous()
    assert dst.numel() == src.numel()
    check(_lib.load().adm_lerp_f32(_ptr(dst), _ptr(src), dst.numel(), float(weight), _stream()), "lerp_f32")
    return dst


# ------------------------------------------------------------------------------------------------ conditional UNet ops
def ws_pack(w, eps=1e-5):
    """K11: weight standardisation + bf16 re-pack.  w fp32 [cout, cin, k, k] -> (wpk bf16 [cout, k*k, pad64(cin)], stats)."""
    _need_cuda(w)
    cout, cin, k, _ = w.shape
    w = w.contiguous()
    wpk = torch.empty(cout, k * k, pad64(cin), device=w.device, dtype=BF16)
    stats = torch.empty(cout, 2, device=w.device, dtype=F32)
    check(_lib.load().adm_ws_pack(_ptr(w), _ptr(wpk), _ptr(stats), cout, cin, k, float(eps), _stream()), "ws_pack")
    return wpk, stats


def ws_pack_bwd(dw_packed, w, stats, out=None, accumulate=False):
    """dw (reference layout) from the packed gradient w.r.t. the standardised weights."""
    cout, cin, k, _ = w.shape
    if out is None:
        out = torch.empty_like(w, memory_format=torch.contiguous_format)
        accumulate = False
    check(_lib.load().adm_ws_pack_bwd(_ptr(dw_packed), _ptr(w.contiguous()), _ptr(stats), _ptr(out), cout, cin, k,
                                      int(accumulate), _stream()), "ws_pack_bwd")
    return out


def _linattn_work(b, heads, n, device):
    import ctypes
    fl = ctypes.c_longlong(0)
    _lib.load().adm_linattn_workspace(b, heads, n, ctypes.byref(fl))
    return torch.empty(fl.value, device=device, dtype=F32)


def linattn_fwd(qkv, heads, scale):
    """K12.  qkv [B, H, W, 3*heads*32] bf16 (q | k | v).  Returns (out [B, H, W, heads*32], ctx, kstat)."""
    _need_cuda(qkv)
    b, h, w, c3 = qkv.shape
    hidden = c3 // 3
    assert hidden == heads * 32 and qkv.dtype == BF16 and qkv.stride(3) == 1
    n = h * w
    out = torch.empty(b, h, w, hidden, device=qkv.device, dtype=BF16)
    ctx = torch.empty(b * heads, 32, 32, device=qkv.device, dtype=F32)
    kstat = torch.empty(b * heads, 32, 2, device=qkv.device, dtype=F32)
    work = _linattn_work(b, heads, n, qkv.device)
    check(_lib.load().adm_linattn_fwd(_ptr(qkv), qkv.stride(2), b, n, heads, 32, float(scale), _ptr(out), out.stride(2),
                                      _ptr(ctx), _ptr(kstat), _ptr(work), _stream()), "linattn_fwd")
    return out, ctx, kstat


def linattn_bwd(dout, qkv, ctx, kstat, heads, scale):
    b, h, w, c3 = qkv.shape
    n = h * w
    assert dout.dtype == BF16 and dout.stride(3) == 1
    dqkv = torch.empty_like(qkv)
    dctx = torch.empty_like(ctx)
    r = torch.empty(b * heads, 32, device=qkv.device, dtype=F32)
    work = _linattn_work(b, heads, n, qkv.device)
    check(_lib.load().adm_linattn_bwd(_ptr(qkv), qkv.stride(2), b, n, heads, 32, float(scale), _ptr(dout),
                                      dout.stride(2), _ptr(ctx), _ptr(kstat), _ptr(dctx), _ptr(r), _ptr(work),
                                      _ptr(dqkv), dqkv.stride(2), _stream()), "linattn_bwd")
    return dqkv


# ------------------------------------------------------------------------------------------------ channel LayerNorm
def chan_layernorm_ok(c):
    return bool(_lib.load().adm_chan_layernorm_ok(int(c)))


def chan_layernorm_fwd(x, g, eps=1e-5):
    """Per-pixel LayerNorm over the channels of an NHWC bf16 tensor with gain g [C] fp32 (cond_unet.py:360-369)."""
    _need_cuda(x, g)
    assert x.dtype == BF16 and x.stride(-1) == 1 and g.dtype == F32 and g.is_contiguous()
    c = x.shape[-1]
    rows = x.numel() // c
    y = torch.empty(x.shape, device=x.device, dtype=BF16)
    check(_lib.load().adm_chan_layernorm_fwd(_ptr(x), x.stride(-2), rows, c, _ptr(g), float(eps), _ptr(y), c, _stream()),
          "chan_layernorm_fwd")
    return y


def chan_layernorm_bwd(dy, x, g, eps=1e-5):
    """Returns (dx bf16 like x, dg fp32 [C])."""
    _need_cuda(dy, x, g)
    assert dy.dtype == BF16 and dy.stride(-1) == 1 and x.stride(-1) == 1
    c = x.shape[-1]
    rows = x.numel() // c
    dx = torch.empty(x.shape, device=x.device, dtype=BF16)
    dg = torch.zeros(c, device=x.device, dtype=F32)
    check(_lib.load().adm_chan_layernorm_bwd(_ptr(dy), dy.stride(-2), _ptr(x), x.stride(-2), rows, c, _ptr(g), float(eps),
                                             _ptr(dx), c, _ptr(dg), _stream()), "chan_layernorm_bwd")
    return dx, dg


# ------------------------------------------------------------------------------------------------ relation layers
def rel_gn_ok(x, groups):
    """True when the fused relation-layer tail takes this NHWC bf16 map (cond_unet.py:236-251)."""
    b, h, w, c = x.shape
    return bool(_lib.load().adm_rel_gn_ok(int(b), int(h), int(w), int(c), int(groups)))


def _rel_work(b, h, w, c, groups, device):
    chunks = _lib.load().adm_rel_gn_chunks(int(b), int(h), int(w), int(c))
    return torch.empty(b, chunks, max(groups, c), 2, device=device, dtype=F32), chunks


def rel_gn_fwd(x, y, z, gamma, beta, groups, eps=1e-5, out_dtype=BF16):
    """out = GroupNorm(x + y) * gamma + beta + bilinear(z) with the sum in fp32 registers; x, y NHWC bf16 [B,H,W,C],
    z fp32 [B,hq,wq,C].  Returns (out, stats fp32 [B,groups,2])."""
    _need_cuda(x, y, z, gamma, beta)
    assert x.dtype == BF16 and y.dtype == BF16 and x.is_contiguous() and y.is_contiguous() and x.shape == y.shape
    assert z.dtype == F32 and z.is_contiguous() and z.shape[0] == x.shape[0] and z.shape[-1] == x.shape[-1]
    assert gamma.dtype == F32 and beta.dtype == F32 and gamma.is_contiguous() and beta.is_contiguous()
    b, h, w, c = x.shape
    out = torch.empty(x.shape, device=x.device, dtype=out_dtype)
    stats = torch.empty(b, groups, 2, device=x.device, dtype=F32)
    work, _ = _rel_work(b, h, w, c, groups, x.device)
    check(_lib.load().adm_rel_gn_fwd(_ptr(x), _ptr(y), _ptr(z), b, h, w, c, int(z.shape[1]), int(z.shape[2]), int(groups),
                                     _ptr(gamma), _ptr(beta), float(eps), _ptr(out), int(out_dtype == F32), _ptr(stats),
                                     _ptr(work), _stream()), "rel_gn_fwd")
    return out, stats


def rel_gn_bwd(dout, x, y, gamma, stats, groups):
    """Returns (dpre bf16 like x, dgamma fp32 [C], dbeta fp32 [C])."""
    _need_cuda(dout, x, y, gamma, stats)
    assert dout.dtype == BF16 and dout.is_contiguous() and dout.shape == x.shape
    b, h, w, c = x.shape
    dpre = torch.empty(x.shape, device=x.device, dtype=BF16)
    work, chunks = _rel_work(b, h, w, c, groups, x.device)
    check(_lib.load().adm_rel_gn_bwd(_ptr(dout), _ptr(x), _ptr(y), b, h, w, c, int(groups), _ptr(gamma), _ptr(stats),
                                     _ptr(dpre), _ptr(work), _stream()), "rel_gn_bwd")
    sums = work.view(-1)[:b * chunks * c * 2].view(b * chunks, c, 2).sum(0)
    return dpre, sums[:, 0].contiguous(), sums[:, 1].contiguous()


def bilinear_fwd(x, size, out_dtype=None):
    """NHWC bilinear resize, align_corners=True (F.interpolate, cond_unet.py:184, :248); x bf16 or fp32, last dim dense."""
    _need_cuda(x)
    assert x.dtype in (BF16, F32) and x.dim() == 4 and x.stride(-1) == 1
    b, h, w, c = x.shape
    assert x.stride(1) == w * x.stride(2) and x.stride(0) == h * x.stride(1)
    out_dtype = out_dtype or x.dtype
    y = torch.empty(b, int(size[0]), int(size[1]), c, device=x.device, dtype=out_dtype)
    check(_lib.load().adm_bilinear_fwd(_ptr(x), x.stride(2), b, h, w, c, _ptr(y), c, int(size[0]), int(size[1]),
                                       int(x.dtype == F32), int(out_dtype == F32), _stream()), "bilinear_fwd")
    return y


def bilinear_bwd(dy, size_in):
    """dy bf16 [B,hout,wout,C] contiguous -> dx fp32 [B,hin,win,C]."""
    _need_cuda(dy)
    assert dy.dtype == BF16 and dy.is_contiguous()
    b, ho, wo, c = dy.shape
    hin, win = int(size_in[0]), int(size_in[1])
    tmp = torch.empty(b, hin, wo, c, device=dy.device, dtype=F32)
    dx = torch.empty(b, hin, win, c, device=dy.device, dtype=F32)
    check(_lib.load().adm_bilinear_bwd(_ptr(dy), b, ho, wo, c, hin, win, _ptr(tmp), _ptr(dx), _stream()), "bilinear_bwd")
    return dx


def avgpool_fwd(x, window):
    """F.pad to a multiple of the window + nn.AvgPool2d(window) on an NHWC bf16 map (cond_unet.py:190-200)."""
    _need_cuda(x)
    assert x.dtype == BF16 and x.is_contiguous()
    b, h, w, c = x.shape
    kh, kw = int(window[0]), int(window[1])
    out = torch.empty(b, -(-h // kh), -(-w // kw), c, device=x.device, dtype=BF16)
    check(_lib.load().adm_avgpool_fwd(_ptr(x), b, h, w, c, kh, kw, _ptr(out), _stream()), "avgpool_fwd")
    return out


def avgpool_bwd(dy, shape, window):
    _need_cuda(dy)
    assert dy.dtype == BF16 and dy.is_contiguous()
    b, h, w, c = shape
    dx = torch.empty(b, h, w, c, device=dy.device, dtype=BF16)
    check(_lib.load().adm_avgpool_bwd(_ptr(dy), b, h, w, c, int(window[0]), int(window[1]), _ptr(dx), _stream()),
          "avgpool_bwd")
    return dx


# ------------------------------------------------------------------------------------------------ AugmentPipe warp
def augment_warp(x, theta, flips, margins):
    """x fp32 [N,C,H,W] (CUDA) -> flipped + warped batch (ddm/augment.py:153-328); theta fp32 [N,6], flips int32 [N,2],
    margins = (mx0, mx1, my0, my1) host ints."""
    _need_cuda(x, theta, flips)
    assert x.dtype == F32 and x.is_contiguous() and theta.dtype == F32 and flips.dtype == torch.int32
    n, c, h, w = x.shape
    y = torch.empty_like(x)
    mx0, mx1, my0, my1 = (int(v) for v in margins)
    check(_lib.load().adm_augment_warp(_ptr(x), _ptr(y), _ptr(theta), _ptr(flips), n, c, h, w, mx0, mx1, my0, my1,
                                       _stream()), "augment_warp")
    return y
