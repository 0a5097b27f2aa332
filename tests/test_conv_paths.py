"""Conv engine path by path: adm_conv_fprop / adm_conv_dgrad / adm_conv_wgrad at the tile edges where implicit-GEMM
kernels go wrong.  Each row of CASES names the kernel its shape must be routed to and the edge it exists for; one
checker runs every row:

  * path     the CUDA kernels recorded under torch.profiler are exactly the expected one, and adm_launch_count() grows
             by exactly one.  Kernel selection depends on the SM count: the table is worked out for the 148 SMs of a B200.
  * inputs   x, dy, the residual and the packed weights are views into NaN-filled buffers (channels past the segment, one
             image before the view and a pixel box of images after it, weight rows past Cout); the bias is a view into a
             NaN-filled fp32 buffer.  A correct kernel reads none of it; a read that reaches the output shows up as NaN,
             also where it meets a zero weight.
  * outputs  fprop and dgrad write through a view of a sentinel-filled buffer with >= 16 extra channels and a pixel box
             of images on either side; wgrad accumulates onto finite random values with a guard row on either side.
             Every element the kernel must not write (the packed wgrad pad columns included) keeps its bits.
  * values   every element against an fp64 reference computed from the same bf16 operands:
                 |got - ref| <= (ceil(K / 16) + s + 2) * 2^-23 * S        (+ 2^-8 |ref| for bf16 outputs)
             S is the same operation on absolute values (plus |bias|, |residual|, |prefill|), K the reduction length and
             s the number of partial sums merged.  bf16 products are exact in fp32; the bound allows one fp32 rounding per
             16-deep MMA step and per merge, with a factor of 2 for the MMA's internal rounding.

The test_checker_* tests (CPU) show that the checker accepts an fp32 convolution and rejects subtly wrong kernels.
"""
import math
from dataclasses import dataclass

import pytest
import torch
import torch.nn.functional as F

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
B200_SMS = 148
SENTINEL = 1000.0
# extra output channels: >= 16, and 40 B (bf16) / 72 B (fp32) leave every other pixel row only 8-byte aligned, so each
# case runs both the vector and the scalar stores of the epilogue
GUARD_COLS = {BF16: 20, F32: 18}
FORCE = "ADM_SPLITK_FORCE"

# kernel names as torch.profiler reports them on the B200 (without "void adm::" and the parameter list)
HALO = "tc_conv_halo_kernel"
SPLITK = "tc_conv_splitk_kernel"
CONV = "tc_gemm_kernel<1>"
ROWS = "tc_wgrad_rows_kernel"
WGRAD = "tc_gemm_kernel<2>"


def pad64(c):
    return (c + 63) // 64 * 64


@dataclass(frozen=True)
class Case:
    name: str
    op: str  # "fprop", "dgrad" or "wgrad" of the conv c1 (+ c2 concatenated) -> cout, k x k, 'same' padding
    n: int
    h: int
    w: int
    c1: int
    c2: int
    cout: int
    k: int
    kernel: str
    edge: str
    out: torch.dtype = BF16  # fprop output (dgrad writes bf16, wgrad accumulates fp32)
    bias: bool = False
    residual: bool = False
    alpha: float = 1.0
    force: str = None  # ADM_SPLITK_FORCE="bn,ks": a split-K (tile width, split) pair the cost model does not pick

    @property
    def id(self):
        return f"{self.name}-{self.op}" + (f"-force{self.force.replace(',', 'x')}" if self.force else "")

    @property
    def kpad(self):
        return pad64(self.c1) + (pad64(self.c2) if self.c2 else 0)

    @property
    def cols(self):
        """Output columns: fprop Cout; dgrad the input channels (the whole packed width for a concat); wgrad kpad."""
        if self.op == "fprop":
            return self.cout
        if self.op == "dgrad":
            return self.kpad if self.c2 else self.c1
        return self.kpad

    @property
    def out_dtype(self):
        return {"fprop": self.out, "dgrad": BF16, "wgrad": F32}[self.op]

    @property
    def box_images(self):
        """Images one pixel box can span (128 pixels): the guard and poison depth before / after the views."""
        return max(1, 128 // (self.h * self.w))


def _rows(name, n, h, w, c1, c2, cout, k, edge, kernels, **kw):
    return [Case(name, op, n, h, w, c1, c2, cout, k, kern, edge, **kw.get(op, {})) for op, kern in kernels.items()]


CASES = [
    *_rows("halo-multitile", 64, 32, 32, 192, 0, 192, 3, "512 pixel tiles: >= 3 per CTA even at bn = 256",
           {"fprop": HALO, "dgrad": HALO}, fprop=dict(bias=True)),
    *_rows("conv-multitile-bni2", 889, 8, 8, 192, 0, 192, 3, "445 tiles of two 8x8 images, the last one half full",
           {"fprop": CONV, "dgrad": CONV}, fprop=dict(residual=True), dgrad=dict(residual=True, alpha=0.5)),
    *_rows("bni2-partial-384", 127, 8, 8, 384, 0, 384, 3, "partial bni = 2 tile at the benchmark's 8x8 width",
           {"fprop": CONV, "dgrad": CONV, "wgrad": ROWS}, fprop=dict(out=F32, bias=True)),
    *_rows("1x1-bni8-partial", 125, 4, 4, 384, 0, 384, 1, "1x1 with a partial bni = 8 tile",
           {"fprop": CONV, "dgrad": CONV, "wgrad": WGRAD}, fprop=dict(bias=True, residual=True)),
    *_rows("splitk-partial", 5, 4, 4, 104, 0, 72, 3, "split-K, partial tile, off-grid channels, every epilogue input",
           {"fprop": SPLITK, "dgrad": SPLITK}, fprop=dict(out=F32, bias=True, residual=True, alpha=-0.75),
           dgrad=dict(residual=True, alpha=-0.75)),
    *_rows("splitk-8x16", 3, 8, 16, 96, 0, 160, 3, "split-K on a non-square image",
           {"fprop": SPLITK, "dgrad": SPLITK, "wgrad": ROWS}),
    *[c for f in ("64,2", "128,3", "48,3", "16,2") for c in
      _rows("splitk-forced", 16, 4, 4, 128, 0, 384, 3, "forced split-K (tile width, split) pairs",
            {"fprop": SPLITK, "dgrad": SPLITK} if f in ("64,2", "128,3") else {"fprop": SPLITK},
            fprop=dict(bias=True, force=f), dgrad=dict(force=f))],
    *_rows("halo-64x32", 24, 64, 32, 96, 0, 96, 3, "halo on a non-square image, off-grid channels",
           {"fprop": HALO, "dgrad": HALO}, fprop=dict(residual=True)),
    *_rows("halo-16x8-concat", 2, 16, 8, 96, 32, 96, 3, "halo, non-square, concat 96 + 32",
           {"fprop": HALO, "dgrad": HALO}, fprop=dict(out=F32, bias=True)),
    *_rows("rows-w128", 2, 128, 128, 64, 0, 64, 3, "tap-row wgrad with two tiles across the width",
           {"wgrad": ROWS, "fprop": HALO}),
    *_rows("rows-w64", 3, 64, 64, 96, 0, 96, 3, "tap-row wgrad at W = 64, off-grid channels", {"wgrad": ROWS}),
    *_rows("rows-w64-cout288", 2, 16, 64, 96, 0, 288, 3, "tap-row wgrad, Cout = 288: odd M-chunk tail",
           {"wgrad": ROWS}),
    *_rows("bw4-32x4", 5, 32, 4, 64, 0, 64, 3, "3x3 at a 4-pixel width: generic wgrad, plain conv",
           {"wgrad": WGRAD, "fprop": CONV, "dgrad": CONV}),
    *_rows("wgrad-concat-1x1", 32, 16, 16, 96, 32, 96, 1, "generic wgrad, concat with pad64(c2) % bn != 0",
           {"wgrad": WGRAD}),
    *_rows("5x5", 3, 16, 16, 72, 0, 96, 5, "5x5, off-grid channels", {"fprop": SPLITK, "dgrad": SPLITK, "wgrad": WGRAD}),
    *_rows("7x7-bni2-partial", 3, 8, 8, 64, 0, 64, 7, "7x7 with a partial bni = 2 tile",
           {"fprop": SPLITK, "dgrad": SPLITK, "wgrad": WGRAD}),
    *_rows("7x7-32x128", 2, 32, 128, 8, 0, 64, 7, "7x7 on a non-square image, 8 input channels",
           {"fprop": SPLITK, "dgrad": SPLITK, "wgrad": WGRAD}),
    *_rows("7x7-32x128-plain", 3, 32, 128, 8, 0, 64, 7, "7x7 with 96 pixel tiles: the plain kernel",
           {"fprop": CONV, "dgrad": CONV}),
]


# ------------------------------------------------------------------------------------------------ operands and reference
def pack_cols(t, c1, c2):
    """[..., c1 + c2] -> [..., pad64(c1) + pad64(c2)]: each source's channels at its 64-aligned offset, zeros between
    (the packed weight and weight-gradient layout)."""
    p1 = pad64(c1)
    out = t.new_zeros(*t.shape[:-1], p1 + (pad64(c2) if c2 else 0))
    out[..., :c1] = t[..., :c1]
    out[..., p1:p1 + c2] = t[..., c1:]
    return out


def poisoned(t, before, after, ld):
    """t as a view into a NaN-filled buffer: `ld` elements per pixel, `before` / `after` images around it."""
    n, h, w, c = t.shape
    buf = torch.full((before + n + after, h, w, ld), float("nan"), dtype=t.dtype, device=t.device)
    view = buf[before:before + n, :, :, :c]
    view.copy_(t)
    return view


def operands(case, device, seed=0):
    """bf16 activations, bf16-exact fp32 weights, fp32 bias, bf16 residual and the fp32 wgrad prefill of one case,
    each placed in its poisoned buffer; `wpk` is the packed weight [cout, taps, kpad] with NaN rows after it."""
    g = torch.Generator(device=device).manual_seed(seed)

    def rnd(*shape, scale=1.0):
        return torch.randn(*shape, generator=g, device=device) * scale

    c, taps, box = case, case.k * case.k, case.box_images
    act = lambda ch: poisoned(rnd(c.n, c.h, c.w, ch).to(BF16), 1, box, pad64(ch) + 8)
    t = {"w": rnd(c.cout, c.c1 + c.c2, c.k, c.k, scale=(taps * (c.c1 + c.c2)) ** -0.5).to(BF16).float()}
    wbuf = torch.full((c.cout + 64, taps, c.kpad), float("nan"), dtype=BF16, device=device)
    t["wpk"] = wbuf[:c.cout]
    t["wpk"].copy_(pack_cols(t["w"].permute(0, 2, 3, 1).reshape(c.cout, taps, -1), c.c1, c.c2))
    t["x1"] = act(c.c1) if c.op != "dgrad" else None
    t["x2"] = act(c.c2) if c.op != "dgrad" and c.c2 else None
    t["dy"] = act(c.cout) if c.op != "fprop" else None
    t["bias"] = None
    if c.bias:
        bbuf = torch.full((c.cols + 32,), float("nan"), device=device)
        t["bias"] = bbuf[16:16 + c.cols]
        t["bias"].copy_(rnd(c.cols, scale=0.5))
    t["res"] = poisoned(rnd(c.n, c.h, c.w, c.cols).to(BF16), 1, box, c.cols + 20) if c.residual else None
    t["prefill"] = rnd(c.cout, taps, c.kpad) if c.op == "wgrad" else None
    return t


def reference(case, t, dtype=F64):
    """(ref, S) in the kernel's output layout, computed in `dtype` from the case's operands; S is the same operation on
    absolute values (only meaningful in fp64)."""
    c, pad = case, case.k // 2
    nchw = lambda x: x.to(dtype).permute(0, 3, 1, 2)
    nhwc = lambda y: y.permute(0, 2, 3, 1)
    w = t["w"].to(dtype)
    x = None
    if c.op != "dgrad":
        x = nchw(t["x1"]) if t["x2"] is None else torch.cat([nchw(t["x1"]), nchw(t["x2"])], 1)
    if c.op == "fprop":
        ref = nhwc(F.conv2d(x, w, padding=pad)) * c.alpha
        s = nhwc(F.conv2d(x.abs(), w.abs(), padding=pad)) * abs(c.alpha)
    elif c.op == "dgrad":
        dy = nchw(t["dy"])
        ref = nhwc(F.conv_transpose2d(dy, w, padding=pad)) * c.alpha
        s = nhwc(F.conv_transpose2d(dy.abs(), w.abs(), padding=pad)) * abs(c.alpha)
        if c.c2:
            ref, s = pack_cols(ref, c.c1, c.c2), pack_cols(s, c.c1, c.c2)
    else:
        dy, pre = nchw(t["dy"]), t["prefill"].to(dtype)
        grads = [torch.nn.grad.conv2d_weight(a, w.shape, b, padding=pad) for a, b in [(x, dy), (x.abs(), dy.abs())]]
        ref, s = (pack_cols(gw.permute(0, 2, 3, 1).reshape(c.cout, c.k * c.k, -1), c.c1, c.c2) for gw in grads)
        ref, s = pre + ref, pre.abs() + s
    if t["bias"] is not None:
        ref, s = ref + t["bias"].to(dtype), s + t["bias"].to(dtype).abs()
    if t["res"] is not None:
        ref, s = ref + t["res"].to(dtype), s + t["res"].to(dtype).abs()
    return ref, s


def reduction_length(case):
    taps = case.k * case.k
    if case.op == "fprop":
        return taps * case.kpad
    if case.op == "dgrad":
        return taps * pad64(case.cout)
    return case.n * case.h * case.w


def partial_sums(case):
    if case.op == "wgrad":
        return 64  # the cap of pick_wgrad_split: the split the kernel picks is not observable
    if case.kernel == SPLITK:
        return int(case.force.split(",")[1]) if case.force else 4  # the forced split, or the cap of pick_splitk
    return 1


# ------------------------------------------------------------------------------------------------ guarded output, checker
def guarded_output(case, t):
    """(buf, view, writable): the output `view` inside a guard buffer, and the mask of the elements a kernel may change.
    fprop / dgrad: sentinel-filled, GUARD_COLS extra channels and a pixel box of images on either side.  wgrad: the
    prefill, with one guard row on either side; the pad columns of the packed layout are not writable."""
    c = case
    dev = t["w"].device
    if c.op == "wgrad":
        row = c.k * c.k * c.kpad
        g = torch.Generator(device=dev).manual_seed(1)
        buf = torch.randn((c.cout + 2) * row, generator=g, device=dev)
        view = buf[row:row + c.cout * row].view(c.cout, c.k * c.k, c.kpad)
        view.copy_(t["prefill"])
        writable = torch.zeros(buf.shape, dtype=torch.bool, device=dev)
        wv = writable[row:row + c.cout * row].view(c.cout, c.k * c.k, c.kpad)
        wv[..., :c.c1] = True
        wv[..., pad64(c.c1):pad64(c.c1) + c.c2] = True
        return buf, view, writable
    b = c.box_images
    buf = torch.full((b + c.n + b, c.h, c.w, c.cols + GUARD_COLS[c.out_dtype]), SENTINEL, dtype=c.out_dtype, device=dev)
    writable = torch.zeros(buf.shape, dtype=torch.bool, device=dev)
    writable[b:b + c.n, ..., :c.cols] = True
    return buf, buf[b:b + c.n, ..., :c.cols], writable


def _bits(x):
    return x.view({BF16: torch.int16, F32: torch.int32}[x.dtype])


def verify(case, before, buf, view, writable, ref, s):
    """Problems (strings) of one result, and the largest |got - ref| / bound over the output."""
    problems = []
    stray = (_bits(before) != _bits(buf)) & ~writable
    if stray.any():
        idx = stray.nonzero()[:4].tolist()
        problems.append(f"{int(stray.sum())} elements outside the output changed, e.g. at {idx}")
    got = view.to(F64)
    if torch.isnan(got).any():
        problems.append(f"{int(torch.isnan(got).sum())} NaN outputs")
    bound = (math.ceil(reduction_length(case) / 16) + partial_sums(case) + 2) * 2.0 ** -23 * s
    if case.out_dtype == BF16:
        bound = bound + 2.0 ** -8 * ref.abs()
    err = (got - ref).abs()
    bad = ~(err <= bound)
    ratio = torch.where(bound > 0, err / bound, torch.where(err > 0, math.inf, 0.0))
    worst = float(ratio.nan_to_num(math.inf).max())
    if bad.any():
        i = tuple(bad.nonzero()[0].tolist())
        problems.append(f"{int(bad.sum())} of {bad.numel()} elements outside the bound, first at {i}: got "
                        f"{float(got[i])}, ref {float(ref[i])}, bound {float(bound[i]):.3g}; max err/bound {worst:.3g}")
    return problems, worst


# ------------------------------------------------------------------------------------------------ GPU: the table
def _device_ready():
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert sms == B200_SMS, (f"the kernel each case must reach is worked out for the {B200_SMS} SMs of a B200; "
                             f"this device has {sms}")
    from adm_b200 import _lib, ops
    return _lib.load(), ops


def _kernels_of(fn):
    """Names of the CUDA kernels fn launches, as recorded by torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        try:
            fn()
        finally:
            torch.cuda.synchronize()
    return [ev.name.split("(")[0].replace("void ", "").replace("adm::", "").strip()
            for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]


def _call(case, t, ops, out):
    if case.op == "fprop":
        return lambda: ops.conv_fprop(t["x1"], t["wpk"], x2=t["x2"], bias=t["bias"], residual=t["res"],
                                      alpha=case.alpha, out=out)
    if case.op == "dgrad":
        return lambda: ops.conv_dgrad(t["dy"], t["wpk"], n_valid=case.cols, residual=t["res"], alpha=case.alpha,
                                      out=out)
    return lambda: ops.conv_wgrad(t["dy"], t["x1"], x2=t["x2"], ntaps=case.k * case.k, out=out)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_conv_path(case, monkeypatch):
    lib, ops = _device_ready()
    if case.force:
        monkeypatch.setenv(FORCE, case.force)
    else:
        monkeypatch.delenv(FORCE, raising=False)
    t = operands(case, "cuda")
    buf, view, writable = guarded_output(case, t)
    before = buf.clone()
    launches = lib.adm_launch_count()
    ran = _kernels_of(_call(case, t, ops, view))
    assert ran == [case.kernel], f"{case.id} ({case.edge}) ran {ran}, expected [{case.kernel}]"
    assert lib.adm_launch_count() == launches + 1
    assert lib.adm_device_error() == 0
    ref, s = reference(case, t)
    problems, worst = verify(case, before, buf, view, writable, ref, s)
    print(f"{case.id}: {case.kernel}, max |err| / bound = {worst:.3g}")
    assert not problems, f"{case.id} ({case.edge}): " + "; ".join(problems)


@pytest.mark.gpu
@pytest.mark.parametrize("op", ["fprop", "dgrad", "wgrad"])
def test_unsupported_geometry_is_an_error(op):
    """12 x 8 images tile neither into a 128-pixel box nor into the halo's 8 x 16: a shape error, nothing launched."""
    lib, ops = _device_ready()
    from adm_b200._lib import AdmError
    case = Case("12x8", op, 2, 12, 8, 64, 0, 64, 3, None, "unsupported geometry")
    t = operands(case, "cuda")
    buf, view, _ = guarded_output(case, t)
    before = buf.clone()
    launches = lib.adm_launch_count()

    def attempt():
        with pytest.raises(AdmError, match="unsupported H x W = 12 x 8"):
            _call(case, t, ops, view)()

    assert _kernels_of(attempt) == [] and lib.adm_launch_count() == launches
    assert lib.adm_device_error() == 0
    assert torch.equal(_bits(buf), _bits(before))


# ------------------------------------------------------------------------------------------------ CPU: the checker's teeth
# Reduced versions of three table geometries.  The "kernel" here is a candidate result written into the guarded output.
HALO_LIKE = Case("halo-like", "fprop", 2, 16, 8, 96, 0, 32, 3, HALO, "halo tile, off-grid channels", bias=True)
PARTIAL = Case("partial-tile", "fprop", 3, 4, 4, 64, 0, 48, 3, SPLITK, "partial bni = 8 tile", out=F32, bias=True,
               residual=True, alpha=-0.75)
TAP_ROW = Case("tap-row", "wgrad", 2, 8, 64, 64, 0, 64, 3, ROWS, "64-pixel K boxes")


def _judge(case, t, write, ref_s=None):
    """Problems of the result that `write(view)` leaves in a fresh guarded output."""
    buf, view, writable = guarded_output(case, t)
    before = buf.clone()
    write(buf, view)
    ref, s = ref_s or reference(case, t)
    return verify(case, before, buf, view, writable, ref, s)[0]


def _store(x):
    return lambda buf, view: view.copy_(x)


@pytest.mark.parametrize("case", [HALO_LIKE, PARTIAL, TAP_ROW], ids=lambda c: c.name)
def test_checker_accepts_rounded_reference_and_fp32_convolution(case):
    t = operands(case, "cpu")
    ref, _ = reference(case, t)
    assert _judge(case, t, _store(ref.to(case.out_dtype))) == []
    # another summation order: fp32 CPU convolution of the same operands
    assert _judge(case, t, _store(reference(case, t, F32)[0].to(case.out_dtype))) == []


def test_checker_rejects_missing_channel_chunk_of_one_tap():
    t = operands(HALO_LIKE, "cpu")
    w = t["w"].clone()
    w[:, :64, 1, 1] = 0  # first 64-channel chunk of the centre tap
    mutant = reference(HALO_LIKE, {**t, "w": w})[0]
    assert _judge(HALO_LIKE, t, _store(mutant.to(BF16)))


def test_checker_rejects_missing_last_image_of_partial_tile():
    t = operands(PARTIAL, "cpu")
    ref = reference(PARTIAL, t)[0].to(F32)
    assert _judge(PARTIAL, t, lambda buf, view: view[:-1].copy_(ref[:-1]))


def test_checker_rejects_column_chunk_shifted_by_one():
    t = operands(HALO_LIKE, "cpu")
    mutant = reference(HALO_LIKE, t)[0].to(BF16)
    mutant[..., 16:32] = mutant[..., 15:31].clone()
    assert _judge(HALO_LIKE, t, _store(mutant))


def test_checker_rejects_cross_image_halo_leak():
    """The taps above row 0 of image i read the last row of image i - 1 instead of the zero padding."""
    t = operands(HALO_LIKE, "cpu")
    c = HALO_LIKE
    x = t["x1"].to(F64).permute(0, 3, 1, 2)
    leak = torch.zeros(c.n, c.c1, c.h + 2, c.w + 2, dtype=F64)
    leak[1:, :, 0, 1:-1] = x[:-1, :, -1, :]
    ref = reference(c, t)[0]
    mutant = ref + F.conv2d(leak, t["w"].to(F64)).permute(0, 2, 3, 1) * c.alpha
    assert _judge(c, t, _store(mutant.to(BF16)))


def test_checker_rejects_wgrad_missing_one_k_box():
    t = operands(TAP_ROW, "cpu")
    x1 = t["x1"].clone()
    x1[1, 3] = 0  # one image row = one 64-pixel K box of the tap-row kernel
    mutant = reference(TAP_ROW, {**t, "x1": x1})[0]
    assert _judge(TAP_ROW, t, _store(mutant.to(F32)))


def test_checker_rejects_write_one_column_past_n():
    t = operands(PARTIAL, "cpu")
    ref = reference(PARTIAL, t)[0].to(F32)

    def write(buf, view):
        view.copy_(ref)
        b = PARTIAL.box_images
        buf[b + 2, 3, 1, PARTIAL.cols] = ref[2, 3, 1, -1]

    assert _judge(PARTIAL, t, write)


def test_cases_cover_every_kernel_of_every_op():
    ran = {(c.op, c.kernel) for c in CASES}
    assert ran == {(op, k) for op in ("fprop", "dgrad") for k in (HALO, SPLITK, CONV)} | {("wgrad", ROWS),
                                                                                          ("wgrad", WGRAD)}
    assert len({c.id for c in CASES}) == len(CASES)
