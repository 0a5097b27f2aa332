"""EDM-style augmentation pipe for the CIFAR-10 DDM config (``use_augment: True``).

Role of /root/reference/ddm/augment.py (``AugmentPipe`` :115-328) as the reference instantiates it
(ddm/ddm_const.py:179-180: ``AugmentPipe(p=0.15, xflip=1e8, yflip=1, scale=1, rotate_frac=1, aniso=1, translate_frac=1)``):
random x / y flips and ONE anti-aliased affine warp (isotropic scale, rotation, anisotropic scale, sub-pixel translation
composed into a single inverse matrix), returning the augmented batch and the 9 conditioning labels
``[xflip, yflip, scale, cos(rot) - 1, sin(rot), aniso * cos(r), aniso * sin(r), tx, ty]`` that enter the UNet through
``map_augment`` (unet/uncond_unet.py:548-549).

The random decisions (a few scalars per sample) are drawn on the host from the global torch RNG in the reference's order, so
with the same seed it reproduces the reference's augmented batch (tests/golden/make_golden_augment.py records one;
tests/test_host.py compares).  CUDA batches then run flips + the whole warp as ONE sm_100a kernel (``adm_augment_warp``,
SURVEY section 8 row f-4: one CTA per sample, nothing but the 32 x 32 image and the sampled grid in shared memory); CPU
tensors (and ``fused = False``) run the same arithmetic as ordinary torch ops (SURVEY row a-4).
Only what the DDM configs use is implemented; integer rotation / translation and the colour transforms (all disabled in
ddm_const.py:179-180) raise.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

# sym6 wavelet low-pass filter (PyWavelets 'sym6' decomposition low-pass), the anti-aliasing kernel of the warp
SYM6 = (0.015404109327027373, 0.0034907120842174702, -0.11799011114819057, -0.048311742585633, 0.4910559419267466,
        0.787641141030194, 0.3379294217276218, -0.07263752278646252, -0.021060292512300564, 0.04472490177066578,
        0.0017677118642428036, -0.007800708325034148)


def _affine(rows, like):
    """[N, 3, 3] matrices from a 3x3 nest of python scalars / [N] tensors."""
    n = like.shape[0]
    cols = [e if torch.is_tensor(e) else torch.full((n,), float(e), device=like.device, dtype=like.dtype)
            for r in rows for e in r]
    return torch.stack(cols, dim=-1).reshape(n, 3, 3)


def _scale(sx, sy, like):
    return _affine([[sx, 0, 0], [0, sy, 0], [0, 0, 1]], like)


def _rot(theta, like):
    c, s = torch.cos(theta), torch.sin(theta)
    return _affine([[c, -s, 0], [s, c, 0], [0, 0, 1]], like)


def _shift(tx, ty, like):
    return _affine([[1, 0, tx], [0, 1, ty], [0, 0, 1]], like)


class AugmentPipe:
    def __init__(self, p=1, xflip=0, yflip=0, rotate_int=0, translate_int=0, translate_int_max=0.125, scale=0,
                 rotate_frac=0, aniso=0, translate_frac=0, scale_std=0.2, rotate_frac_max=1, aniso_std=0.2,
                 aniso_rotate_prob=0.5, translate_frac_std=0.125, brightness=0, contrast=0, lumaflip=0, hue=0,
                 saturation=0, **unused):
        if any(float(v) > 0 for v in (rotate_int, translate_int, brightness, contrast, lumaflip, hue, saturation)):
            raise NotImplementedError("adm_b200 AugmentPipe: only flips and the fractional geometric warp are implemented "
                                      "(everything the DDM configs enable, ddm_const.py:179-180)")
        self.p = float(p)
        self.xflip, self.yflip = float(xflip), float(yflip)
        self.scale, self.rotate_frac, self.aniso, self.translate_frac = (float(scale), float(rotate_frac), float(aniso),
                                                                         float(translate_frac))
        self.scale_std, self.rotate_frac_max, self.aniso_std = float(scale_std), float(rotate_frac_max), float(aniso_std)
        self.aniso_rotate_prob, self.translate_frac_std = float(aniso_rotate_prob), float(translate_frac_std)
        # CUDA batches run flips + warp as ONE kernel (adm_augment_warp); fused = False keeps the torch-op sequence below
        # (the same arithmetic, ~40 launches), which is also what runs on CPU tensors
        self.fused = True

    # ------------------------------------------------------------------------------------------ random parameters
    def draw(self, n, h, w, device):
        """The random decisions of one call, in the reference's RNG order.  Returns (flip_x [N] bool, flip_y [N] bool,
        inverse warp matrix [N, 3, 3] or None, labels [N, 9-ish])."""
        def gate(prob, shape):
            return torch.rand(shape, device=device) < prob * self.p

        labels, fx, fy = [], None, None
        if self.xflip > 0:
            wv = torch.randint(2, [n, 1, 1, 1], device=device)
            wv = torch.where(gate(self.xflip, [n, 1, 1, 1]), wv, torch.zeros_like(wv))
            fx = wv.reshape(n) == 1
            labels.append(wv.reshape(n, 1).float())
        if self.yflip > 0:
            wv = torch.randint(2, [n, 1, 1, 1], device=device)
            wv = torch.where(gate(self.yflip, [n, 1, 1, 1]), wv, torch.zeros_like(wv))
            fy = wv.reshape(n) == 1
            labels.append(wv.reshape(n, 1).float())
        like = torch.zeros(n, device=device)
        g_inv = None
        if self.scale > 0:
            wv = torch.randn([n], device=device)
            wv = torch.where(gate(self.scale, [n]), wv, torch.zeros_like(wv))
            s = (wv * self.scale_std).exp2()
            g_inv = _scale(1 / s, 1 / s, like)
            labels.append(wv.reshape(n, 1))
        if self.rotate_frac > 0:
            wv = (torch.rand([n], device=device) * 2 - 1) * (math.pi * self.rotate_frac_max)
            wv = torch.where(gate(self.rotate_frac, [n]), wv, torch.zeros_like(wv))
            m = _rot(wv, like)  # the reference's rotate2d_inv(-w) = rotate2d(w)
            g_inv = m if g_inv is None else g_inv @ m
            labels += [(wv.cos() - 1).reshape(n, 1), wv.sin().reshape(n, 1)]
        if self.aniso > 0:
            wv = torch.randn([n], device=device)
            r = (torch.rand([n], device=device) * 2 - 1) * math.pi
            wv = torch.where(gate(self.aniso, [n]), wv, torch.zeros_like(wv))
            r = torch.where(torch.rand([n], device=device) < self.aniso_rotate_prob, r, torch.zeros_like(r))
            s = (wv * self.aniso_std).exp2()
            m = _rot(-r, like) @ _scale(1 / s, s, like) @ _rot(r, like)
            g_inv = m if g_inv is None else g_inv @ m
            labels += [(wv * r.cos()).reshape(n, 1), (wv * r.sin()).reshape(n, 1)]
        if self.translate_frac > 0:
            wv = torch.randn([2, n], device=device)
            wv = torch.where(gate(self.translate_frac, [1, n]), wv, torch.zeros_like(wv))
            m = _shift(-wv[0] * (w * self.translate_frac_std), -wv[1] * (h * self.translate_frac_std), like)
            g_inv = m if g_inv is None else g_inv @ m
            labels += [wv[0].reshape(n, 1), wv[1].reshape(n, 1)]
        lab = torch.cat(labels, dim=1) if labels else torch.zeros(n, 0, device=device)
        return fx, fy, g_inv, lab

    # ------------------------------------------------------------------------------------------ the warp
    @staticmethod
    def warp(images, g_inv):
        """Anti-aliased affine warp: reflect-pad by the margin the transformed corners need, 2x upsample with the sym6
        low-pass, bilinear sample through g_inv, sym6 low-pass + 2x decimate, crop (ddm/augment.py:236-271)."""
        n, c, h, w = images.shape
        dev = g_inv.device
        taps = torch.tensor(SYM6, dtype=torch.float32, device=dev)
        pad4 = len(SYM6) // 4
        cx, cy = (w - 1) / 2, (h - 1) / 2
        corners = torch.tensor([[-cx, -cy, 1], [cx, -cy, 1], [cx, cy, 1], [-cx, cy, 1]], device=dev, dtype=g_inv.dtype)
        moved = g_inv @ corners.t()  # [N, 3, 4]
        ext = moved[:, :2, :].permute(1, 0, 2).flatten(1)  # [xy, N*4]
        ext = torch.cat([-ext, ext]).max(dim=1).values  # [x0, y0, x1, y1]
        ext = ext + torch.tensor([pad4 * 2 - cx, pad4 * 2 - cy] * 2, device=dev, dtype=ext.dtype)
        ext = ext.clamp(min=0).min(torch.tensor([w - 1, h - 1] * 2, device=dev, dtype=ext.dtype))
        # batch-wide padding: a host value.  g_inv lives on the host when the parameters were drawn there (CUDA batches), so
        # this does not wait for the device
        mx0, my0, mx1, my1 = (int(v) for v in ext.ceil().to(torch.int32).tolist())
        g_inv = g_inv.to(images.device, non_blocking=True)
        dev = images.device
        taps = taps.to(dev)
        images = F.pad(images, [mx0, mx1, my0, my1], mode="reflect")
        like = g_inv[:, 0, 0]
        g_inv = _shift((mx0 - mx1) / 2, (my0 - my1) / 2, like) @ g_inv
        # 2x upsample: zero-stuff, then the (flipped) low-pass along x and along y
        k_up = taps.flip(0)[None, None, :].repeat(c, 1, 1)
        up_pad = (len(SYM6) + 1) // 2
        images = torch.stack([images, torch.zeros_like(images)], dim=4).reshape(n, c, images.shape[2], -1)[:, :, :, :-1]
        images = F.conv2d(images, k_up.unsqueeze(2), groups=c, padding=[0, up_pad])
        images = torch.stack([images, torch.zeros_like(images)], dim=3).reshape(n, c, -1, images.shape[3])[:, :, :-1, :]
        images = F.conv2d(images, k_up.unsqueeze(3), groups=c, padding=[up_pad, 0])
        two, half = _scale(2, 2, like), _scale(0.5, 0.5, like)
        g_inv = two @ g_inv @ half
        g_inv = _shift(-0.5, -0.5, like) @ g_inv @ _shift(0.5, 0.5, like)
        # sample on the (h + 2 pad4) * 2 grid in normalised coordinates
        out_h, out_w = (h + pad4 * 2) * 2, (w + pad4 * 2) * 2
        g_inv = _scale(2 / images.shape[3], 2 / images.shape[2], like) @ g_inv @ _scale(out_w / 2, out_h / 2, like)
        grid = F.affine_grid(theta=g_inv[:, :2, :], size=[n, c, out_h, out_w], align_corners=False)
        images = F.grid_sample(images, grid, mode="bilinear", padding_mode="zeros", align_corners=False)
        # low-pass + decimate + crop
        k_dn = taps[None, None, :].repeat(c, 1, 1)
        dn_pad = (len(SYM6) - 1) // 2
        images = F.conv2d(images, k_dn.unsqueeze(2), groups=c, stride=[1, 2], padding=[0, dn_pad])[:, :, :, pad4:-pad4]
        images = F.conv2d(images, k_dn.unsqueeze(3), groups=c, stride=[2, 1], padding=[dn_pad, 0])[:, :, pad4:-pad4, :]
        return images

    # ------------------------------------------------------------------------------------------ the warp, one kernel
    @staticmethod
    def warp_plan(g_inv, h, w):
        """Host side of the warp (a few floats per sample): the batch-wide reflect margins (:245-250) and the 2 x 3 matrix
        the reference hands to affine_grid (:252-266) — the same compositions as ``warp`` above, on the host tensors."""
        n = g_inv.shape[0]
        pad4 = len(SYM6) // 4
        cx, cy = (w - 1) / 2, (h - 1) / 2
        corners = torch.tensor([[-cx, -cy, 1], [cx, -cy, 1], [cx, cy, 1], [-cx, cy, 1]], dtype=g_inv.dtype)
        moved = g_inv @ corners.t()
        ext = moved[:, :2, :].permute(1, 0, 2).flatten(1)
        ext = torch.cat([-ext, ext]).max(dim=1).values
        ext = ext + torch.tensor([pad4 * 2 - cx, pad4 * 2 - cy] * 2, dtype=ext.dtype)
        ext = ext.clamp(min=0).min(torch.tensor([w - 1, h - 1] * 2, dtype=ext.dtype))
        mx0, my0, mx1, my1 = (int(v) for v in ext.ceil().to(torch.int32).tolist())
        like = g_inv[:, 0, 0]
        g = _shift((mx0 - mx1) / 2, (my0 - my1) / 2, like) @ g_inv
        g = _scale(2, 2, like) @ g @ _scale(0.5, 0.5, like)
        g = _shift(-0.5, -0.5, like) @ g @ _shift(0.5, 0.5, like)
        wu, hu = 2 * (w + mx0 + mx1), 2 * (h + my0 + my1)
        out_h, out_w = (h + pad4 * 2) * 2, (w + pad4 * 2) * 2
        g = _scale(2 / wu, 2 / hu, like) @ g @ _scale(out_w / 2, out_h / 2, like)
        return (mx0, mx1, my0, my1), g[:, :2, :].reshape(n, 6).to(torch.float32).contiguous()

    @staticmethod
    def fused_ok(images):
        if not images.is_cuda or images.dtype != torch.float32 or images.shape[1] > 4:
            return False
        from .. import _lib
        n, c, h, w = images.shape
        return _lib.load().adm_augment_warp_smem(c, h, w) <= 200 * 1024

    def warp_fused(self, images, fx, fy, g_inv):
        """Flips + the whole anti-aliased warp as ONE sm_100a kernel (adm_augment_warp, one CTA per sample)."""
        from .. import ops
        n, c, h, w = images.shape
        margins, theta = self.warp_plan(g_inv, h, w)
        flips = torch.zeros(n, 2, dtype=torch.int32)
        if fx is not None:
            flips[:, 0] = fx.to(torch.int32)
        if fy is not None:
            flips[:, 1] = fy.to(torch.int32)
        dev = images.device
        return ops.augment_warp(images.contiguous(), theta.to(dev, non_blocking=True), flips.to(dev, non_blocking=True),
                                margins)

    def __call__(self, images):
        n, c, h, w = images.shape
        # The random decisions are a few scalars per sample: they are drawn on the HOST (also for CUDA batches), so that
        # the batch-wide padding of the warp is known without synchronising with the device.
        fx, fy, g_inv, labels = self.draw(n, h, w, torch.device("cpu"))
        dev = images.device
        if g_inv is not None and self.fused and self.fused_ok(images):
            return self.warp_fused(images, fx, fy, g_inv), labels.to(dev, torch.float32, non_blocking=True)
        if fx is not None:
            images = torch.where(fx.to(dev, non_blocking=True).reshape(n, 1, 1, 1), images.flip(3), images)
        if fy is not None:
            images = torch.where(fy.to(dev, non_blocking=True).reshape(n, 1, 1, 1), images.flip(2), images)
        if g_inv is not None:
            images = self.warp(images, g_inv)
        return images, labels.to(dev, torch.float32, non_blocking=True)
