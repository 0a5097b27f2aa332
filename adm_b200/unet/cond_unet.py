"""B200-native mirror of /root/reference/unet/cond_unet.py: the conditional two-decoder ``Unet`` of the latent
super-resolution config (configs/super-resolution/div2k_cond_ddm_const_ldm.yaml).  Same class names, constructor
arguments and ``state_dict`` layout as the reference (``Unet`` :592-793, forward :823-917).

Execution model: the module graph is ordinary ``nn.Module``s driven by torch autograd, activations travel as NHWC bf16
tensors, and every hot op is one of the hand-written sm_100a kernels through ``adm_b200.functional``:

  * ``ResnetBlock`` / ``Block`` / ``WeightStandardizedConv2d`` (:345-358, :427-469): K11 weight-standardise+pack, tcgen05
    implicit-GEMM conv3x3 (fprop / dgrad / wgrad), fused GroupNorm + (1+scale)/shift + SiLU;
  * ``LinearAttention`` (:503-531): K12 fused two-softmax linear attention; ``Attention`` (:533-555): tcgen05 batched
    GEMMs + fused softmax with the head dim zero-padded 32 -> 64 inside the projection weights;
  * ``SpatialAtt`` + residual (:119-137, :871-872), 1x1 / 3x3 ``nn.Conv2d`` of the trunk, ``nn.GroupNorm``.

Left to PyTorch (SURVEY §8 f-3, "next" rows): the Swin-B condition encoder (built from torchvision's blocks under the
reference's attribute names), ``RelationNet`` / ``BasicAttetnionLayer``, the 7x7 stem conv, the 4x4 stride-2
``Downsample`` conv, bilinear / nearest resampling and the time MLP.  They run under bf16 autocast on the same tensors.
There is no CPU fallback: the kernels raise on non-CUDA tensors.
"""
from __future__ import annotations

import math
from functools import partial

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import functional as AF
from .. import ops


def exists(x):
    return x is not None


def default(val, d):
    if exists(val):
        return val
    return d() if callable(d) else d


def _nchw(x):  # NHWC tensor -> logical NCHW view (channels_last strides, no copy)
    return x.permute(0, 3, 1, 2)


def _nhwc(x):  # logical NCHW tensor -> NHWC bf16 contiguous
    return x.permute(0, 2, 3, 1).to(torch.bfloat16).contiguous()


# ------------------------------------------------------------------------------------------------ condition-side helpers
class PositionEmbeddingSine(nn.Module):
    """cond_unet.py:16-64 — sine/cosine position code added to the pooled query / key windows ([B, H, W, D] in, same out)."""

    def __init__(self, num_pos_feats=64, temperature=10000, normalize=False, scale=None):
        super().__init__()
        if scale is not None and normalize is False:
            raise ValueError("normalize should be True if scale is passed")
        self.num_pos_feats, self.temperature, self.normalize = num_pos_feats, temperature, normalize
        self.scale = 2 * math.pi if scale is None else scale

    def forward(self, x):
        b, h, w, d = x.shape
        half = d // 2
        ys = torch.arange(1, h + 1, dtype=torch.float32, device=x.device).view(1, h, 1).expand(b, h, w)
        xs = torch.arange(1, w + 1, dtype=torch.float32, device=x.device).view(1, 1, w).expand(b, h, w)
        if self.normalize:
            ys = ys / (h + 1e-5) * self.scale
            xs = xs / (w + 1e-5) * self.scale
        idx = torch.arange(half, dtype=torch.float32, device=x.device)
        div = self.temperature ** (2 * torch.div(idx, 2, rounding_mode="floor") / half)
        px, py = xs[..., None] / div, ys[..., None] / div
        px = torch.stack((px[..., 0::2].sin(), px[..., 1::2].cos()), dim=4).flatten(3)
        py = torch.stack((py[..., 0::2].sin(), py[..., 1::2].cos()), dim=4).flatten(3)
        return torch.cat((py, px), dim=3).contiguous()


class PositionEmbeddingLearned(nn.Module):
    """cond_unet.py:66-90 (only built when cond_pe is set)."""

    def __init__(self, feature_size, num_pos_feats=256):
        super().__init__()
        self.row_embed = nn.Embedding(feature_size[0], num_pos_feats)
        self.col_embed = nn.Embedding(feature_size[1], num_pos_feats)
        nn.init.uniform_(self.row_embed.weight)
        nn.init.uniform_(self.col_embed.weight)

    def forward(self, x):
        h, w = x.shape[-2:]
        xe = self.col_embed(torch.arange(w, device=x.device))
        ye = self.row_embed(torch.arange(h, device=x.device))
        pos = torch.cat([xe.unsqueeze(0).repeat(h, 1, 1), ye.unsqueeze(1).repeat(1, w, 1)], dim=-1)
        pos = pos.permute(2, 0, 1).unsqueeze(0).repeat(x.shape[0], 1, 1, 1)
        return torch.cat([x, pos], dim=1)


class SpatialAtt(nn.Module):
    """cond_unet.py:119-137.  Parameter container; the arithmetic is the fused spatial_att kernel (see Unet.forward)."""

    def __init__(self, in_dim):
        super().__init__()
        self.map = nn.Conv2d(in_dim, 1, 1)
        self.q_conv = nn.Conv2d(1, 1, 1)
        self.k_conv = nn.Conv2d(1, 1, 1)
        self.activation = nn.Softsign()

    def scalars(self):
        return torch.cat([self.map.bias.reshape(1), self.q_conv.weight.reshape(1), self.q_conv.bias.reshape(1),
                          self.k_conv.weight.reshape(1), self.k_conv.bias.reshape(1)])

    def forward(self, h, res):
        """h, res NHWC bf16: softsign(att(h)) * h + res."""
        return AF.spatial_att(h, res, self.map.weight.reshape(-1), self.scalars())


class Mlp(nn.Module):
    """cond_unet.py:139-158."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.ReLU, drop=0.):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Conv2d(in_features, hidden_features, kernel_size=1)
        self.act = act_layer()
        self.fc2 = nn.Conv2d(hidden_features, out_features, kernel_size=1)
        self.drop = nn.Dropout(drop)

    def forward(self, x):
        return self.drop(self.fc2(self.drop(self.act(self.fc1(x)))))


def _init_like_reference(module):
    """cond_unet.py:184-197 (kaiming convs, xavier linears, unit norms)."""
    for m in module.modules():
        if isinstance(m, nn.Conv2d):
            nn.init.kaiming_normal_(m.weight)
            if m.bias is not None:
                nn.init.constant_(m.bias, 0.)
        elif isinstance(m, (nn.BatchNorm2d, nn.LayerNorm)):
            nn.init.constant_(m.weight, 1.)
            nn.init.constant_(m.bias, 0.)
        elif isinstance(m, nn.Linear):
            nn.init.xavier_normal_(m.weight)
            nn.init.constant_(m.bias, 0.)


def _pad_to(x, win):
    ph = (win[0] - x.shape[2] % win[0]) % win[0]
    pw = (win[1] - x.shape[3] % win[1]) % win[1]
    return F.pad(x, (0, pw, 0, ph)) if (ph or pw) else x


class BasicAttetnionLayer(nn.Module):
    """cond_unet.py:160-252: window-pooled cross attention from the condition map (queries) to the feature map
    (keys / values)."""

    def __init__(self, embed_dim=128, nhead=8, ffn_dim=512, window_size1=[4, 4], window_size2=[1, 1], dropout=0.1):
        super().__init__()
        self.window_size1, self.window_size2, self.nhead = window_size1, window_size2, nhead
        self.avgpool_q = nn.AvgPool2d(kernel_size=window_size1)
        self.avgpool_k = nn.AvgPool2d(kernel_size=window_size2)
        self.softmax = nn.Softmax(dim=-1)
        self.q_lin = nn.Linear(embed_dim, embed_dim)
        self.k_lin = nn.Linear(embed_dim, embed_dim)
        self.v_lin = nn.Linear(embed_dim, embed_dim)
        self.mlp = Mlp(in_features=embed_dim, hidden_features=ffn_dim, drop=dropout)
        self.pos_enc = PositionEmbeddingSine(embed_dim)
        self.concat_conv = nn.Conv2d(2 * embed_dim, embed_dim, 1)
        self.gn = nn.GroupNorm(8, embed_dim)
        self.out_conv = nn.Conv2d(embed_dim, embed_dim, 1)
        _init_like_reference(self)

    def forward(self, x1, x2, last=True):
        """x1 (condition features) and x2 (trunk features): NHWC bf16.  Everything at full resolution runs on the sm_100a
        kernels: the concat 1x1 conv on the GEMM engine, the window average pools, and — for the last layer of a stack
        (every layer of the shipped configs: layers = 1) — the whole tail ``GroupNorm(x2 + conv) + out_conv(up(pooled))``
        as one fused pass (``AF.relation_tail``): the 1x1 ``out_conv`` commutes with the bilinear resize (per-pixel
        linear map, resize weights sum to one), so it runs on the pooled tokens and the resize + residual GroupNorm is a
        single read of x2 / conv and a single bf16 write with the sum in fp32 registers.  The window-pooled cross
        attention itself (a few hundred tokens) stays torch ops.  With ``_REL_FUSED = False`` every layer runs the unfused
        tail (fp32 residual add + GroupNorm, bilinear resize, full-resolution out_conv) as torch ops."""
        b, _, _, c1 = x1.shape
        _, h2, w2, c2 = x2.shape
        gn = self.gn
        fused = (last and _REL_FUSED and x2.is_cuda and x2.dtype == torch.bfloat16 and c2 % 8 == 0
                 and ops.rel_gn_ok(x2, gn.num_groups))
        x2r = None if fused else x2.float()  # unfused: the residual stream of stacked relation layers stays fp32
        x2 = x2.to(torch.bfloat16)           # what the convs / pooling read
        up = _bilinear(x1, (h2, w2))
        y = _conv1x1(torch.cat([up.to(torch.bfloat16), x2], dim=-1), self.concat_conv)
        if fused:
            shortcut = None
        else:
            # fp32 GroupNorm on the channels-last view: the residual stream of the relation layer stays fp32 end to end, as
            # under the reference's fp32 arithmetic (with the bf16 GroupNorm kernel one Downsample weight gradient of the
            # golden check drops from cosine 0.9995 to 0.9983)
            pre = x2r + y.float()
            shortcut = F.group_norm(_nchw(pre), gn.num_groups, gn.weight, gn.bias, gn.eps).permute(0, 2, 3, 1)
        pooled = _window_pool(x1, self.window_size1, self.avgpool_q)  # [b, hq, wq, c]
        hq, wq = pooled.shape[1:3]
        q = (pooled + self.pos_enc(pooled).to(pooled.dtype)).reshape(b, -1, c2)
        k = _window_pool(x2, self.window_size2, self.avgpool_k)
        k = (k + self.pos_enc(k).to(k.dtype)).reshape(b, -1, c1)
        nq, nk, hd = q.shape[1], k.shape[1], c1 // self.nhead
        qh = self.q_lin(q).reshape(b, nq, self.nhead, hd).permute(0, 2, 1, 3)
        kh = self.k_lin(k).reshape(b, nk, self.nhead, hd).permute(0, 2, 1, 3)
        vh = self.v_lin(k).reshape(b, nk, self.nhead, hd).permute(0, 2, 1, 3)
        attn = self.softmax(qh @ kh.transpose(-2, -1))  # no 1/sqrt(d): as in the reference
        o = (attn @ vh).transpose(1, 2).reshape(b, hq, wq, c1)
        pooled = pooled + o.to(pooled.dtype)
        m = self.mlp
        hid = m.drop(m.act(F.linear(pooled, m.fc1.weight.flatten(1), m.fc1.bias)))  # the Mlp's 1x1 convs on [b, hq, wq, c]
        pooled = pooled + m.drop(F.linear(hid, m.fc2.weight.flatten(1), m.fc2.bias)).to(pooled.dtype)
        if fused:
            z = F.linear(pooled, self.out_conv.weight.flatten(1), self.out_conv.bias)  # out_conv on the pooled tokens
            return AF.relation_tail(x2, y, z, gn.weight, gn.bias, gn.num_groups, gn.eps)  # bf16
        pooled = _bilinear(pooled.to(torch.bfloat16).contiguous(), (h2, w2))
        return shortcut.float() + _conv1x1(pooled, self.out_conv).float()  # fp32 (rounded once, by RelationNet.forward)


_REL_FUSED = True


def _window_pool(x, window, pool):
    """F.pad to a multiple of the window + AvgPool2d on an NHWC map -> [b, ceil(h / kh), ceil(w / kw), c]."""
    if x.is_cuda and x.dtype == torch.bfloat16 and x.shape[-1] % 8 == 0:
        return AF.avg_pool_window(x, window)
    return pool(_pad_to(_nchw(x), window)).permute(0, 2, 3, 1)


def _bilinear(x, size):
    """NHWC -> NHWC bilinear resize (align_corners=True) through the channels-last view: no layout copy."""
    if tuple(x.shape[1:3]) == tuple(size):
        return x
    if x.is_cuda and x.dtype == torch.bfloat16 and x.shape[-1] % 8 == 0:
        return AF.bilinear_resize(x, size)
    y = F.interpolate(x.permute(0, 3, 1, 2), size=size, mode="bilinear", align_corners=True)
    return y.permute(0, 2, 3, 1).contiguous()


def _conv1x1(x, conv):
    """nn.Conv2d(k = 1) parameters on an NHWC bf16 tensor: the implicit-GEMM kernel where the image tiles, else a matmul."""
    x = x.to(torch.bfloat16)
    if _conv_tiles(x.shape[1], x.shape[2]) and x.shape[-1] % 8 == 0:
        return AF.conv2d(x.contiguous(), conv.weight, conv.bias)
    return F.linear(x, conv.weight.flatten(1).to(x.dtype), conv.bias.to(x.dtype) if conv.bias is not None else None)


class RelationNet(nn.Module):
    """cond_unet.py:254-280."""

    def __init__(self, in_channel1=128, in_channel2=128, nhead=8, layers=3, embed_dim=128, ffn_dim=512,
                 window_size1=[4, 4], window_size2=[1, 1]):
        super().__init__()
        self.layers = layers
        self.input_conv1 = nn.Sequential(nn.Conv2d(in_channel1, embed_dim, 1),
                                         nn.BatchNorm2d(embed_dim, momentum=0.03, eps=0.001))
        self.input_conv2 = nn.Sequential(nn.Conv2d(in_channel2, embed_dim, 1),
                                         nn.BatchNorm2d(embed_dim, momentum=0.03, eps=0.001))
        self.attentions = nn.ModuleList(
            BasicAttetnionLayer(embed_dim=embed_dim, nhead=nhead, ffn_dim=ffn_dim, window_size1=window_size1,
                                window_size2=window_size2, dropout=0.1) for _ in range(layers))

    def forward(self, cond, feat):
        """cond, feat: NHWC bf16.  1x1 conv on the kernels, BatchNorm on the channels-last view."""
        def stem(seq, x):
            y = seq[1](_nchw(_conv1x1(x, seq[0])))
            return y.permute(0, 2, 3, 1).to(torch.bfloat16).contiguous()
        cond, feat = stem(self.input_conv1, cond), stem(self.input_conv2, feat)
        for i, att in enumerate(self.attentions):
            feat = att(cond, feat, last=i == len(self.attentions) - 1)
        return feat.to(torch.bfloat16).contiguous()


# ------------------------------------------------------------------------------------------------ Swin-B condition encoder
class _Permute(nn.Module):
    def __init__(self, dims):
        super().__init__()
        self.dims = dims

    def forward(self, x):
        return x.permute(*self.dims)


class SwinTransformer(nn.Module):
    """unet/swin_transformer.py:308-426 assembled from torchvision's own ``SwinTransformerBlock`` / ``PatchMerging``
    under the reference's attribute names (``first_coonv``, ``features``, ``norm``, ``head``); forward returns the four
    stage feature maps as NCHW tensors (:412-426)."""

    def __init__(self, patch_size, embed_dim, depths, num_heads, window_size, mlp_ratio=4.0, dropout=0.0,
                 attention_dropout=0.0, stochastic_depth_prob=0.0, num_classes=1000, in_channels=3):
        super().__init__()
        from torchvision.models.swin_transformer import PatchMerging, SwinTransformerBlock
        norm_layer = partial(nn.LayerNorm, eps=1e-5)
        self.first_coonv = nn.Sequential(
            nn.Conv2d(in_channels, embed_dim, kernel_size=tuple(patch_size), stride=tuple(patch_size)),
            _Permute([0, 2, 3, 1]), norm_layer(embed_dim))
        layers, total, bid = [], sum(depths), 0
        for i_stage, depth in enumerate(depths):
            dim = embed_dim * 2 ** i_stage
            stage = []
            for i_layer in range(depth):
                sd = stochastic_depth_prob * float(bid) / (total - 1)
                stage.append(SwinTransformerBlock(dim, num_heads[i_stage], window_size=window_size,
                                                  shift_size=[0 if i_layer % 2 == 0 else w // 2 for w in window_size],
                                                  mlp_ratio=mlp_ratio, dropout=dropout,
                                                  attention_dropout=attention_dropout, stochastic_depth_prob=sd,
                                                  norm_layer=norm_layer))
                bid += 1
            layers.append(nn.Sequential(*stage))
            if i_stage < len(depths) - 1:
                layers.append(PatchMerging(dim, norm_layer))
        self.features = nn.ModuleList(layers)
        nf = embed_dim * 2 ** (len(depths) - 1)
        self.norm = norm_layer(nf)
        self.avgpool = nn.AdaptiveAvgPool2d(1)
        self.head = nn.Linear(nf, num_classes)
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.trunc_normal_(m.weight, std=0.02)
                if m.bias is not None:
                    nn.init.zeros_(m.bias)

    def forward(self, x):
        feats = []
        x = self.first_coonv(x)
        for i, layer in enumerate(self.features):
            x = layer(x)
            if i in (0, 2, 4, 6):
                feats.append(x.permute(0, 3, 1, 2).contiguous())
        return feats


def swin_b(in_channels=3, **kw):
    """swin_transformer.py:612-640 without the ImageNet download (weights come from the model checkpoint)."""
    return SwinTransformer(patch_size=[4, 4], embed_dim=128, depths=[2, 2, 18, 2], num_heads=[4, 8, 16, 32],
                           window_size=[7, 7], stochastic_depth_prob=0.5, in_channels=in_channels, **kw)


# ------------------------------------------------------------------------------------------------ trunk building blocks
class Residual(nn.Module):
    def __init__(self, fn):
        super().__init__()
        self.fn = fn

    def forward(self, x, *args, **kwargs):
        return self.fn(x, *args, **kwargs) + x


class _Conv(nn.Conv2d):
    """nn.Conv2d parameters (1x1 or 3x3, stride 1) executed by the tcgen05 implicit-GEMM engine on NHWC bf16."""

    def forward(self, x):
        return AF.conv2d(x, self.weight, self.bias)


class _Upsample(nn.Upsample):
    def forward(self, x):  # nearest x2 on NHWC
        return x.repeat_interleave(2, dim=1).repeat_interleave(2, dim=2)


def Upsample(dim, dim_out=None):
    """cond_unet.py:336-340."""
    return nn.Sequential(_Upsample(scale_factor=2, mode="nearest"), _Conv(dim, default(dim_out, dim), 3, padding=1))


# The PyTorch-side modules (Swin, RelationNet, stem / down convs: 7.5 % of the FLOPs) run in SIDE_DTYPE on the
# channels-last view of the trunk tensors: bf16 autocast (tensor-core cuDNN / cuBLAS) by default.  Measured against the
# reference's gradients (tests/gpu_checks/check_cond.py) bf16 and fp32 side modules give the same per-parameter cosines
# (min 0.99849 vs 0.99854, both on the mid-attention bias), while fp32 costs ~25 ms per B=16 step in SIMT sgemm.
SIDE_DTYPE = torch.bfloat16


def _side(x):
    return x if SIDE_DTYPE == torch.bfloat16 else x.to(SIDE_DTYPE)


class _DownConv(nn.Conv2d):
    """4x4 stride-2 padding-1 conv (cond_unet.py:342-343) on the implicit-GEMM engine: on the space-to-depth image
    X'[i, j, (p, q, c)] = x[2i + p, 2j + q, c] it is a 3x3 padding-1 conv — out[i, j] reads rows 2i - 1 .. 2i + 2, i.e.
    (i - 1, p = 1), (i, p = 0), (i, p = 1), (i + 1, p = 0) — whose weight W'[co, (p, q, c), di, dj] = w[co, c, 2 di + p + 1,
    2 dj + q + 1] (zero where that index leaves 0 .. 3: 16 of the 36 (tap, sub-pixel) pairs are live, 2.25 x the FLOPs of a
    conv that is 1.1 % of the network's).  The re-indexing of the weights is differentiable torch indexing."""

    def _s2d_weight(self):
        w = self.weight  # [co, c, 4, 4]
        co, c = w.shape[:2]
        zero = w.new_zeros(co, c)
        taps = []
        for di in (-1, 0, 1):
            for dj in (-1, 0, 1):
                sub = []
                for p in (0, 1):
                    for q in (0, 1):
                        a, b = 2 * di + p + 1, 2 * dj + q + 1
                        sub.append(w[:, :, a, b] if 0 <= a <= 3 and 0 <= b <= 3 else zero)
                taps.append(torch.stack(sub, dim=1))      # [co, 4 (p, q), c]
        return torch.stack(taps, dim=-1).reshape(co, 4 * c, 3, 3)  # [co, (p, q, c), di, dj]

    def forward(self, x):
        b, h, w, c = x.shape
        ok = (self.kernel_size == (4, 4) and self.stride == (2, 2) and self.padding == (1, 1) and h % 2 == 0
              and w % 2 == 0 and c % 2 == 0 and _conv_tiles(h // 2, w // 2))
        if not ok:
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=SIDE_DTYPE == torch.bfloat16):
                return _nhwc(super().forward(_side(_nchw(x))))
        xs = x.reshape(b, h // 2, 2, w // 2, 2, c).permute(0, 1, 3, 2, 4, 5).reshape(b, h // 2, w // 2, 4 * c)
        return AF.conv2d(xs, self._s2d_weight(), self.bias)


def _conv_tiles(h, w):
    """Image sizes the implicit-GEMM kernels tile (128-pixel output boxes, 64-pixel K boxes of the weight gradient)."""
    def box(pixels):
        if w >= pixels:
            return w % pixels == 0
        if pixels % w:
            return False
        rows = pixels // w
        return h % rows == 0 if h >= rows else rows % h == 0
    return box(128) and box(64)


def Downsample(dim, dim_out=None):
    return _DownConv(dim, default(dim_out, dim), 4, 2, 1)


class WeightStandardizedConv2d(nn.Conv2d):
    """cond_unet.py:345-358: K11 standardise+pack, then the implicit-GEMM conv."""

    def forward(self, x):
        assert self.stride == (1, 1), "adm_b200: stride-1 weight-standardised convs only (the configured path)"
        return AF.conv2d(x, self.weight, self.bias, ws=True, ws_eps=1e-5)


class LayerNorm(nn.Module):
    """cond_unet.py:360-369: per-pixel normalisation over channels with gain g (no bias), eps 1e-5."""

    def __init__(self, dim):
        super().__init__()
        self.g = nn.Parameter(torch.ones(1, dim, 1, 1))

    def forward(self, x):  # NHWC
        if x.is_cuda and ops.chan_layernorm_ok(x.shape[-1]):
            return AF.channel_layer_norm(x, self.g, 1e-5)
        return F.layer_norm(x.float(), (x.shape[-1],), self.g.reshape(-1), None, 1e-5).to(torch.bfloat16)


class PreNorm(nn.Module):
    def __init__(self, dim, fn):
        super().__init__()
        self.fn = fn
        self.norm = LayerNorm(dim)

    def forward(self, x):
        return self.fn(self.norm(x))


class GaussianFourierProjection(nn.Module):
    """cond_unet.py:396-405."""

    def __init__(self, embedding_size=256, scale=1.0):
        super().__init__()
        self.W = nn.Parameter(torch.randn(embedding_size) * scale, requires_grad=False)

    def forward(self, x):
        p = x[:, None] * self.W[None, :] * 2 * math.pi
        return torch.cat([torch.sin(p), torch.cos(p)], dim=-1)


class SinusoidalPosEmb(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.dim = dim

    def forward(self, x):
        half = self.dim // 2
        e = torch.exp(torch.arange(half, device=x.device) * -(math.log(10000) / (half - 1)))
        e = x[:, None] * e[None, :]
        return torch.cat((e.sin(), e.cos()), dim=-1)


class RandomOrLearnedSinusoidalPosEmb(nn.Module):
    """cond_unet.py:407-422."""

    def __init__(self, dim, is_random=False):
        super().__init__()
        assert dim % 2 == 0
        self.weights = nn.Parameter(torch.randn(dim // 2), requires_grad=not is_random)

    def forward(self, x):
        x = x[:, None]
        f = x * self.weights[None, :] * 2 * math.pi
        return torch.cat((x, f.sin(), f.cos()), dim=-1)


class Block(nn.Module):
    """cond_unet.py:427-443: WS-conv3x3 -> GroupNorm -> (1+scale), shift -> SiLU; the last three are ONE kernel."""

    def __init__(self, dim, dim_out, groups=8):
        super().__init__()
        self.proj = WeightStandardizedConv2d(dim, dim_out, 3, padding=1)
        self.norm = nn.GroupNorm(groups, dim_out)
        self.act = nn.SiLU()

    def forward(self, x, scale_shift=None):
        x = self.proj(x)
        return AF.group_norm_act(x, self.norm.weight, self.norm.bias, self.norm.num_groups, self.norm.eps,
                                 scale_shift=scale_shift, act=True)


class ResnetBlock(nn.Module):
    """cond_unet.py:445-469."""

    def __init__(self, dim, dim_out, *, time_emb_dim=None, groups=8):
        super().__init__()
        self.mlp = nn.Sequential(nn.SiLU(), nn.Linear(time_emb_dim, dim_out * 2)) if exists(time_emb_dim) else None
        self.block1 = Block(dim, dim_out, groups=groups)
        self.block2 = Block(dim_out, dim_out, groups=groups)
        self.res_conv = _Conv(dim, dim_out, 1) if dim != dim_out else nn.Identity()

    def forward(self, x, time_emb=None):
        ss = self.mlp(time_emb).float() if exists(self.mlp) and exists(time_emb) else None  # [B, 2C] = (scale | shift)
        h = self.block1(x, scale_shift=ss)
        h = self.block2(h)
        return h + self.res_conv(x)


class LinearAttention(nn.Module):
    """cond_unet.py:503-531: to_qkv (1x1, no bias) -> K12 fused linear attention -> to_out (1x1 + LayerNorm)."""

    def __init__(self, dim, heads=4, dim_head=32):
        super().__init__()
        self.scale = dim_head ** -0.5
        self.heads = heads
        hidden = dim_head * heads
        self.to_qkv = _Conv(dim, hidden * 3, 1, bias=False)
        self.to_out = nn.Sequential(_Conv(hidden, dim, 1), LayerNorm(dim))

    def forward(self, x):
        return self.to_out(AF.linear_attention(self.to_qkv(x), self.heads, self.scale))


class Attention(nn.Module):
    """cond_unet.py:533-555.  The head dim (32) is zero-padded to the 64-wide K slab of the tensor-core GEMMs inside the
    projection weights, so q.k and p.v are unchanged and no activation is re-laid-out."""

    def __init__(self, dim, heads=4, dim_head=32):
        super().__init__()
        self.scale = dim_head ** -0.5
        self.heads, self.dim_head = heads, dim_head
        hidden = dim_head * heads
        self.to_qkv = nn.Conv2d(dim, hidden * 3, 1, bias=False)
        self.to_out = nn.Conv2d(hidden, dim, 1)

    def forward(self, x):
        h, d = self.heads, self.dim_head
        pad = (-d) % 64
        cin = self.to_qkv.weight.shape[1]
        wq = F.pad(self.to_qkv.weight.reshape(3, h, d, cin), (0, 0, 0, pad)).reshape(3 * h * (d + pad), cin, 1, 1)
        qkv = AF.conv2d(x, wq)
        a = AF.attention(qkv, h, self.scale)
        dim = self.to_out.weight.shape[0]
        wo = F.pad(self.to_out.weight.reshape(dim, h, d), (0, pad)).reshape(dim, h * (d + pad), 1, 1)
        return AF.conv2d(a, wo, self.to_out.bias)


class _GroupNorm(nn.GroupNorm):
    def forward(self, x):  # NHWC bf16, no activation
        return AF.group_norm_act(x, self.weight, self.bias, self.num_groups, self.eps, act=False)


class _Decouple(nn.Sequential):
    """GroupNorm -> conv3x3 -> SpatialAtt, plus the residual of `x + decouple(x)` fused into the last kernel."""

    def forward(self, x):
        return self[2](self[1](self[0](x)), x)


# ------------------------------------------------------------------------------------------------ the network
class Unet(nn.Module):
    """cond_unet.py:592-917 (the reference derives from pl.LightningModule only for its base class)."""

    def __init__(self, dim, init_dim=None, out_dim=None, dim_mults=(1, 2, 4, 8), cond_in_dim=1, cond_dim=64,
                 cond_dim_mults=(2, 4, 8), channels=1, out_mul=1, self_condition=False, resnet_block_groups=8,
                 learned_variance=False, learned_sinusoidal_cond=False, random_fourier_features=False,
                 learned_sinusoidal_dim=16, window_sizes1=[[16, 16], [8, 8], [4, 4], [2, 2]],
                 window_sizes2=[[16, 16], [8, 8], [4, 4], [2, 2]], fourier_scale=16, precondition=True, ckpt_path=None,
                 ignore_keys=[], **kwargs):
        super().__init__()
        kwargs.pop("class_name", None)
        cfg = kwargs.pop("cfg", None)
        if cfg is not None:  # train_cond_ldm.py:47-49 passes the unet cfg node as well
            kwargs = {**dict(cfg), **kwargs}
        self.cond_pe = kwargs.get("cond_pe", False)
        num_pos_feats = kwargs.get("num_pos_feats") if self.cond_pe else 0
        self.channels, self.self_condition = channels, self_condition
        input_channels = channels * (2 if self_condition else 1)
        init_dim = default(init_dim, dim)
        cond_net = kwargs.get("cond_net", None)
        if cond_net == "swin":
            f_condnet = 128
            self.init_conv_mask = swin_b(in_channels=1 if kwargs.get("single_channel_cond", False) else 3)
        elif cond_net in ("effnet", "resnet"):
            raise NotImplementedError(f"adm_b200 implements cond_net='swin' (the configured path), not {cond_net!r}")
        else:
            raise NotImplementedError
        self.init_conv = nn.Sequential(nn.Conv2d(input_channels + f_condnet, init_dim, 7, padding=3),
                                       _GroupNorm(num_groups=min(init_dim // 4, 8), num_channels=init_dim))
        if self.cond_pe:
            self.cond_pos_embedding = nn.Sequential(
                PositionEmbeddingLearned(feature_size=kwargs.get("cond_feature_size"),
                                         num_pos_feats=kwargs.get("num_pos_feats") // 2),
                nn.Conv2d(num_pos_feats + init_dim, init_dim, 1))
        dims = [init_dim, *map(lambda m: dim * m, dim_mults)]
        dims_rev = dims[::-1]
        in_out = list(zip(dims[:-1], dims[1:]))
        self.projects = nn.ModuleList(nn.Conv2d(f_condnet * 2 ** i, dims[i], 1) for i in range(4))
        block_klass = partial(ResnetBlock, groups=resnet_block_groups)
        time_dim = dim * 4
        self.random_or_learned_sinusoidal_cond = learned_sinusoidal_cond or random_fourier_features
        if self.random_or_learned_sinusoidal_cond:
            sinu = RandomOrLearnedSinusoidalPosEmb(learned_sinusoidal_dim, random_fourier_features)
            fourier_dim = learned_sinusoidal_dim + 1
        else:
            sinu = GaussianFourierProjection(dim // 2, scale=fourier_scale)
            fourier_dim = dim
        self.time_mlp = nn.Sequential(sinu, nn.Linear(fourier_dim, time_dim), nn.GELU(), nn.Linear(time_dim, time_dim))

        self.downs = nn.ModuleList([])
        self.downs_mask = nn.ModuleList([])
        self.ups = nn.ModuleList([])
        self.relation_layers_down = nn.ModuleList([])
        self.relation_layers_up = nn.ModuleList([])
        self.ups2 = nn.ModuleList([])
        self.relation_layers_up2 = nn.ModuleList([])
        nres = len(in_out)
        for ind, (dim_in, dim_out) in enumerate(in_out):
            is_last = ind >= nres - 1
            self.downs.append(nn.ModuleList([
                block_klass(dim_in, dim_in, time_emb_dim=time_dim),
                block_klass(dim_in, dim_in, time_emb_dim=time_dim),
                Residual(PreNorm(dim_in, LinearAttention(dim_in))),
                Downsample(dim_in, dim_out) if not is_last else _Conv(dim_in, dim_out, 3, padding=1)]))
            self.relation_layers_down.append(RelationNet(in_channel1=dims[ind], in_channel2=dims[ind], nhead=8, layers=1,
                                                         embed_dim=dims[ind], ffn_dim=dims[ind] * 2,
                                                         window_size1=window_sizes1[ind], window_size2=window_sizes2[ind]))
        mid_dim = dims[-1]
        self.mid_block1 = block_klass(mid_dim, mid_dim, time_emb_dim=time_dim)
        self.mid_attn = Residual(PreNorm(mid_dim, Attention(mid_dim)))
        self.mid_block2 = block_klass(mid_dim, mid_dim, time_emb_dim=time_dim)
        self.decouple1 = _Decouple(_GroupNorm(num_groups=min(mid_dim // 4, 8), num_channels=mid_dim),
                                   _Conv(mid_dim, mid_dim, 3, padding=1), SpatialAtt(mid_dim))
        self.decouple2 = _Decouple(_GroupNorm(num_groups=min(mid_dim // 4, 8), num_channels=mid_dim),
                                   _Conv(mid_dim, mid_dim, 3, padding=1), SpatialAtt(mid_dim))
        for ind, (dim_in, dim_out) in enumerate(reversed(in_out)):
            is_last = ind == len(in_out) - 1
            for ups, rel in ((self.ups, self.relation_layers_up), (self.ups2, self.relation_layers_up2)):
                ups.append(nn.ModuleList([
                    block_klass(dim_out + dim_in, dim_out, time_emb_dim=time_dim),
                    block_klass(dim_out + dim_in, dim_out, time_emb_dim=time_dim),
                    Residual(PreNorm(dim_out, LinearAttention(dim_out))),
                    Upsample(dim_out, dim_in) if not is_last else _Conv(dim_out, dim_in, 3, padding=1)]))
                rel.append(RelationNet(in_channel1=dims_rev[ind + 1], in_channel2=dims_rev[ind], nhead=8, layers=1,
                                       embed_dim=dims_rev[ind], ffn_dim=dims_rev[ind] * 2,
                                       window_size1=window_sizes1[::-1][ind], window_size2=window_sizes2[::-1][ind]))
        default_out_dim = channels * (1 if not learned_variance else 2)
        self.out_dim = default(out_dim, default_out_dim)
        self.final_res_block = block_klass(dim * 2, dim, time_emb_dim=time_dim)
        self.final_conv = _Conv(dim, self.out_dim * out_mul, 1)
        self.final_res_block2 = block_klass(dim * 2, dim, time_emb_dim=time_dim)
        self.final_conv2 = _Conv(dim, self.out_dim, 1)
        self.precondition = precondition
        if ckpt_path is not None:
            self.init_from_ckpt(ckpt_path, ignore_keys=ignore_keys)
        if kwargs.get("fix_bb", False):
            for p in self.init_conv_mask.parameters():
                p.requires_grad = False

    def init_from_ckpt(self, path, ignore_keys=list()):
        sd = torch.load(path, map_location="cpu")["model"]
        for k in list(sd.keys()):
            if any(k.startswith(ik) for ik in ignore_keys):
                print("Deleting key {} from state_dict.".format(k))
                del sd[k]
        msg = self.load_state_dict(sd, strict=False)
        print(f"Restored from {path}")
        print("==>Load Unet Info: ", msg)

    @staticmethod
    def _relate(layer, cond, x):
        """RelationNet on NHWC bf16 tensors (cond: the projected Swin feature map of this level, converted once)."""
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=SIDE_DTYPE == torch.bfloat16):
            return layer(cond, x).to(torch.bfloat16)

    def _decoder(self, x, ups, relations, skips, hms, r, final_block, final_conv, t):
        skips, hms = list(skips), list(hms)
        for (block1, block2, attn, upsample), rel in zip(ups, relations):
            x = block1(torch.cat((x, skips.pop()), dim=-1), t)
            x = self._relate(rel, hms.pop(), x)
            x = block2(torch.cat((x, skips.pop()), dim=-1), t)
            x = attn(x)
            x = upsample(x)
        x = final_block(torch.cat((x, r), dim=-1), t)
        return final_conv(x)

    def encode_condition(self, mask, size):
        """The part of ``forward`` that depends on the condition only (cond_unet.py:724-733): Swin-B features of the
        condition image, their 1x1 projections (NHWC bf16, shared by the encoder and both decoders) and the bilinear
        resize of the first feature map that is concatenated to the input of the stem.  A sampler whose condition is
        fixed over its N steps computes it once and passes it back as ``forward(..., cond_feats=...)``."""
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=SIDE_DTYPE == torch.bfloat16):
            hm = self.init_conv_mask(mask.to(torch.float32))
            up0 = F.interpolate(hm[0].float().contiguous(memory_format=torch.channels_last), size=tuple(size),
                                mode="bilinear")
            hm = [_nhwc(proj(f)) for proj, f in zip(self.projects, hm)]
        return up0, hm

    def forward(self, x, time, mask, x_self_cond=None, sigma_max=1, *args, cond_feats=None, **kwargs):
        if not x.is_cuda:
            raise RuntimeError("adm_b200: the conditional UNet runs on CUDA (sm_100a) only; there is no CPU fallback")
        x = x.to(torch.float32)
        time = time.to(torch.float32).reshape(-1)
        if time.numel() == 1 and x.shape[0] != 1:
            time = time.expand(x.shape[0])
        if self.self_condition:
            x_self_cond = default(x_self_cond, lambda: torch.zeros_like(x))
            x = torch.cat((x_self_cond, x), dim=1)
        t4 = time.reshape(-1, 1, 1, 1)
        c_skip1, c_skip2 = -1 + t4, t4.sqrt()
        c_out1, c_out2 = t4 / (t4 + 1).sqrt(), (1 - t4).sqrt() / (1 + t4).sqrt()
        c_noise = time.log()
        x_in = x
        up0, hm = cond_feats if cond_feats is not None else self.encode_condition(mask, x.shape[-2:])
        stem_in = torch.cat([x, up0], dim=1)
        # 7x7 stem (cond_unet.py:656, 7 % of the FLOPs): the implicit-GEMM conv with 49 taps; the 131 input channels are
        # zero-padded to a multiple of 8 on the activation and on the weight
        stem, sx = self.init_conv[0], _nhwc(stem_in)
        if _conv_tiles(sx.shape[1], sx.shape[2]) and stem.kernel_size == (7, 7) and stem.padding == (3, 3):
            pad = (-sx.shape[-1]) % 8
            h0 = AF.conv2d(F.pad(sx, (0, pad)), F.pad(stem.weight, (0, 0, 0, 0, 0, pad)), stem.bias)
        else:
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=SIDE_DTYPE == torch.bfloat16):
                h0 = _nhwc(stem(stem_in.contiguous(memory_format=torch.channels_last)))
        xh = self.init_conv[1](h0)
        r = xh
        t = self.time_mlp(c_noise)
        skips = []
        for i, ((block1, block2, attn, downsample), rel) in enumerate(zip(self.downs, self.relation_layers_down)):
            xh = block1(xh, t)
            skips.append(xh)
            xh = self._relate(rel, hm[i], xh)
            xh = block2(xh, t)
            xh = attn(xh)
            skips.append(xh)
            xh = downsample(xh)
        xh = self.mid_block1(xh, t)
        xh = self.mid_attn(xh)
        xh = self.mid_block2(xh, t)
        b1, b2 = self.decouple1(xh), self.decouple2(xh)
        f1 = self._decoder(b1, self.ups, self.relation_layers_up, skips, hm, r, self.final_res_block, self.final_conv, t)
        f2 = self._decoder(b2, self.ups2, self.relation_layers_up2, skips, hm, r, self.final_res_block2,
                           self.final_conv2, t)
        x1 = _nchw(f1).float()
        x2 = _nchw(f2).float()
        if self.precondition:
            x1 = c_skip1 * x_in + c_out1 * x1
            x2 = c_skip2 * x_in + c_out2 * x2
        return x1, x2
