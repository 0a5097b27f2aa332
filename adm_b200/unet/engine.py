"""Fused sm_100a execution engine for the two-decoder DhariwalUNet (forward + hand-written backward).

Follows /root/reference/unet/uncond_unet.py: EDMPrecond.forward :614-635, DhariwalUNet.forward :544-581,
UNetBlock.forward :189-211, SpatialAtt.forward :27-37, with this data layout:

* activations NHWC bf16 (channels innermost, so one 64-channel slab of a pixel row is one 128 B TMA/UMMA swizzle row);
* weights: fp32 masters stay in the reference layout inside the nn.Modules; bf16 packed copies [Cout][tap][Cin] are derived
  caches, rebuilt when a parameter's version changes;
* channel concats (torch.cat([x, skip]), :570-571) are never materialised: GroupNorm kernels and the GEMM engine take two
  sources;
* per-(sample, channel) sum / sum-of-squares tables carry the GroupNorm statistics.

Gradients are accumulated straight into ``param.grad`` (fp32, reference layout) by ``backward`` — the engine plays the
role of autograd's AccumulateGrad for its own parameters.
"""
from __future__ import annotations

import contextlib
from types import SimpleNamespace as NS

import torch

from .. import ops
from ..ops import BF16, F32, pad64


def _groups(c):
    return min(32, c // 4)


class UNetEngine:
    def __init__(self, net):
        self.net = net
        self._cache = {}
        self._epoch = 0
        self._seed_next = 1  # index of the next training forward (mixed into the dropout seeds)
        self.base_seed = 0x1234
        # ordered block table + offsets into the batched affine GEMM
        self.block_list = []
        off = 0
        for sec in ("enc", "dec", "dec2"):
            for name, m in getattr(net, sec).items():
                if hasattr(m, "affine"):
                    self.block_list.append((f"{sec}.{name}", m, off))
                    off += m.affine.out_features
        self.affine_total = off
        self._perm = {}
        self.grad_hook = None  # callable(list_of_params) invoked as soon as those gradients are final (DP overlap)
        # set by the training arena (adm_b200.train.TrainStep): (wall bf16 [T, emb], ball fp32 [T], dwall fp32, dball fp32,
        # fp32 master slice of wall, parameter versions)
        # when every block's affine weight / bias are laid out back to back in the parameter arena
        self.affine_pack = None
        self.affine_grad_overwrite = False  # set by TrainStep when grad_accum == 1 (gradients are zero before backward)
        # Weight / bias gradients of the convs run on a side stream, concurrently with the data-gradient chain: a wgrad
        # only feeds the optimizer, and every GEMM is a persistent kernel whose last partial wave leaves SMs idle (and
        # the 4x4 / 8x8 levels never fill 148 SMs) — the other stream's CTAs take those SMs.  Joined at every _notify.
        self._side = None
        self._side_pending = []
        # device-resident step counter mixed into every dropout seed (fresh masks per CUDA-graph replay); owned by the
        # training step (adm_b200.train.TrainStep) and passed to the GroupNorm kernels per call
        self.seed_counter = None

    def seed_position(self, value=None):
        """Get (or restore, from a checkpoint) the position in the dropout-mask stream."""
        if value is not None:
            self._seed_next = int(value) + 1
        return self._seed_next - 1

    # ------------------------------------------------------------------------------------------ arena fast paths
    def packable_params(self):
        """Conv weights this engine consumes in the plain packed order [Cout][tap][Cin] with no row permutation and
        no channel padding: an arena may store exactly that order (channels-last) and attach a bf16 shadow
        (``weight._adm_pack = (bf16 [Cout, taps, Cin], fp32 grad [Cout, taps, Cin])``) so that neither a re-pack of the
        weights nor an un-pack of their gradients is needed."""
        net = self.net
        convs = []
        for _, m, _ in self.block_list:
            convs += [m.conv0, m.conv1]
            if m.skip is not None and m.skip.weight is not None:
                convs.append(m.skip)
            if m.num_heads:
                convs.append(m.proj)
        convs += [net.out_conv, net.out_conv2, net.decouple1[0], net.decouple2[0]]
        chans = {m.in_channels for _, m, _ in self.block_list} | {m.out_channels for _, m, _ in self.block_list}
        if any(c % 64 for c in chans):
            return []
        return [c.weight for c in convs if c.weight.shape[1] % 64 == 0]

    @staticmethod
    def _pack_of(w):
        """(bf16 packed weights, fp32 packed gradient) of an arena-resident channels-last parameter, or None."""
        pk = getattr(w, "_adm_pack", None)
        if pk is None:
            return None
        if w._version != pk[2]:  # modified through torch (load_state_dict, ...) since the shadow was written
            ops.cast_bf16_into(pk[3], pk[0])
            if pk[4] is not None:  # and its transposed twin for the data gradient
                co, kk, ci = pk[0].shape
                tiles = ops.weight_transpose_tiles(0, co, kk, ci).to(pk[0].device)
                ops.transpose_weight_tiles(pk[0], pk[4], tiles)
            w._adm_pack = pk = (pk[0], pk[1], w._version, pk[3], pk[4])
        return pk

    @staticmethod
    def _qkv_pack_of(blk, perm):
        """(bf16 [3C, 1, C] weights, fp32 [3C] bias) of an attention block in the executed (q | k | v) x head x d row order
        when a parameter arena keeps them (``qkv.weight._adm_qkv``, re-derived by ONE batched row gather per optimizer step,
        adm_b200.train.ParamArena), else None."""
        qp = getattr(blk.qkv.weight, "_adm_qkv", None)
        if qp is None:
            return None
        w, b = blk.qkv.weight, blk.qkv.bias
        if (w._version, b._version) != qp[2]:  # written through torch since the last gather (load_state_dict, ...)
            ops.pack_conv_weight(w.detach().contiguous(), row_perm=perm[0], out=qp[0])
            torch.index_select(b.detach(), 0, perm[1], out=qp[1])
            w._adm_qkv = qp = (qp[0], qp[1], (w._version, b._version))
        return qp[0], qp[1]

    # ------------------------------------------------------------------------------------------ weight caches
    def invalidate(self):
        """Call after parameters were updated through raw pointers (the fused optimizer)."""
        self._epoch += 1

    def _cached(self, key, params, build):
        ver = tuple((p.data_ptr(), p._version) for p in params) + (self._epoch,)
        hit = self._cache.get(key)
        if hit is not None and hit[0] == ver:
            return hit[1]
        val = build(hit[1] if hit is not None else None)
        self._cache[key] = (ver, val)
        return val

    def signature(self):
        """Changes whenever any parameter may have changed (optimizer epoch or a torch-side in-place write)."""
        return self._epoch, sum(p._version for p in self.net.parameters())

    def pointer_signature(self):
        """Changes when parameters are re-homed (a training or EMA arena took them over): anything that baked device
        pointers of derived operands (a captured CUDA graph) must be rebuilt, not just refreshed."""
        return hash(tuple(p.data_ptr() for p in self.net.parameters()))

    def _dev(self):
        return self.net.map_layer0.weight.device

    def conv_w(self, conv, c1=None, c2=0, perm=None):
        w = conv.weight
        pk = self._pack_of(w) if perm is None else None
        if pk is not None:
            return pk[0]
        return self._cached(("cw", id(conv)), [w],
                            lambda old: ops.pack_conv_weight(w.detach(), c1, c2, row_perm=perm, out=old))

    # Every builder below re-derives INTO the buffer of the previous value when there is one, so that device pointers
    # stay stable: a CUDA graph captured over a forward pass (sampler) stays valid across weight updates.
    def lin_w(self, lin):
        w = lin.weight

        def build(old):
            if old is None:
                return ops.cast_bf16(w.detach())
            return ops.cast_bf16_into(w.detach().contiguous(), old)
        return self._cached(("lw", id(lin)), [w], build)

    def aug_w(self):
        w = self.net.map_augment.weight  # [mc, augment_dim] -> zero padded to 16 columns

        def build(old):
            wp = torch.zeros(w.shape[0], 16, device=w.device, dtype=F32)
            wp[:, :w.shape[1]] = w.detach()
            return ops.cast_bf16(wp) if old is None else ops.cast_bf16_into(wp, old)
        return self._cached(("aug",), [w], build)

    def affine_all(self):
        if self.affine_pack is not None:
            ap = self.affine_pack
            ver = tuple(m.affine.weight._version for _, m, _ in self.block_list)
            if ver != ap[5]:  # written through torch since the shadow was derived (load_state_dict, ...)
                ops.cast_bf16_into(ap[4], ap[0])
                self.affine_pack = ap = ap[:5] + (ver,)
            return ap[0], ap[1]
        ps = [m.affine.weight for _, m, _ in self.block_list] + [m.affine.bias for _, m, _ in self.block_list]

        def build(old):
            wall = old[0] if old is not None else torch.empty(self.affine_total, self.net.emb_channels,
                                                                device=self._dev(), dtype=BF16)
            for _, m, off in self.block_list:
                o = m.affine.out_features
                ops._lib.check(ops._lib.load().adm_cast_f32_bf16(m.affine.weight.data_ptr(), wall[off:off + o].data_ptr(),
                                                                 m.affine.weight.numel(), ops._stream()), "cast")
            biases = [m.affine.bias.detach() for _, m, _ in self.block_list]
            ball = torch.cat(biases) if old is None else torch.cat(biases, out=old[1])
            return wall, ball
        return self._cached(("affine_all",), ps, build)

    def qkv_perm(self, c, heads):
        """packed row (which, head, d) <- reference row head*3d + d*3 + which (uncond_unet.py:205)."""
        key = (c, heads)
        if key not in self._perm:
            d = c // heads
            which, hh, dd = torch.meshgrid(torch.arange(3), torch.arange(heads), torch.arange(d), indexing="ij")
            perm = (hh * 3 * d + dd * 3 + which).reshape(-1)
            self._perm[key] = (perm.to(self._dev(), torch.int32), perm.to(self._dev(), torch.int64))
        return self._perm[key]

    # ------------------------------------------------------------------------------------------ gradient helpers
    def _fork_side(self, *keep):
        """Side stream ordered after everything issued so far on the current stream; `keep` (tensors the side work
        reads) stay referenced until the join, so the allocator cannot hand their memory to a later main-stream op."""
        if self._side is None:
            self._side = torch.cuda.Stream()
        self._side.wait_stream(torch.cuda.current_stream())
        self._side_pending.append(keep)
        return self._side

    def _join_side(self):
        if self._side_pending:
            torch.cuda.current_stream().wait_stream(self._side)
            self._side_pending.clear()

    def _notify(self, *modules, skip_affine=True):
        self._join_side()
        if self.grad_hook is None:
            return
        ps = []
        for m in modules:
            for name, p in m.named_parameters():
                if skip_affine and name.startswith("affine."):
                    continue
                ps.append(p)
        self.grad_hook(ps)

    @staticmethod
    def _grad(p):
        if p.grad is None:
            p.grad = torch.zeros_like(p, memory_format=torch.contiguous_format)
        return p.grad

    def _conv_param_grads(self, conv, dy, x1, x2=None, perm=None, dy_cols=None, bias_done=False):
        """dW (tcgen05 wgrad, packed) -> reference layout; db via column sums (unless the producer of dy already
        accumulated them: bias_done)."""
        if bias_done:
            bias = None
        else:
            bias = conv.bias
        if dy.is_cuda:
            with torch.cuda.stream(self._fork_side(dy, x1, x2, dy_cols)):
                self._conv_weight_grad(conv, dy, x1, x2, perm)
                if bias is not None:
                    self._bias_grad(bias, dy if dy_cols is None else dy_cols, perm)
            return
        self._conv_weight_grad(conv, dy, x1, x2, perm)
        if bias is not None:
            self._bias_grad(bias, dy if dy_cols is None else dy_cols, perm)

    def _conv_weight_grad(self, conv, dy, x1, x2=None, perm=None):
        k = conv.weight.shape[-1]
        c1 = x1.shape[-1]
        c2 = x2.shape[-1] if x2 is not None else 0
        cin_ref = conv.weight.shape[1]
        pk = self._pack_of(conv.weight) if perm is None else None
        if pk is not None and conv.weight.grad is not None and conv.weight.grad.data_ptr() == pk[1].data_ptr():
            ops.conv_wgrad(dy, x1, x2=x2, ntaps=k * k, out=pk[1])  # straight into the (channels-last) gradient arena
            return
        g = self._grad(conv.weight)
        if perm is not None and k == 1 and x2 is None and c1 == cin_ref and c1 % 64 == 0 and g.is_contiguous():
            # row-permuted 1x1 conv (qkv): the wgrad epilogue scatters its rows into the reference-ordered gradient
            ops.conv_wgrad(dy, x1, ntaps=1, out=g.view(g.shape[0], 1, c1), row_map=perm[0])
            return
        dwp = ops.conv_wgrad(dy, x1, x2=x2, ntaps=k * k)
        if x2 is None and c1 != cin_ref:  # zero-padded network input (3 -> 8 channels)
            c1 = cin_ref
        ops.unpack_conv_wgrad(dwp, c1, c2, k, out=self._grad(conv.weight), accumulate=True,
                              row_perm=perm[0] if perm is not None else None)

    def _bias_grad(self, bias, dy, perm=None):
        g = self._grad(bias)
        c = dy.shape[-1]
        if perm is None and c == g.numel():
            ops.col_sums(dy, g)
        elif perm is not None and c == g.numel() and g.is_contiguous():
            ops.col_sums(dy, g, out_map=perm[0])
        else:
            tmp = torch.zeros(c, device=dy.device, dtype=F32)
            ops.col_sums(dy, tmp)
            if perm is not None:
                g.index_add_(0, perm[1], tmp)
            else:
                g.add_(tmp[:g.numel()])

    def _dgrad(self, dy, conv, wpk, c1=None, c2=0, residual=None):
        """Data gradient of `conv` in its INPUT channel count (the packed weights pad every source to 64 channels:
        channel counts like 96 / 288 of the CelebAHQ-latent config come back padded and are cut here; a concat input
        whose first part is not a multiple of 64 is re-joined)."""
        cin = conv.weight.shape[1]
        c1 = cin if c1 is None else c1
        pk = self._pack_of(conv.weight)
        if pk is not None and pk[4] is not None and pk[0].data_ptr() == wpk.data_ptr():
            # arena-resident conv: dX = fprop(dY, W^T with mirrored taps) on the K-major dgrad shadow
            return ops.conv_fprop(dy, pk[4], residual=residual)
        if c2 and c1 % 64:
            full = ops.conv_dgrad(dy, wpk, residual=residual)
            p1 = pad64(c1)
            return torch.cat([full[..., :c1], full[..., p1:p1 + c2]], dim=-1)
        return ops.conv_dgrad(dy, wpk, n_valid=c1 + c2, residual=residual)

    # Attention heads whose width is not a multiple of 64 (d = 72 when C = 288 in the CelebAHQ-latent config; the head
    # width is out_channels // 64 heads, uncond_unet.py:173): every head is zero-padded to dpad = pad64(d) INSIDE the
    # projection weights — q.k and p.v are unchanged, the activations need no re-layout, and the tensor-core GEMMs keep
    # their 64-wide K slabs.  Padded fp32 weights are derived with torch index ops (cached per parameter version).
    def _head_rows(self, c, heads):
        key = ("rows", c, heads)  # cached: built once per shape (a host -> device copy, not capturable into a CUDA graph)
        if key not in self._perm:
            d = c // heads
            which, hh, dd = torch.meshgrid(torch.arange(3), torch.arange(heads), torch.arange(d), indexing="ij")
            self._perm[key] = (hh * 3 * d + dd * 3 + which).to(self._dev())  # [3, heads, d] -> reference qkv row
        return self._perm[key]

    def qkv_padded(self, blk):
        c, heads = blk.out_channels, blk.num_heads
        d, dpad = c // heads, pad64(c // heads)

        def build(old):
            rows = self._head_rows(c, heads)
            w = torch.zeros(3, heads, dpad, c, device=self._dev(), dtype=F32)
            w[:, :, :d] = blk.qkv.weight.detach().reshape(3 * c, c)[rows]
            b = torch.zeros(3, heads, dpad, device=self._dev(), dtype=F32)
            b[:, :, :d] = blk.qkv.bias.detach()[rows]
            wpk = ops.pack_conv_weight(w.reshape(3 * heads * dpad, c, 1, 1), out=old[0] if old is not None else None)
            bq = b.reshape(-1).contiguous()
            if old is not None:  # keep the device pointer stable: captured sampler graphs read this buffer
                bq = old[1].copy_(bq)
            return wpk, bq, rows
        return self._cached(("qkvpad", id(blk)), [blk.qkv.weight, blk.qkv.bias], build)

    def proj_padded(self, blk):
        c, heads = blk.out_channels, blk.num_heads
        d, dpad = c // heads, pad64(c // heads)

        def build(old):
            w = torch.zeros(c, heads, dpad, device=self._dev(), dtype=F32)
            w[:, :, :d] = blk.proj.weight.detach().reshape(c, heads, d)
            return ops.pack_conv_weight(w.reshape(c, heads * dpad, 1, 1), out=old)
        return self._cached(("projpad", id(blk)), [blk.proj.weight], build)

    # ------------------------------------------------------------------------------------------ UNetBlock
    def block_fwd(self, blk, x1, x2, params, training, seed, save):
        c = NS(blk=blk, x1=x1, x2=x2, params=params, seed=seed)
        cin1 = x1.shape[-1]
        cin2 = x2.shape[-1] if x2 is not None else 0
        cin, cout = cin1 + cin2, blk.out_channels
        mode = 1 if blk.down else (2 if blk.up else 0)
        c.mode = mode
        c.drop_p = float(blk.dropout) if training else 0.0
        c.sums0, c.a0 = ops.gn_forward(x1, x2, blk.norm0.weight, blk.norm0.bias, _groups(cin), blk.norm0.eps, act=True,
                                       resample=mode)
        # after the fused concat-GroupNorm the conv sees ONE tensor a0 with cin channels
        c.h0 = ops.conv_fprop(c.a0, self.conv_w(blk.conv0), bias=blk.conv0.bias)
        c.sums1, c.a1 = ops.gn_forward(c.h0, None, blk.norm1.weight, blk.norm1.bias, _groups(cout), blk.norm1.eps,
                                       params=params, act=True, drop_p=c.drop_p, seed=seed, seed_counter=self.seed_counter)
        if blk.skip is not None and blk.skip.weight is not None:
            res = ops.conv_fprop(x1, self.conv_w(blk.skip, cin1, cin2), x2=x2, bias=blk.skip.bias)
        elif mode:
            res = ops.resample(x1, mode)
        else:
            res = x1
        c.h1 = ops.conv_fprop(c.a1, self.conv_w(blk.conv1), bias=blk.conv1.bias, residual=res)
        out = c.h1
        if blk.num_heads:
            c.sums2, c.a2 = ops.gn_forward(c.h1, None, blk.norm2.weight, blk.norm2.bias, _groups(cout), blk.norm2.eps,
                                           act=False)
            if (cout // blk.num_heads) % 64:  # head width 72 / 96: zero-padded heads
                wq, bq, _ = self.qkv_padded(blk)
                c.qkv = ops.conv_fprop(c.a2, wq, bias=bq)
                c.att, c.p = ops.attention_fwd(c.qkv, blk.num_heads, scale=(cout // blk.num_heads) ** -0.5,
                                               need_p=save is not None)
                out = ops.conv_fprop(c.att, self.proj_padded(blk), bias=blk.proj.bias, residual=c.h1)
            else:
                perm = self.qkv_perm(cout, blk.num_heads)
                qp = self._qkv_pack_of(blk, perm)
                if qp is not None:  # arena: (q | k | v)-ordered weights / bias re-derived by one batched gather per step
                    wq, bq = qp
                else:
                    bq = self._cached(("qkvb", id(blk)), [blk.qkv.bias],
                                      lambda old: blk.qkv.bias.detach()[perm[1]].contiguous() if old is None
                                      else torch.index_select(blk.qkv.bias.detach(), 0, perm[1], out=old))
                    wq = self.conv_w(blk.qkv, perm=perm[0])
                c.qkv = ops.conv_fprop(c.a2, wq, bias=bq)
                c.att, c.p = ops.attention_fwd(c.qkv, blk.num_heads, need_p=save is not None)
                out = ops.conv_fprop(c.att, self.conv_w(blk.proj), bias=blk.proj.bias, residual=c.h1)
        if save is not None:
            save.append(c)
        return out

    def export_dropout_masks(self, tape):
        """The dropout keep-masks (already scaled by 1/(1-p)) a training forward drew, one NCHW fp32 tensor per UNetBlock,
        keyed by the block's state_dict prefix.  The masks are a stateless hash of (seed, element index), so they are
        regenerated here by running the GroupNorm-apply kernel over a tensor of ones with the block's own seed.
        Used by the parity tests to feed the reference's dropout (uncond_unet.py:200) the same masks."""
        names = {id(m): name for name, m, _ in self.block_list}
        out = {}
        for c in tape.items:
            if not hasattr(c, "blk") or not c.drop_p:
                continue
            n, h, w, ch = c.h0.shape
            coef = torch.zeros(n, ch, 4, device=c.h0.device, dtype=F32)
            coef[..., 0] = 1.0
            ones = torch.ones(n, h, w, ch, device=c.h0.device, dtype=BF16)
            m = ops.gn_apply(ones, None, coef, act=False, drop_p=c.drop_p, seed=c.seed, seed_counter=self.seed_counter)
            out["model." + names[id(c.blk)]] = m.float().permute(0, 3, 1, 2).contiguous()
        return out

    def bias_sinks(self, blk):
        """Bias gradients that equal the column sums of the gradient at a block's OUTPUT (they can be accumulated by
        whichever kernel produces that gradient): proj.bias with attention, else conv1.bias (+ the 1x1 skip's bias)."""
        if blk.num_heads:
            return [self._grad(blk.proj.bias)]
        sinks = [self._grad(blk.conv1.bias)]
        if blk.skip is not None and blk.skip.weight is not None and blk.skip.bias is not None:
            sinks.append(self._grad(blk.skip.bias))
        return sinks

    def block_bwd(self, c, dout, dparams, dout_bias_done=False, input_sinks=None):
        """dout: gradient at the block output.  Returns (dx1, dx2).
        dout_bias_done: the producer of `dout` already added its column sums to bias_sinks(blk).
        input_sinks: bias_sinks of the block that produced x1 — this block's last kernel accumulates colsum(dx1) there."""
        blk = c.blk
        cin1 = c.x1.shape[-1]
        cin2 = c.x2.shape[-1] if c.x2 is not None else 0
        cin, cout = cin1 + cin2, blk.out_channels
        has_skip_conv = blk.skip is not None and blk.skip.weight is not None
        h1_sinks = [self._grad(blk.conv1.bias)] + ([self._grad(blk.skip.bias)] if has_skip_conv else [])
        if blk.num_heads and (cout // blk.num_heads) % 64:
            heads, d = blk.num_heads, cout // blk.num_heads
            dpad = pad64(d)
            wq, _, rows = self.qkv_padded(blk)
            wp = self.proj_padded(blk)
            # proj: weight gradient comes back in the padded column layout (head, dpad)
            dwp = ops.conv_wgrad(dout, c.att, ntaps=1)  # [cout, 1, heads*dpad]
            self._grad(blk.proj.weight).add_(
                dwp[:, 0, :heads * dpad].reshape(cout, heads, dpad)[:, :, :d].reshape(blk.proj.weight.shape))
            if not dout_bias_done:
                self._bias_grad(blk.proj.bias, dout)
            datt = ops.conv_dgrad(dout, wp)
            dqkv = ops.attention_bwd(datt, c.qkv, c.p, heads, scale=d ** -0.5, a=c.att)
            dwq = ops.conv_wgrad(dqkv, c.a2, ntaps=1)  # [3*heads*dpad, 1, pad64(cout)]
            gq = dwq[:, 0, :cout].reshape(3, heads, dpad, cout)[:, :, :d]
            self._grad(blk.qkv.weight).view(3 * cout, cout).index_add_(0, rows.reshape(-1), gq.reshape(-1, cout))
            bsum = torch.zeros(3 * heads * dpad, device=dqkv.device, dtype=F32)
            ops.col_sums(dqkv, bsum)
            self._grad(blk.qkv.bias).index_add_(0, rows.reshape(-1), bsum.reshape(3, heads, dpad)[:, :, :d].reshape(-1))
            da2 = ops.conv_dgrad(dqkv, wq, n_valid=cout)
        elif blk.num_heads:
            perm = self.qkv_perm(cout, blk.num_heads)
            self._conv_param_grads(blk.proj, dout, c.att, bias_done=dout_bias_done)
            datt = self._dgrad(dout, blk.proj, self.conv_w(blk.proj))
            dqkv = ops.attention_bwd(datt, c.qkv, c.p, blk.num_heads, a=c.att)
            self._conv_param_grads(blk.qkv, dqkv, c.a2, perm=perm)
            qp = self._qkv_pack_of(blk, perm)
            da2 = self._dgrad(dqkv, blk.qkv, qp[0] if qp is not None else self.conv_w(blk.qkv, perm=perm[0]))
        if blk.num_heads:
            dh1, _ = ops.gn_bwd(da2, c.h1, None, c.sums2, blk.norm2.weight, blk.norm2.bias, _groups(cout),
                                act=False, dgamma=self._grad(blk.norm2.weight),
                                dbeta=self._grad(blk.norm2.bias), add=dout, add_mode=0,
                                dbias1=h1_sinks[0], dbias1b=h1_sinks[1] if len(h1_sinks) > 1 else None)
            h1_bias_done = True
        else:
            dh1 = dout
            h1_bias_done = dout_bias_done
        # h1 = conv1(a1) + b1 + skip(x)
        self._conv_param_grads(blk.conv1, dh1, c.a1, bias_done=h1_bias_done)
        da1 = self._dgrad(dh1, blk.conv1, self.conv_w(blk.conv1))
        # da1 / da0 are consumed only by the GroupNorm backward: dy_scratch lets it keep the pre-activation gradient there
        dh0, _ = ops.gn_bwd(da1, c.h0, None, c.sums1, blk.norm1.weight, blk.norm1.bias, _groups(cout),
                            params=c.params, act=True, drop_p=c.drop_p, seed=c.seed, seed_counter=self.seed_counter,
                            dgamma=self._grad(blk.norm1.weight), dbeta=self._grad(blk.norm1.bias), dparams=dparams,
                            dbias1=self._grad(blk.conv0.bias), dy_scratch=True)
        # h0 = conv0(a0) + b0
        self._conv_param_grads(blk.conv0, dh0, c.a0, bias_done=True)
        da0 = self._dgrad(dh0, blk.conv0, self.conv_w(blk.conv0))
        if has_skip_conv:
            self._conv_param_grads(blk.skip, dh1, c.x1, c.x2, bias_done=h1_bias_done)
            add = self._dgrad(dh1, blk.skip, self.conv_w(blk.skip, cin1, cin2), cin1, cin2)
            add_mode = 0
        else:
            add, add_mode = dh1, c.mode
        s0 = input_sinks[0] if input_sinks else None
        s1 = input_sinks[1] if input_sinks and len(input_sinks) > 1 else None
        return ops.gn_bwd(da0, c.x1, c.x2, c.sums0, blk.norm0.weight, blk.norm0.bias, _groups(cin),
                          act=True, resample=c.mode, dgamma=self._grad(blk.norm0.weight),
                          dbeta=self._grad(blk.norm0.bias), add=add, add_mode=add_mode, dbias1=s0, dbias1b=s1,
                          dy_scratch=True)

    # ------------------------------------------------------------------------------------------ embedding MLP
    def embed_fwd(self, c_noise, aug, save):
        net = self.net
        e = NS()
        pe = net.map_noise(c_noise)  # host glue on [B, mc]
        e.aug16 = None
        if net.map_augment is not None and aug is not None:
            a16 = torch.zeros(aug.shape[0], 16, device=aug.device, dtype=F32)
            a16[:, :aug.shape[1]] = aug
            e.aug16 = ops.cast_bf16(a16)
            pe = pe + ops.gemm_nt(e.aug16, self.aug_w())
        e.pe_b = ops.cast_bf16(pe)
        e.e0 = ops.gemm_nt(e.pe_b, self.lin_w(net.map_layer0), bias=net.map_layer0.bias)
        _, e.s0b = ops.silu(e.e0, want_f32=False)
        e.e1 = ops.gemm_nt(e.s0b, self.lin_w(net.map_layer1), bias=net.map_layer1.bias)
        _, e.embb = ops.silu(e.e1, want_f32=False)
        wall, ball = self.affine_all()
        params_all = ops.gemm_nt(e.embb, wall, bias=ball)  # [B, sum 2*Cout] fp32: every block's (scale | shift)
        if save is not None:
            save.append(e)
        return params_all

    def _linear_grads(self, lin, dyb, xb):
        """dW = dy^T x (MN-major x MN-major GEMM), db = column sums; dyb/xb bf16 [B, out] / [B, in]."""
        dw = ops.gemm_tn(dyb, xb)
        g = self._grad(lin.weight)
        if dw.shape == g.shape:
            g.add_(dw)
        else:
            g.add_(dw[:, :g.shape[1]])
        if lin.bias is not None:
            ops.col_sums(dyb, self._grad(lin.bias))

    def embed_bwd(self, e, dparams_all):
        net = self.net
        dpb = ops.cast_bf16(dparams_all)
        wall, _ = self.affine_all()
        if self.affine_pack is not None:  # all affine weights / biases are contiguous in the gradient arena
            # the [sum 2*Cout, emb] result is 123 MB for K = batch = 128: purely output bound.  When the arena's gradients
            # are known to be zero here (one micro-batch per optimizer step) a plain store replaces 31 M vector atomics.
            ops.gemm_tn(dpb, e.embb, out=self.affine_pack[2], accumulate=not self.affine_grad_overwrite)
            ops.col_sums(dpb, self.affine_pack[3])
        else:
            dwall = ops.gemm_tn(dpb, e.embb)  # [sum 2*Cout, emb]
            for _, m, off in self.block_list:
                o = m.affine.out_features
                ops.unpack_conv_wgrad(dwall[off:off + o], net.emb_channels, 0, 1, out=self._grad(m.affine.weight),
                                      accumulate=True)
                ops.col_sums(dpb[:, off:off + o], self._grad(m.affine.bias))
        # [B, sum 2*Cout] x [sum 2*Cout, emb]: K = 45 k with three output tiles -> split K over the idle SMs
        splits = max(1, min(40, wall.shape[0] // 1024))
        demb = ops.gemm_nn(dpb, wall, splits=splits)
        _, de1b = ops.silu_bwd(e.e1, demb, want_f32=False)
        self._linear_grads(net.map_layer1, de1b, e.s0b)
        ds0 = ops.gemm_nn(de1b, self.lin_w(net.map_layer1))
        _, de0b = ops.silu_bwd(e.e0, ds0, want_f32=False)
        self._linear_grads(net.map_layer0, de0b, e.pe_b)
        if e.aug16 is not None:
            dpe = ops.gemm_nn(de0b, self.lin_w(net.map_layer0))
            self._linear_grads(net.map_augment, ops.cast_bf16(dpe), e.aug16)

    # ------------------------------------------------------------------------------------------ decouple branch
    def decouple_fwd(self, seq, x, save):
        conv, sa = seq[0], seq[1]
        d = NS(seq=seq, x=x)
        d.h = ops.conv_fprop(x, self.conv_w(conv), bias=conv.bias)
        d.w_map = sa.map.weight.detach().reshape(-1)
        d.scal = torch.cat([sa.map.bias.detach(), sa.q_conv.weight.detach().reshape(-1), sa.q_conv.bias.detach(),
                            sa.k_conv.weight.detach().reshape(-1), sa.k_conv.bias.detach()])
        out, d.att, d.o = ops.spatial_att_fwd(d.h, x, d.w_map, d.scal)
        if save is not None:
            save.append(d)
        return out

    def decouple_bwd(self, d, dy):
        """Returns the gradient w.r.t. the bottleneck x of this branch (conv path + identity path)."""
        conv, sa = d.seq[0], d.seq[1]
        c = d.x.shape[-1]
        dw_map = torch.zeros(c, device=dy.device, dtype=F32)
        dscal = torch.zeros(5, device=dy.device, dtype=F32)
        dh = ops.spatial_att_bwd(dy, d.h, d.w_map, d.scal, d.att, d.o, dw_map, dscal)
        self._grad(sa.map.weight).add_(dw_map.reshape(sa.map.weight.shape))
        self._grad(sa.map.bias).add_(dscal[0:1])
        self._grad(sa.q_conv.weight).add_(dscal[1:2].reshape(1, 1, 1, 1))
        self._grad(sa.q_conv.bias).add_(dscal[2:3])
        self._grad(sa.k_conv.weight).add_(dscal[3:4].reshape(1, 1, 1, 1))
        self._grad(sa.k_conv.bias).add_(dscal[4:5])
        self._conv_param_grads(conv, dh, d.x)
        return self._dgrad(dh, conv, self.conv_w(conv), residual=dy)

    # ------------------------------------------------------------------------------------------ whole network
    def _run_fwd(self, xin, c_noise, aug, training, tape):
        net = self.net
        save = tape.items if tape is not None else None
        step_seed = 0
        if training:
            step_seed = self.base_seed * 1000003 + self._seed_next
            self._seed_next += 1
        emb_save = [] if tape is not None else None
        params_all = self.embed_fwd(c_noise, aug, emb_save)
        boff = {id(m): off for _, m, off in self.block_list}
        if tape is not None:
            tape.emb = emb_save[0]
            tape.dparams_all = torch.zeros_like(params_all)

        def run_block(m, x1, x2, idx):
            off = boff[id(m)]
            return self.block_fwd(m, x1, x2, params_all[:, off:off + m.affine.out_features], training,
                                  step_seed * 4099 + idx, save)

        x = xin
        skips = []  # output of every encoder entry
        idx = 0
        for name, m in net.enc.items():
            if hasattr(m, "affine"):
                x = run_block(m, x, None, idx)
            else:
                x = ops.conv_fprop(x, self.conv_w(m, c1=m.in_channels), bias=m.bias)
                if tape is not None:
                    tape.first = NS(conv=m, x=xin)
            idx += 1
            skips.append(x)
        outs = []
        # The two decoders only share their inputs (bottleneck, skips, embedding): the second one is enqueued on the
        # side stream, forked HERE (before decoder 1 is enqueued), so their kernels interleave on the SMs — most of
        # them leave a partial last wave, the 4x4 / 8x8 levels never fill the GPU.  Host order (and the tape) unchanged.
        fork = None
        if x.is_cuda:
            if self._side is None:
                self._side = torch.cuda.Stream()
            fork = torch.cuda.Event()
            fork.record(torch.cuda.current_stream())
        for di, (dec, dname, norm, oconv) in enumerate(((net.dec, "decouple1", net.out_norm, net.out_conv),
                                                       (net.dec2, "decouple2", net.out_norm2, net.out_conv2))):
            ctx = contextlib.nullcontext()
            if di == 1 and fork is not None:
                self._side.wait_event(fork)
                self._side_pending.append((x, skips, params_all))
                ctx = torch.cuda.stream(self._side)
            with ctx:
                h = self.decouple_fwd(getattr(net, dname), x, save)
                sk = list(skips)
                for name, m in dec.items():
                    x2 = sk.pop() if h.shape[-1] != m.in_channels else None
                    h = run_block(m, h, x2, idx)
                    idx += 1
                o = NS(x=h, norm=norm, conv=oconv)
                o.sums, o.a = ops.gn_forward(h, None, norm.weight, norm.bias, _groups(h.shape[-1]), norm.eps, act=True)
                f = ops.conv_fprop(o.a, self.conv_w(oconv), bias=oconv.bias, out_dtype=F32, keep_pad=True)
                if save is not None:
                    save.append(o)
                outs.append(f)  # [N,H,W,4] fp32, channels >= img_channels are zero
        self._join_side()
        if tape is not None:
            tape.n_skips = len(skips)
        return outs[0], outs[1]

    def forward(self, x, sigma, aug=None, training=False, need_grad=False):
        """EDMPrecond.forward.  x NCHW float, sigma [B] or scalar.  Returns (D_x, D_y, tape)."""
        if not x.is_cuda:
            raise RuntimeError("adm_b200: the UNet runs on CUDA (sm_100a) only; there is no CPU fallback")
        x = x.to(F32).contiguous()
        n = x.shape[0]
        sigma = sigma.to(F32).reshape(-1)
        if sigma.numel() == 1:
            sigma = sigma.expand(n)
        sigma = sigma.contiguous()
        tape = NS(items=[], x=x, sigma=sigma) if need_grad else None
        xin = ops.unet_input(x, sigma, ld_out=8)
        f1, f2 = self._run_fwd(xin, sigma.log(), aug, training, tape)
        d1, d2 = ops.unet_output(f1, f2, x, sigma)
        return d1, d2, tape

    def forward_raw(self, xin_nchw, noise_labels, aug=None):
        """DhariwalUNet.forward on an already scaled input; returns (F_x, F_y) NCHW fp32 (inference only)."""
        n = xin_nchw.shape[0]
        ones = torch.full((n,), 1.0, device=xin_nchw.device)  # c_in(1) == 1: reuse the input kernel as a layout change
        xin = ops.unet_input(xin_nchw.to(F32).contiguous(), ones, ld_out=8)
        f1, f2 = self._run_fwd(xin, noise_labels.to(F32).reshape(-1).expand(n).contiguous(), aug, False, None)
        c = self.net.out_channels
        return (f1[..., :c].permute(0, 3, 1, 2).contiguous(), f2[..., :c].permute(0, 3, 1, 2).contiguous())

    def backward(self, tape, dd1, dd2):
        """Accumulates parameter gradients for upstream gradients (dD_x, dD_y), NCHW fp32."""
        net = self.net
        c_img = net.out_channels
        df1, df2 = ops.unet_output_bwd(dd1.contiguous().float(), dd2.contiguous().float(), tape.sigma, ld_out=8)
        items = tape.items
        boff = {id(m): off for _, m, off in self.block_list}
        dskips = [None] * tape.n_skips
        dbott = None
        pos = len(items)
        for df in (df2, df1):  # decoders in reverse order of execution
            pos -= 1
            o = items[pos]
            dfv = df[..., :c_img]
            self._conv_param_grads(o.conv, dfv, o.a, dy_cols=df)
            da = self._dgrad(dfv, o.conv, self.conv_w(o.conv))
            # each kernel that produces the gradient at a block's output also accumulates its column sums into that
            # block's bias gradients (bias_sinks), so the decoder chain needs no separate col_sums passes
            sinks = self.bias_sinks(items[pos - 1].blk)
            dh, _ = ops.gn_bwd(da, o.x, None, o.sums, o.norm.weight, o.norm.bias, _groups(o.x.shape[-1]),
                               act=True, dgamma=self._grad(o.norm.weight), dbeta=self._grad(o.norm.bias),
                               dbias1=sinks[0], dbias1b=sinks[1] if len(sinks) > 1 else None,
                               dy_scratch=True)
            self._notify(o.conv, o.norm)
            si = 0  # forward pops skips from the end, so walking the decoder backwards meets skips[0], skips[1], ...
            while not hasattr(items[pos - 1], "seq"):
                pos -= 1
                c = items[pos]
                off = boff[id(c.blk)]
                prev = items[pos - 1]
                sinks = self.bias_sinks(prev.blk) if hasattr(prev, "blk") else None
                dx1, dx2 = self.block_bwd(c, dh, tape.dparams_all[:, off:off + c.blk.affine.out_features],
                                          dout_bias_done=True, input_sinks=sinks)
                self._notify(c.blk)
                if c.x2 is not None:
                    dskips[si] = dx2 if dskips[si] is None else ops.add_bf16(dskips[si], dx2)
                    si += 1
                dh = dx1
            pos -= 1
            dx = self.decouple_bwd(items[pos], dh)
            self._notify(items[pos].seq)
            dbott = dx if dbott is None else ops.add_bf16(dbott, dx)
        # encoder, last block first; skips[i] is the output of encoder entry i
        enc = list(net.enc.values())
        d = dbott
        for i in range(len(enc) - 1, -1, -1):
            g = d if dskips[i] is None else ops.add_bf16(d, dskips[i])
            m = enc[i]
            if hasattr(m, "affine"):
                pos -= 1
                c = items[pos]
                off = boff[id(m)]
                d, _ = self.block_bwd(c, g, tape.dparams_all[:, off:off + m.affine.out_features])
            else:
                self._conv_param_grads(m, g, tape.first.x)
            self._notify(m)
        assert pos == 0, pos
        self.embed_bwd(tape.emb, tape.dparams_all)
        self._notify(net, skip_affine=False)


class _UNetFn(torch.autograd.Function):
    """One autograd node for the whole preconditioned UNet.  ``anchor`` only exists to make autograd call backward;
    parameter gradients are accumulated into ``.grad`` by the engine itself."""

    @staticmethod
    def forward(ctx, anchor, engine, x, sigma, aug, training):
        d1, d2, tape = engine.forward(x, sigma, aug, training=training, need_grad=True)
        ctx.engine, ctx.tape = engine, tape
        return d1, d2

    @staticmethod
    def backward(ctx, g1, g2):
        tape, ctx.tape = ctx.tape, None
        if tape is None:
            raise RuntimeError("adm_b200 UNet: backward through the same forward twice is not supported")
        if g1 is None:
            g1 = torch.zeros_like(tape.x)
        if g2 is None:
            g2 = torch.zeros_like(tape.x)
        ctx.engine.backward(tape, g1, g2)
        return None, None, None, None, None, None


def unet_apply(engine, x, sigma, aug=None):
    net = engine.net
    want_grad = torch.is_grad_enabled() and any(p.requires_grad for p in net.parameters())
    if not want_grad:
        d1, d2, _ = engine.forward(x, sigma, aug, training=net.training, need_grad=False)
        return d1, d2
    anchor = torch.zeros((), device=x.device, requires_grad=True)
    return _UNetFn.apply(anchor, engine, x, sigma, aug, net.training)
