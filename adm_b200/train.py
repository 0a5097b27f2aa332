"""Data-parallel training step around the DDPM module: flat parameter/gradient arenas, bucketed NCCL all-reduce
overlapped with the engine's backward, fused clip + AdamW over the arena.

Mirrors the step body of the reference Trainer (/root/reference/train_uncond_dpm.py:247-310): micro-batch loop,
``clip_grad_norm_(1.0)`` (:292), AdamW(lr, weight_decay=1e-4) (:179-180), warm-up + polynomial LambdaLR (:169-182).
Semantics we define explicitly (the reference's DDP wiring is accidental, SURVEY §2): gradients are the MEAN over
ranks of per-rank gradients, reduced once per optimizer step (not per micro-batch).

``AutogradDataParallel`` gives the same semantics to a model that trains through torch autograd and a torch optimizer
(the conditional UNet of scripts/train_cond_ldm.py): one flat gradient arena, one all-reduce per optimizer step.
"""
from __future__ import annotations

import math

import torch
import torch.distributed as dist

from . import ops


def completion_order(net):
    """Parameters of EDMPrecond in the order their gradients are finalised by UNetEngine.backward."""
    m = net.model
    order = []

    def block_params(blk):
        names = []
        if blk.num_heads:
            names += ["proj", "qkv", "norm2"]
        names += ["conv1", "norm1", "conv0", "skip", "norm0"]
        for nme in names:
            sub = getattr(blk, nme, None)
            if sub is not None:
                order.extend(p for p in sub.parameters())

    for dec, dname, norm, oconv in ((m.dec2, "decouple2", m.out_norm2, m.out_conv2),
                                    (m.dec, "decouple1", m.out_norm, m.out_conv)):
        order.extend(oconv.parameters())
        order.extend(norm.parameters())
        for blk in reversed(list(dec.values())):
            block_params(blk)
        order.extend(getattr(m, dname).parameters())
    for blk in reversed(list(m.enc.values())):
        if hasattr(blk, "affine"):
            block_params(blk)
        else:
            order.extend(blk.parameters())
    # every block's affine (time-embedding) weight, then every bias, back to back in the engine's block order:
    # their gradients all come from ONE grouped GEMM at the end of backward, and the contiguous layout lets that GEMM
    # (and the forward one) address them as a single [sum 2*Cout, emb] matrix inside the arena.
    affine = [blk.affine for sec in (m.enc, m.dec, m.dec2) for blk in sec.values() if hasattr(blk, "affine")]
    order.extend(a.weight for a in affine)
    order.extend(a.bias for a in affine)
    order.extend(m.map_layer1.parameters())
    order.extend(m.map_layer0.parameters())
    if m.map_augment is not None:
        order.extend(m.map_augment.parameters())
    seen, out = set(), []
    for p in order:
        if id(p) not in seen:
            seen.add(id(p))
            out.append(p)
    rest = [p for p in net.parameters() if id(p) not in seen]
    return out + rest


class ParamArena:
    """Re-homes every parameter (and its .grad) of a module into two flat fp32 buffers, in gradient-completion order."""

    def __init__(self, module, order=None, align=8, channels_last=()):
        """channels_last: conv weights [Cout, Cin, k, k] to store physically as [Cout][k][k][Cin] — the packed operand
        order of the GEMM engine.  They keep their logical (reference) shape as a permuted view, so state_dict /
        load_state_dict are unaffected, and on CUDA they get a bf16 shadow (written by the fused AdamW kernel) plus a
        packed view of their gradient: ``p._adm_pack = (bf16 [Cout, k*k, Cin], fp32 grad [Cout, k*k, Cin], version,
        fp32 flat slice, bf16 [Cin, k*k, Cout] or None)``.  The last entry is the DGRAD shadow: the same weights
        transposed with the taps mirrored (Cout a multiple of 64), re-derived from the bf16 shadow by ONE batched tile
        transpose per optimizer step, so the data gradient of a conv runs through the fprop kernels on a K-major
        operand instead of the slower MN-major view of the fprop-packed weights."""
        params = order if order is not None else list(module.parameters())
        dev = params[0].device
        cl = {id(p) for p in channels_last}
        offs, total = [], 0
        for p in params:
            offs.append(total)
            total += (p.numel() + align - 1) // align * align
        self.params = params
        self.offsets = offs
        self.numel = total
        self.flat = torch.zeros(total, device=dev, dtype=torch.float32)
        self.grads = torch.zeros(total, device=dev, dtype=torch.float32)
        self.shadow = torch.zeros(total, device=dev, dtype=torch.bfloat16) if (cl and dev.type == "cuda") else None
        self.shadow_t = torch.zeros(total, device=dev, dtype=torch.bfloat16) if self.shadow is not None else None
        self.t_tiles = None
        tiles = []
        self._grad_views = []
        for p, o in zip(params, offs):
            n = p.numel()
            if id(p) in cl:
                co, ci, kh, kw = p.shape
                view = self.flat[o:o + n].view(co, kh, kw, ci).permute(0, 3, 1, 2)
                gview = self.grads[o:o + n].view(co, kh, kw, ci).permute(0, 3, 1, 2)
            else:
                view = self.flat[o:o + n].view(p.shape)
                gview = self.grads[o:o + n].view(p.shape)
            view.copy_(p.data)
            p.data = view
            p.grad = gview
            self._grad_views.append(gview)
            if id(p) in cl and self.shadow is not None:
                wt = None
                if self.shadow_t is not None and co % 64 == 0 and ci % 64 == 0 and o % 8 == 0:
                    wt = self.shadow_t[o:o + n].view(ci, kh * kw, co)
                    tiles.append(ops.weight_transpose_tiles(o, co, kh * kw, ci))
                p._adm_pack = (self.shadow[o:o + n].view(co, kh * kw, ci), self.grads[o:o + n].view(co, kh * kw, ci),
                               p._version, self.flat[o:o + n], wt)
        if tiles:
            self.t_tiles = torch.cat(tiles).to(dev)
        self.refresh_shadow()

    def refresh_shadow(self):
        """Re-derive the bf16 shadow from the fp32 masters (after construction or an out-of-band parameter write)."""
        if self.shadow is not None:
            ops.cast_bf16_into(self.flat, self.shadow)
            self.refresh_dgrad_shadow()
            for p in self.params:
                pk = getattr(p, "_adm_pack", None)
                if pk is not None:
                    p._adm_pack = (pk[0], pk[1], p._version, pk[3], pk[4])

    def refresh_dgrad_shadow(self):
        """shadow_t <- transposed / tap-mirrored bf16 shadow of every conv that has one (one kernel launch)."""
        if self.t_tiles is not None:
            ops.transpose_weight_tiles(self.shadow, self.shadow_t, self.t_tiles)

    def slice_of(self, params):
        """(offset, numel) of a run of parameters that sit back to back in the arena, else None."""
        idx = {id(p): i for i, p in enumerate(self.params)}
        first = idx.get(id(params[0]))
        if first is None:
            return None
        o = self.offsets[first]
        end = o
        for j, p in enumerate(params):
            i = idx.get(id(p))
            if i != first + j or self.offsets[i] != end:
                return None
            end += p.numel()
        return o, end - o

    def rebind_grads(self):
        """If someone set .grad to None (optimizer.zero_grad(set_to_none=True)), point it back into the arena."""
        for p, o, gv in zip(self.params, self.offsets, self._grad_views):
            g = p.grad
            if g is None or g.data_ptr() != self.grads.data_ptr() + 4 * o:
                p.grad = gv

    def zero_grad(self):
        self.grads.zero_()

    def broadcast(self, src=0, group=None, extra=()):
        """Rank `src`'s parameter arena, then each tensor of `extra` (in place), to every rank of `group`."""
        for t in (self.flat, *extra):
            dist.broadcast(t, src=src, group=group)


class AutogradDataParallel:
    """Data parallelism for a model that trains through torch autograd and a torch optimizer (the conditional UNet),
    where TrainStep's engine-driven reduction does not apply.

    The trainable parameters are re-homed into a ParamArena, so every ``.grad`` is a view of ONE flat fp32 buffer that
    autograd accumulates into.  The step is: ``zero_grad()``, forward + backward of every micro-batch, ``all_reduce()``
    once after the last one (one collective over the whole buffer), ``clip_mean_()``, optimizer step.  The gradient is
    the mean over ranks (DESIGN.md §1); the 1/world factor is folded into the clipping pass.  Gradients must be zeroed
    through ``zero_grad()``: setting ``.grad`` to None would detach it from the buffer."""

    def __init__(self, module, params, process_group=None):
        """module: the whole model (its parameters outside `params` and its buffers are replicated too);
        params: the trainable parameters."""
        self.module, self.pg = module, process_group
        self.world = dist.get_world_size(process_group) if (dist.is_available() and dist.is_initialized()) else 1
        self.arena = ParamArena(module, order=list(params))
        self.sync()

    @torch.no_grad()
    def sync(self, src=0):
        """Rank `src`'s weights to every rank: the trainable arena, the frozen parameters and every buffer.  Called at
        construction (replicas may start from different seeds) and after a checkpoint load on rank `src`."""
        if self.world == 1:
            return
        homed = {id(p) for p in self.arena.params}
        rest = [t.data for t in (*self.module.parameters(), *self.module.buffers()) if id(t) not in homed]
        self.arena.broadcast(src, self.pg, rest)

    def broadcast_object(self, obj, src=0):
        """A picklable value of rank `src` on every rank."""
        if self.world == 1:
            return obj
        box = [obj]
        dist.broadcast_object_list(box, src=src, group=self.pg)
        return box[0]

    @torch.no_grad()
    def sync_optimizer(self, opt, src=0):
        """Rank `src`'s torch.optim state to every rank: the hyperparameters of each parameter group except the
        learning rate (the trainer sets that every step) and the per-parameter state, allocated with rank `src`'s
        shapes, dtypes and devices on the ranks that have none (a fresh optimizer before its first step)."""
        if self.world == 1:
            return
        params = [p for g in opt.param_groups for p in g["params"]]
        meta = None
        if dist.get_rank(self.pg) == src:
            groups = [{k: v for k, v in g.items() if k not in ("params", "lr")} for g in opt.param_groups]
            state = []
            for p in params:
                st = opt.state.get(p, {})
                state.append(({k: (tuple(v.shape), v.dtype, v.device == p.device) for k, v in st.items()
                               if torch.is_tensor(v)},
                              {k: v for k, v in st.items() if not torch.is_tensor(v)}))
            meta = (groups, state)
        groups, state = self.broadcast_object(meta, src)
        for g, hyper in zip(opt.param_groups, groups):
            g.update(hyper)
        for p, (tensors, values) in zip(params, state):
            if not tensors and not values:
                continue
            st = opt.state[p]
            st.update(values)
            for k, (shape, dtype, on_param) in tensors.items():
                t = st.get(k)
                if not torch.is_tensor(t) or tuple(t.shape) != shape or t.dtype != dtype:
                    t = st[k] = torch.empty(shape, dtype=dtype, device=p.device if on_param else "cpu")
                if t.device == p.device:
                    dist.broadcast(t, src=src, group=self.pg)
                else:  # a host scalar (torch keeps a non-capturable step count there): through the parameter's device
                    buf = t.to(p.device)
                    dist.broadcast(buf, src=src, group=self.pg)
                    t.copy_(buf)

    def zero_grad(self):
        self.arena.zero_grad()

    def all_reduce(self):
        """Sum the gradient buffer over the ranks: one collective, stream-ordered after the backward that filled it."""
        if self.world > 1:
            dist.all_reduce(self.arena.grads, op=dist.ReduceOp.SUM, group=self.pg)

    def clip_mean_(self, max_norm):
        """Summed gradients -> their mean over the ranks, clipped to `max_norm` the way
        ``torch.nn.utils.clip_grad_norm_`` clips it, in one pass over the buffer and without a host synchronisation
        (it can be captured in a CUDA graph).  Returns the norm of the mean gradient before clipping."""
        g = self.arena.grads
        norm = torch.linalg.vector_norm(g) / self.world
        g.mul_(torch.clamp(max_norm / (norm + 1e-6), max=1.0) / self.world)
        return norm


def lr_lambda(step, train_num_steps, lr, min_lr, warmup=5000):
    """train_uncond_dpm.py:169-177: linear warm-up to 1 over `warmup` steps, then (1 - iter/total)^0.96 with a floor."""
    if step < warmup:
        return (step + 1) / warmup
    return max(min_lr / lr, (1 - (step - warmup) / max(1, train_num_steps - warmup)) ** 0.96)


class TrainStep:
    """One data-parallel optimizer step of DDM-const training on this rank's GPU."""

    def __init__(self, dpm, lr=1e-4, weight_decay=1e-4, betas=(0.9, 0.999), eps=1e-8, max_grad_norm=1.0,
                 grad_accum=1, bucket_mb=64, process_group=None, lr_schedule=None):
        self.dpm = dpm
        self.net = dpm.model
        self.engine = self.net.model.engine
        self.world = dist.get_world_size(process_group) if (dist.is_available() and dist.is_initialized()) else 1
        self.pg = process_group
        self.arena = ParamArena(self.net, completion_order(self.net), channels_last=self.engine.packable_params())
        self._bind_affine()
        self._grads_clean = True  # the gradient arena is all zeros (fresh, or zeroed by the last optimizer step)
        self._bind_qkv()
        self.m = torch.zeros_like(self.arena.flat)
        self.v = torch.zeros_like(self.arena.flat)
        self.lr, self.wd, self.betas, self.eps = lr, weight_decay, betas, eps
        self.max_grad_norm = max_grad_norm
        self.grad_accum = grad_accum
        self.step_count = 0
        self.lr_schedule = lr_schedule
        dev = self.arena.flat.device
        self.sqnorm = torch.zeros(1, device=dev, dtype=torch.float32)
        self.hyper = torch.zeros(3, device=dev, dtype=torch.float32)
        # per-step scalars travel through a small ring of pinned buffers: the H2D copy is asynchronous, and the host may
        # run several (graph-replayed) steps ahead of the device, so a single buffer would be overwritten too early
        self._hyper_ring = [torch.zeros(3, dtype=torch.float32).pin_memory() if dev.type == "cuda" else torch.zeros(3)
                            for _ in range(4)]
        self._hyper_events = [None] * 4
        self._ring_i = 0
        # gradient buckets in completion order
        n = self.arena.numel
        per = max(1, bucket_mb * (1 << 20) // 4)
        self.buckets = [(s, min(n, s + per)) for s in range(0, n, per)]
        self.comm_stream = torch.cuda.Stream(device=dev) if (self.world > 1 and dev.type == "cuda") else None
        self._seg_capture = None
        self.segments = None
        self._param_end = {}
        for p, o in zip(self.arena.params, self.arena.offsets):
            self._param_end[id(p)] = o + p.numel()
        self.sync_params(moments=False)
        # device-resident step counter mixed into every dropout seed (fresh masks per CUDA-graph replay)
        self.seed_counter = torch.zeros(1, device=dev, dtype=torch.int64) if dev.type == "cuda" else None
        self.engine.seed_counter = self.seed_counter  # passed per call to the GroupNorm kernels (no global state)
        self.graph = None

    def _bind_affine(self):
        """Hand the engine ONE [sum 2*Cout, emb] view of all affine weights (bf16 shadow), biases and their gradients."""
        a, eng = self.arena, self.engine
        eng.affine_pack = None
        if a.shadow is None:
            return
        mods = [m.affine for _, m, _ in eng.block_list]
        ws, bs = a.slice_of([m.weight for m in mods]), a.slice_of([m.bias for m in mods])
        if ws is None or bs is None:
            return
        emb = mods[0].in_features
        t = ws[1] // emb
        assert t == eng.affine_total and bs[1] == t
        eng.affine_pack = (a.shadow[ws[0]:ws[0] + ws[1]].view(t, emb), a.flat[bs[0]:bs[0] + t],
                           a.grads[ws[0]:ws[0] + ws[1]].view(t, emb), a.grads[bs[0]:bs[0] + t],
                           a.flat[ws[0]:ws[0] + ws[1]], tuple(m.weight._version for m in mods))

    def _bind_qkv(self):
        """The qkv projections run in (q | k | v) x head x d row order (the reference interleaves (head, d, {q,k,v}),
        unet/uncond_unet.py:205).  Instead of re-packing 24 weights and biases every step, keep ONE bf16 buffer with all of
        them in executed order plus a byte-offset table, and re-derive it from the arena's bf16 shadow (weights) and fp32
        masters (biases) with two batched row-gather launches per optimizer step."""
        a, eng = self.arena, self.engine
        self._qkv = None
        if a.shadow is None:
            return
        off = {id(p): o for p, o in zip(a.params, a.offsets)}
        blocks = [m for _, m, _ in eng.block_list
                  if m.num_heads and m.out_channels % 64 == 0 and (m.out_channels // m.num_heads) % 64 == 0
                  and id(m.qkv.weight) in off and id(m.qkv.bias) in off]
        if not blocks or len({m.out_channels for m in blocks}) != 1:
            return
        c = blocks[0].out_channels
        dev = a.flat.device
        wbuf = torch.empty(len(blocks) * 3 * c * c, device=dev, dtype=torch.bfloat16)
        bbuf = torch.empty(len(blocks) * 3 * c, device=dev, dtype=torch.float32)
        wt, bt = [], []
        for i, m in enumerate(blocks):
            perm = eng.qkv_perm(c, m.num_heads)[1].cpu()  # executed row r holds reference row perm[r]
            r = torch.arange(3 * c)
            wt.append(torch.stack([(off[id(m.qkv.weight)] + perm * c) * 2, (i * 3 * c * c + r * c) * 2], dim=1))
            bt.append(torch.stack([(off[id(m.qkv.bias)] + perm) * 4, (i * 3 * c + r) * 4], dim=1))
            w, b = m.qkv.weight, m.qkv.bias
            w._adm_qkv = (wbuf[i * 3 * c * c:(i + 1) * 3 * c * c].view(3 * c, 1, c), bbuf[i * 3 * c:(i + 1) * 3 * c],
                          (w._version, b._version))
        self._qkv = (wbuf, bbuf, torch.cat(wt).to(torch.int64).contiguous().to(dev),
                     torch.cat(bt).to(torch.int64).contiguous().to(dev), c, blocks)

    def refresh_derived(self):
        """Operands derived from the arena once per optimizer step: the transposed dgrad shadow and the qkv packs."""
        a = self.arena
        a.refresh_dgrad_shadow()
        if self._qkv is not None:
            wbuf, bbuf, wtab, btab, c, blocks = self._qkv
            ops.gather_rows(a.shadow, wbuf, wtab, 2 * c)
            ops.gather_rows(a.flat, bbuf, btab, 4)
            for m in blocks:
                w, b = m.qkv.weight, m.qkv.bias
                w._adm_qkv = (w._adm_qkv[0], w._adm_qkv[1], (w._version, b._version))

    def refresh(self):
        """Call after parameters were written outside the fused optimizer (load_state_dict, manual edits)."""
        self.arena.refresh_shadow()
        self.refresh_derived()
        self.engine.invalidate()

    def sync_params(self, src=0, moments=True):
        """Data parallelism needs identical replicas: rank `src`'s parameter arena (and optimizer moments, when they
        exist) are broadcast to every rank — what accelerate / DDP do for the reference at wrap time
        (train_uncond_dpm.py:197-198).  Called at construction and after a checkpoint load."""
        if self.world > 1:
            self.arena.broadcast(src, self.pg, (self.m, self.v) if moments else ())
        self.refresh()

    # ------------------------------------------------------------------------------------------ gradient reduction
    # The arena is laid out in gradient-completion order, so "everything below offset X is final" grows monotonically
    # during backward.  Each bucket is all-reduced (NCCL, sum) on a side stream the moment it is entirely final, which
    # overlaps the transfer over NVLink with the rest of the backward pass.  1/world is folded into the AdamW kernel.
    def _arm(self):
        self._done_upto, self._next_bucket = 0, 0
        self.engine.grad_hook = self._on_grads if (self.world > 1 or self._seg_capture is not None) else None

    def _on_grads(self, params):
        for p in params:
            e = self._param_end.get(id(p))
            if e is not None and e > self._done_upto:
                self._done_upto = e
        self._flush(self._done_upto)

    def _flush(self, upto):
        if self._next_bucket >= len(self.buckets) or self.buckets[self._next_bucket][1] > upto:
            return
        if self._seg_capture is not None:  # segmented graph capture: cut the graph here, reduce between replays
            first = self._next_bucket
            while self._next_bucket < len(self.buckets) and self.buckets[self._next_bucket][1] <= upto:
                self._next_bucket += 1
            self._cut_segment((first, self._next_bucket))
            return
        if self.comm_stream is None:  # host tensors (gloo tests): reduce synchronously
            while self._next_bucket < len(self.buckets) and self.buckets[self._next_bucket][1] <= upto:
                s, e = self.buckets[self._next_bucket]
                dist.all_reduce(self.arena.grads[s:e], op=dist.ReduceOp.SUM, group=self.pg)
                self._next_bucket += 1
            return
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self.comm_stream.wait_event(ev)
        with torch.cuda.stream(self.comm_stream):
            while self._next_bucket < len(self.buckets) and self.buckets[self._next_bucket][1] <= upto:
                s, e = self.buckets[self._next_bucket]
                dist.all_reduce(self.arena.grads[s:e], op=dist.ReduceOp.SUM, group=self.pg)
                self._next_bucket += 1

    def _allreduce(self):
        """Reduce whatever the overlapped path has not launched yet, then join the side stream."""
        if self.world == 1:
            return
        self._flush(self.arena.numel)
        if self.comm_stream is not None:
            torch.cuda.current_stream().wait_stream(self.comm_stream)
        self.engine.grad_hook = None

    # ------------------------------------------------------------------------------------------ the step
    def _push_hyper(self):
        """lr, 1 - beta1^step, sqrt(1 - beta2^step) of the CURRENT step_count -> device (stream-ordered, eager)."""
        i = self._ring_i
        self._ring_i = (i + 1) % len(self._hyper_ring)
        if self._hyper_events[i] is not None:
            self._hyper_events[i].synchronize()  # the copy that last used this slot has been consumed
        buf = self._hyper_ring[i]
        step = self.step_count
        buf[0] = self.lr * (self.lr_schedule(step - 1) if self.lr_schedule is not None else 1.0)
        buf[1] = 1.0 - self.betas[0] ** step
        buf[2] = math.sqrt(1.0 - self.betas[1] ** step)
        self.hyper.copy_(buf, non_blocking=True)
        if self.hyper.is_cuda:
            ev = torch.cuda.Event()
            ev.record()
            self._hyper_events[i] = ev

    def optimizer_step(self):
        self.step_count += 1
        self._push_hyper()
        if self.seed_counter is not None:
            self.seed_counter.add_(1)
        self.device_update()

    # ------------------------------------------------------------------------------------------ CUDA graph
    def capture(self, x_example, warmup=2):
        """Captures one full step (forward, backward, [all-reduce], clip + AdamW, weight re-pack) on `x_example`'s
        shape into a CUDA graph.  Per-step scalars (lr, bias corrections, dropout seed counter) live in device memory."""
        assert self.grad_accum == 1, "graph capture covers the single-micro-batch step"
        self.static_x = x_example.clone()
        kw = self._static_augment(x_example)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self.micro_step(self.static_x, **kw)
                self.optimizer_step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        from . import _lib
        l0 = _lib.load().adm_launch_count()
        with torch.cuda.graph(g):
            self.seed_counter.add_(1)
            self.static_loss = self.micro_step(self.static_x, **kw)
            self.device_update()
        self.launches_per_step = _lib.load().adm_launch_count() - l0  # kernels of ours inside one replay
        self.graph = g
        return g

    def _static_augment(self, x_example):
        """With use_augment the augmentation (data glue with a data-dependent padding, ddm/augment.py:236-250) runs
        eagerly BEFORE each replay; the graph reads the augmented batch and its labels from static tensors."""
        self.static_aug = None
        if self.dpm.use_augment and self.dpm.augment is not None:
            _, lab = self.dpm.augment(x_example)
            self.static_aug = torch.zeros_like(lab)
            return {"augment_labels": self.static_aug}
        return {}

    def prefetch(self, x):
        """Stage the NEXT batch (device or pinned host tensor) for the following replay().  With an augmentation pipe this
        runs the pipe on a side stream, i.e. concurrently with the step that is executing — its ~40 small kernels fill
        the gaps of the step instead of sitting in front of it."""
        if getattr(self, "static_aug", None) is None:
            self._pending = (x, None, None)
            return
        if getattr(self, "_aug_stream", None) is None:
            self._aug_stream = torch.cuda.Stream()
        with torch.cuda.stream(self._aug_stream):
            xa, lab = self.dpm.augment(x.to(self.static_x.device, non_blocking=True))
            ev = torch.cuda.Event()
            ev.record()
        self._pending = (xa, lab, ev)

    def replay(self, x=None):
        """One optimizer step through the captured graph on the batch staged by prefetch() (or on `x`, staged now)."""
        if x is not None:
            self.prefetch(x)
        pend, self._pending = getattr(self, "_pending", None), None
        if pend is not None:
            xa, lab, ev = pend
            if ev is None:
                self.static_x.copy_(xa, non_blocking=True)
            else:
                cur = torch.cuda.current_stream()
                cur.wait_event(ev)
                self.static_x.copy_(xa)
                self.static_aug.copy_(lab)
                xa.record_stream(cur)
                lab.record_stream(cur)
        self.step_count += 1
        self._push_hyper()
        if self.segments is not None:
            return self._replay_segments()
        self.graph.replay()
        return self.static_loss

    # ------------------------------------------------------------------------------------------ segmented graphs (DP)
    # With several ranks the step cannot be ONE graph (capturing the NCCL collectives hung on this stack), and eager
    # launching makes the host the bottleneck (~1200 launches per step).  So the step is captured as a CHAIN of graphs,
    # cut at every point where a gradient bucket becomes complete; between two replays the bucket's all-reduce is
    # launched eagerly on the communication stream, which keeps the overlap of the transfer with the rest of backward.
    def _cut_segment(self, bucket_range):
        cap = self._seg_capture
        cap["graph"].capture_end()
        cap["segments"].append((cap["graph"], bucket_range))
        g = torch.cuda.CUDAGraph()
        g.capture_begin(pool=cap["pool"])
        cap["graph"] = g

    def capture_dp(self, x_example, warmup=2, t=None, noise=None):
        """t / noise: optional STATIC tensors baked into the graphs (tests); by default they are drawn inside."""
        assert self.grad_accum == 1, "graph capture covers the single-micro-batch step"
        self.static_x = x_example.clone()
        kw = self._static_augment(x_example)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self.micro_step(self.static_x, t, noise, **kw)
                self.optimizer_step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.pg)
        from . import _lib
        l0 = _lib.load().adm_launch_count()
        pool = torch.cuda.graph_pool_handle()
        self._cap_stream = torch.cuda.Stream()
        self._cap_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self._cap_stream):
            g = torch.cuda.CUDAGraph()
            g.capture_begin(pool=pool)
            self._seg_capture = dict(graph=g, segments=[], pool=pool)
            try:
                self.seed_counter.add_(1)
                self.static_loss = self.micro_step(self.static_x, t, noise, **kw)
                self._flush(self.arena.numel)  # whatever is left of the gradient arena
                self.engine.grad_hook = None
                a = self.arena
                gscale = 1.0 / (self.world * self.grad_accum)
                self.sqnorm.zero_()
                ops.sq_norm(a.grads, self.sqnorm)
                ops.adamw(a.flat, a.grads, self.m, self.v, self.lr, self.betas[0], self.betas[1], self.eps, self.wd,
                          max(1, self.step_count), grad_scale=gscale, max_norm=self.max_grad_norm, sqnorm=self.sqnorm,
                          hyper_dev=self.hyper, p_bf16=a.shadow)
                self.refresh_derived()
                a.zero_grad()
                self._grads_clean = True
                self.engine.invalidate()
                self._seg_capture["graph"].capture_end()
                self.segments = self._seg_capture["segments"] + [(self._seg_capture["graph"], None)]
            finally:
                self._seg_capture = None
        torch.cuda.current_stream().wait_stream(self._cap_stream)
        self.launches_per_step = _lib.load().adm_launch_count() - l0
        return self.segments

    def _replay_segments(self):
        cur = torch.cuda.current_stream()
        for g, rng in self.segments:
            if rng is None:  # the optimizer segment: every bucket must have been reduced
                if self.comm_stream is not None:
                    cur.wait_stream(self.comm_stream)
                g.replay()
                break
            g.replay()
            if self.world > 1:
                ev = torch.cuda.Event()
                ev.record(cur)
                self.comm_stream.wait_event(ev)
                with torch.cuda.stream(self.comm_stream):
                    for b in range(rng[0], rng[1]):
                        s, e = self.buckets[b]
                        dist.all_reduce(self.arena.grads[s:e], op=dist.ReduceOp.SUM, group=self.pg)
        return self.static_loss

    def device_update(self):
        """Everything after backward that runs on the device (capturable in a CUDA graph)."""
        a = self.arena
        self._allreduce()
        gscale = 1.0 / (self.world * self.grad_accum)
        self.sqnorm.zero_()
        ops.sq_norm(a.grads, self.sqnorm)
        ops.adamw(a.flat, a.grads, self.m, self.v, self.lr, self.betas[0], self.betas[1], self.eps, self.wd,
                  max(1, self.step_count), grad_scale=gscale, max_norm=self.max_grad_norm, sqnorm=self.sqnorm,
                  hyper_dev=self.hyper, p_bf16=a.shadow)
        self.refresh_derived()
        a.zero_grad()
        self._grads_clean = True
        self.engine.invalidate()

    def micro_step(self, x, t=None, noise=None, last=True, **kw):
        """forward + backward of one micro-batch; returns the (detached) loss tensor.  Gradient reduction is armed only
        on the last micro-batch of an accumulation window."""
        self.arena.rebind_grads()
        if last:
            self._arm()
        else:
            self.engine.grad_hook = None
        # first backward into a zeroed arena: the grouped affine weight gradient may be stored instead of accumulated
        self.engine.affine_grad_overwrite = self._grads_clean and self.engine.affine_pack is not None
        self._grads_clean = False
        if set(kw) <= {"augment_labels"}:
            return self._direct_step(x, t, noise, kw.get("augment_labels"))
        if t is None:
            loss, _ = self.dpm(x, **kw)
        else:
            loss, _ = self.dpm.p_losses(x, t, noise=noise, **kw)
        loss.backward()
        return loss.detach()

    def _direct_step(self, x, t, noise, aug):
        """DDPM.forward + p_losses + backward (ddm_const.py:274-364) driven straight through the engine on the calling
        thread — K1 q_sample, UNet forward with tape, K2 loss + gradients, hand-written backward — without building an
        autograd graph (same arithmetic as ``dpm(x)`` followed by ``loss.backward()``)."""
        dpm = self.dpm
        if not x.is_cuda:
            raise RuntimeError("adm_b200.TrainStep runs on CUDA (sm_100a) only; there is no CPU fallback")
        with torch.no_grad():
            if dpm.scale_input != 1:
                x = x * dpm.scale_input
            if t is None:
                t = torch.rand(x.shape[0], device=x.device) * (1. - dpm._eps) + dpm._eps
            if noise is None:
                noise = torch.randn_like(x) if dpm.start_dist == "normal" else 2 * torch.rand_like(x) - 1.
            if aug is None and dpm.use_augment and dpm.augment is not None:
                x, aug = dpm.augment(x)
            x = x.contiguous().float()
            noise = noise.contiguous().float()
            x_noisy = ops.qsample(x, noise, t)
            d1, d2, tape = self.engine.forward(x_noisy, t, aug, training=self.net.training, need_grad=True)
            lps, dc, de = ops.ddm_loss(d1, d2, x, noise, t, dpm._eps, bool(dpm.weighting_loss), dpm._loss_flags())
            self.engine.backward(tape, dc, de)
            return lps[:x.shape[0]].sum() / x.shape[0]

    def __call__(self, batches):
        """batches: list of `grad_accum` image tensors (this rank's shard).  Returns the mean loss tensor."""
        total = None
        for i, x in enumerate(batches):
            l = self.micro_step(x, last=(i == len(batches) - 1))
            total = l if total is None else total + l
        self.optimizer_step()
        return total / len(batches)
