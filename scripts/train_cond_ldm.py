#!/usr/bin/env python
"""Conditional latent training entry point: the role of /root/reference/train_cond_ldm.py (`accelerate launch
train_cond_ldm.py --cfg ...`) on one or several GPUs, without accelerate:

    python scripts/train_cond_ldm.py --cfg configs/super-resolution/div2k_cond_ddm_const_ldm.yaml [--graph]
    torchrun --nproc-per-node N scripts/train_cond_ldm.py --cfg configs/super-resolution/div2k_cond_ddm_const_ldm.yaml [--graph]

Builds the frozen first stage, the conditional UNet and the LatentDiffusion module from the YAML with
construct_class_by_name (train_cond_ldm.py:37-62) and runs the reference's loop (:212-330): micro-batches through
``LatentDiffusion.training_step`` (frozen AE encode + DDM-const step on the sm_100a kernels under torch autograd), clip 1.0,
torch AdamW, warm-up / polynomial LambdaLR, EMA, ``model-{k}.pt`` checkpoints with the reference's keys (the optimizer here IS
torch.optim.AdamW, so 'opt' and 'lr_scheduler' interchange with the reference's files too).  ``--graph`` replays the whole
step (AE encode, forward, autograd backward, clip, AdamW) as one CUDA graph, the way ``bench.py --config div2k`` measures it.

Under torchrun every rank trains a replica of rank 0's weights on its own data (``adm_b200.train.AutogradDataParallel``):
the gradients of each optimizer step are summed over the ranks in ONE all-reduce after the last micro-batch and clipped
as their mean; rank 0 alone keeps the EMA, logs and saves, and a resume reads rank 0's file and broadcasts it.  With
``--graph`` and several ranks the step is two CUDA graphs (forward + backward, then clip + AdamW) with the all-reduce
launched eagerly between them; one rank keeps the single graph.  Measured with ``tools/bench_cond_dp.py`` on one NVIDIA
B200 at a 1000 W power limit, DIV2K config at batch 8 with ``--graph``: 95.7 ms/step, 83.6 img/s at N = 1; N >= 2 not
measured yet (DESIGN.md §5).
"""
import argparse
import os
import sys
from pathlib import Path

import torch
import torch.distributed as dist
import yaml

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from adm_b200.ddm.ema import EMA  # noqa: E402
from adm_b200.train import AutogradDataParallel  # noqa: E402
from scripts.train_uncond_ldm import build_model  # noqa: E402


def synthetic_loader(batch, image_size, down, seed):
    """{'image': [B,3,H,W], 'cond': [B,3,H/down,W/down]} in [-1, 1]: the super-resolution pairs of the DIV2K config
    (pinned for asynchronous copies when there is a GPU)."""
    g = torch.Generator().manual_seed(seed)
    pin = (lambda x: x.pin_memory()) if torch.cuda.is_available() else (lambda x: x)
    while True:
        yield {"image": pin(2 * torch.rand(batch, 3, *image_size, generator=g) - 1),
               "cond": pin(2 * torch.rand(batch, 3, image_size[0] // down, image_size[1] // down, generator=g) - 1)}


def sharded_cycle(loader, sampler):
    """Endless iteration over a DataLoader with a DistributedSampler, reshuffled every epoch."""
    epoch = 0
    while True:
        sampler.set_epoch(epoch)
        yield from loader
        epoch += 1


def make_loader(data_cfg, batch, down, rank=0, world=1):
    """This rank's endless batch stream: synthetic pairs seeded with the rank, or the configured dataset (a
    DistributedSampler shard with drop_last when there are several ranks)."""
    d = data_cfg
    if d.get("class_name", "synthetic") == "synthetic":
        return synthetic_loader(batch, d["image_size"], down, seed=rank)
    from adm_b200.ddm.utils import construct_class_by_name
    from adm_b200.trainer import cycle
    ds = construct_class_by_name(**{k: v for k, v in d.items() if k not in ("batch_size", "num_workers")})
    if world > 1:
        sampler = torch.utils.data.DistributedSampler(ds, num_replicas=world, rank=rank, shuffle=True, drop_last=True)
        return sharded_cycle(torch.utils.data.DataLoader(ds, batch_size=batch, sampler=sampler, pin_memory=True,
                                                         num_workers=d.get("num_workers", 0), drop_last=True), sampler)
    return cycle(torch.utils.data.DataLoader(ds, batch_size=batch, shuffle=True, pin_memory=True,
                                             num_workers=d.get("num_workers", 0), drop_last=True))


class CondTrainer:
    """train_cond_ldm.py:96-330 without accelerate / tensorboard.  Data parallel when a process group of several ranks
    is initialised; the single-rank step is exactly the one-GPU loop."""

    def __init__(self, model, data_loader, gradient_accumulate_every=1, train_lr=1e-4, train_wd=1e-4,
                 train_num_steps=100000, save_and_sample_every=1000, results_folder="./results", log_freq=20,
                 resume_milestone=0, cfg=None, use_graph=False):
        cfg = cfg or {}
        self.model, self.dl = model, iter(data_loader)
        self.accum, self.train_num_steps = gradient_accumulate_every, train_num_steps
        self.save_and_sample_every, self.log_freq, self.train_lr = save_and_sample_every, log_freq, train_lr
        tcfg = cfg.get("trainer", {})
        warmup_iter, min_lr = tcfg.get("warmup_iter", 5000), tcfg.get("min_lr", 1e-6)

        def warm_up_lr(it):  # train_cond_ldm.py:139-146
            if it <= warmup_iter:
                return (it + 1) / warmup_iter
            return max((1 - (it - warmup_iter) / train_num_steps) ** 0.96, min_lr / train_lr)
        self.lr_lambda = warm_up_lr
        self.params = [p for p in model.parameters() if p.requires_grad]
        self.device = self.params[0].device
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        # Several ranks: rank 0's weights everywhere, every .grad a view of one flat buffer summed once per step.
        # BatchNorm buffers of the RelationNet stems are not synchronised per step (the reference's DDP broadcasts rank
        # 0's at every forward): training-mode BatchNorm normalises with batch statistics, so the running statistics
        # change no gradient, and the only ones that reach a checkpoint are rank 0's, the rank that saves.
        multi = dist.is_initialized() and dist.get_world_size() > 1
        self.dp = AutogradDataParallel(model, self.params) if multi else None
        self.use_graph = use_graph and gradient_accumulate_every == 1
        # the learning rate lives in a device scalar so that a captured step replays with the scheduler's current value
        self.lr_t = torch.tensor(train_lr * warm_up_lr(0), device=self.device, dtype=torch.float32)
        self.opt = torch.optim.AdamW(self.params, lr=self.lr_t, weight_decay=train_wd, fused=True,
                                     capturable=self.use_graph)
        self.results_folder = Path(results_folder)
        self.ema = None
        if self.rank == 0:
            self.results_folder.mkdir(exist_ok=True, parents=True)
            self.ema = EMA(model, ema_model=None, beta=0.9996, update_after_step=tcfg.get("ema_update_after_step", 100),
                           update_every=tcfg.get("ema_update_every", 10))
        self.step, self.graph, self.graph_update, self.static = 0, None, None, None
        found = os.path.isfile(str(self.results_folder / f"model-{resume_milestone}.pt"))
        if self.dp is not None:
            found = self.dp.broadcast_object(found)  # only rank 0 is guaranteed to have the file
        if found:
            self.load(resume_milestone)
        self.start_step = self.step

    # ------------------------------------------------------------------------------------------ checkpoints (:176-210)
    def save(self, milestone):
        if self.rank != 0:
            return
        data = {"step": self.step, "model": self.model.state_dict(), "opt": self.opt.state_dict(),
                "lr_scheduler": {"last_epoch": self.step}, "ema": self.ema.state_dict(), "scaler": None}
        torch.save(data, str(self.results_folder / f"model-{milestone}.pt"))

    def load(self, milestone):
        """Rank 0 reads the file; with several ranks its weights, AdamW state and step then go to every rank."""
        if self.rank == 0:
            data = torch.load(str(self.results_folder / f"model-{milestone}.pt"), map_location="cpu", weights_only=False)
            self.model.load_state_dict(data["model"])
            self.step = data["step"]
            self.opt.load_state_dict(data["opt"])
            if "ema" in data:
                self.ema.load_state_dict(data["ema"])
        if self.dp is not None:
            self.step = self.dp.broadcast_object(self.step)
            self.dp.sync()
            self.dp.sync_optimizer(self.opt)
        self.opt.param_groups[0]["lr"] = self.lr_t  # keep the device scalar (load_state_dict restores a copy)

    # ------------------------------------------------------------------------------------------ the loop (:212-330)
    def _to_device(self, batch):
        return {k: (v.to(self.device, non_blocking=True) if torch.is_tensor(v) else v) for k, v in batch.items()}

    def _backward(self, batches):
        """Forward and backward of every micro-batch (gradients accumulate); returns the mean loss."""
        total = None
        for batch in batches:
            loss, _ = self.model.training_step(batch)
            (loss / len(batches)).backward()
            total = loss.detach() if total is None else total + loss.detach()
        return total / len(batches)

    def _one(self, batches):
        if self.dp is None:
            self.opt.zero_grad(set_to_none=True)
            loss = self._backward(batches)
            torch.nn.utils.clip_grad_norm_(self.params, 1.0)
        else:
            self.dp.zero_grad()
            loss = self._backward(batches)
            self.dp.all_reduce()  # once per optimizer step, after the last micro-batch
            self.dp.clip_mean_(1.0)
        self.opt.step()
        return loss

    def _capture(self):
        """One rank: the whole step as one graph.  Several ranks: the NCCL all-reduce stays outside the graphs
        (capturing collectives hung on this stack, DESIGN.md §5), so forward + backward into the gradient buffer is
        one graph and clip + AdamW another, sharing its memory pool."""
        stream = torch.cuda.current_stream()
        if self.dp is None:
            torch.cuda.synchronize()
            self.opt.zero_grad(set_to_none=True)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=stream):
                self.static_loss = self._one([self.static])
            return
        dist.barrier()
        torch.cuda.synchronize()  # no collective in flight while a graph is being captured
        self.graph, self.graph_update = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=stream):
            self.dp.zero_grad()
            self.static_loss = self._backward([self.static])
        with torch.cuda.graph(self.graph_update, pool=self.graph.pool(), stream=stream):
            self.dp.clip_mean_(1.0)
            self.opt.step()

    def _replay(self):
        self.graph.replay()
        if self.graph_update is not None:
            self.dp.all_reduce()
            self.graph_update.replay()
        return self.static_loss

    def train_one_step(self):
        self.lr_t.fill_(self.train_lr * self.lr_lambda(self.step))
        batches = [self._to_device(next(self.dl)) for _ in range(self.accum)]
        if self.use_graph:
            # three eager steps in this process first (allocator warm-up, lazy initialisation), after a resume too
            if self.graph is None and self.step - self.start_step >= 3:
                self.static = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in batches[0].items()}
                self._capture()
            if self.graph is not None:
                for k, v in batches[0].items():
                    if torch.is_tensor(v):
                        self.static[k].copy_(v, non_blocking=True)
                loss = self._replay()
            else:
                loss = self._one(batches)
        else:
            loss = self._one(batches)
        self.step += 1
        if self.ema is not None:
            self.ema.update()
        return loss

    def train(self):
        while self.step < self.train_num_steps:
            loss = self.train_one_step()
            if self.rank == 0 and self.step % self.log_freq == 0:
                print(f"[Train Step] {self.step}/{self.train_num_steps}: loss {loss.item():.4f} lr {self.lr_t.item():.3e}",
                      flush=True)
            if self.step != 0 and self.step % self.save_and_sample_every == 0:
                self.save(self.step // self.save_and_sample_every)
        if self.rank == 0:
            print("training complete", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg", required=True)
    ap.add_argument("--steps", type=int, default=None, help="override trainer.train_num_steps")
    ap.add_argument("--batch", type=int, default=None, help="override data.batch_size (per GPU)")
    ap.add_argument("--graph", action="store_true", help="replay the step as CUDA graphs (gradient_accumulate_every 1)")
    ap.add_argument("--log-freq", type=int, default=None)
    args = ap.parse_args()
    cfg = yaml.safe_load(open(args.cfg))
    ldm, dl = setup(cfg, args.batch)
    t = cfg["trainer"]
    trainer = CondTrainer(ldm, dl, gradient_accumulate_every=1 if args.graph else t["gradient_accumulate_every"],
                          train_lr=t["lr"], train_num_steps=args.steps or t["train_num_steps"],
                          save_and_sample_every=t["save_and_sample_every"], results_folder=t["results_folder"],
                          log_freq=args.log_freq or t["log_freq"], resume_milestone=t.get("resume_milestone", 0), cfg=cfg,
                          use_graph=args.graph)
    trainer.train()
    if dist.is_initialized():
        dist.destroy_process_group()


def setup(cfg, batch=None):
    """This process's GPU (LOCAL_RANK), the NCCL process group under torchrun, the model in training mode and this
    rank's batch stream (`batch` per GPU, default data.batch_size)."""
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    rank = dist.get_rank() if dist.is_initialized() else 0
    # autograd's AccumulateGrad nodes must not be bound to the default stream if the step is to be captured: run on a side one
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    torch.cuda.set_stream(side)
    # seed + rank for t, noise and dropout; the initial weights are rank 0's (CondTrainer broadcasts them)
    torch.manual_seed(1234 + rank)
    ldm = build_model(cfg, device)
    ldm.train()
    d = cfg["data"]
    return ldm, make_loader(d, batch or d["batch_size"], ldm.first_stage_model.down_ratio, rank, world)


if __name__ == "__main__":
    main()
