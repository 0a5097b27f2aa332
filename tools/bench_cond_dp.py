"""Data-parallel throughput of the conditional (DIV2K) training step through scripts/train_cond_ldm.py's CondTrainer:

    torchrun --nproc-per-node N tools/bench_cond_dp.py [--steps 30] [--warmup 8] [--no-graph] [--out FILE.json]

Same set-up as the training script (frozen AE encode + cond UNet 225 M, batch 8 per GPU by default, synthetic pairs
seeded with the rank, EMA on rank 0, one CUDA graph per step on one rank, two graphs around an eager all-reduce on
several).  `--warmup` eager and replayed steps (the graphs are captured after the third), then `--steps` timed steps
with a host clock that starts after a barrier and a device synchronise and stops after a device synchronise.  Prints
one JSON line on rank 0: per rank and in aggregate the step time and img/s (aggregate step time = the slowest rank),
each rank's device name and power limit read in the same run.  Checkpoints go to a temporary directory."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import torch
import torch.distributed as dist
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from scripts.train_cond_ldm import CondTrainer, setup  # noqa: E402


def device_info():
    """Name and power limit of this rank's GPU (nvidia-smi, read only)."""
    props = torch.cuda.get_device_properties(torch.cuda.current_device())
    info = {"name": props.name, "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                            "-i", f"GPU-{props.uuid}"], capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(q.stdout.strip().splitlines()[0])
    except Exception as e:  # reported, not guessed
        info["power_limit_w"] = f"unavailable ({type(e).__name__})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg", default=os.path.join(ROOT, "configs/super-resolution/div2k_cond_ddm_const_ldm.yaml"))
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--batch", type=int, default=8, help="per GPU (default: 8, the batch of bench.py --config div2k)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--out", default=None, help="also write the JSON result here (rank 0)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_cond_dp.py measures on the GPU; no CUDA device found")
    cfg = yaml.safe_load(open(args.cfg))
    ldm, dl = setup(cfg, args.batch)
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    batch = args.batch
    tmp = tempfile.mkdtemp(prefix="bench_cond_dp_")
    try:
        t = cfg["trainer"]
        tr = CondTrainer(ldm, dl, gradient_accumulate_every=1, train_lr=t["lr"], train_num_steps=10 ** 9,
                         save_and_sample_every=10 ** 9, results_folder=tmp, log_freq=10 ** 9, cfg=cfg,
                         use_graph=not args.no_graph)
        for _ in range(max(args.warmup, 5)):  # at least two replays of the captured graphs
            loss = tr.train_one_step()

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            loss = tr.train_one_step()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / args.steps
        mine = {"rank": rank, "step_ms": round(ms, 3), "img_per_s": round(batch * 1e3 / ms, 2),
                "loss": float(loss.item()), **device_info()}
        ranks = [None] * world
        if world > 1:
            dist.all_gather_object(ranks, mine)
        else:
            ranks = [mine]
        if rank == 0:
            slowest = max(r["step_ms"] for r in ranks)
            res = {"workload": "DIV2K 512x512 conditional latent training step through CondTrainer "
                               f"({os.path.relpath(args.cfg, ROOT)}), batch {batch} per GPU, AE encode + fwd + bwd + clip + AdamW + EMA",
                   "world": world, "graph": not args.no_graph, "steps": args.steps, "warmup": args.warmup,
                   "step_ms": slowest, "img_per_s": round(world * batch * 1e3 / slowest, 2), "ranks": ranks}
            line = json.dumps(res)
            print(line, flush=True)
            if args.out:
                with open(args.out, "w") as f:
                    f.write(line + "\n")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
