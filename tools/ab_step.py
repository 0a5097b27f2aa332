"""A/B timing of the captured CIFAR training step under different environments, one subprocess per variant, interleaved
over several rounds so box drift hits every variant equally.  Two builds of the library are compared through
ADM_B200_LIB (the Python package is this tree's in both; "" is the in-tree build):

    python tools/ab_step.py "ADM_B200_LIB=/path/to/other/adm_b200/libadm_b200.so" "" [--rounds 2] [--steps 30] [--sample]
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def child(steps, sample):
    import torch
    import bench
    from adm_b200.train import TrainStep
    dev = torch.device("cuda", 0)
    dpm = bench.build_model(dev)
    dpm.train()
    step = TrainStep(dpm)
    B = int(os.environ.get("ADM_AB_BATCH", "128"))
    x = 2 * torch.rand(B, 3, 32, 32, device=dev) - 1
    step.capture(x)
    step.prefetch(x)
    for _ in range(5):
        step.replay()
        step.prefetch(x)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step.replay()
        step.prefetch(x)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    out = f"train {ms:.3f} ms/step ({B / ms * 1000:.0f} img/s at batch {B}) loss {float(loss):.2f}"
    if sample:
        dpm.eval()
        dpm.sampling_timesteps = 10
        with torch.no_grad():
            dpm.sample(batch_size=128)
            torch.cuda.synchronize()
            e0.record()
            dpm.sample(batch_size=128)
            e1.record()
            torch.cuda.synchronize()
        out += f" | sample10 {128 / (e0.elapsed_time(e1) / 1000):.1f} img/s"
    print(out, flush=True)


if __name__ == "__main__":
    if sys.argv[1] == "--child":
        child(int(sys.argv[2]), sys.argv[3] == "1")
        sys.exit(0)
    args = sys.argv[1:]
    rounds, steps, sample = 2, 30, False
    variants = []
    i = 0
    while i < len(args):
        if args[i] == "--rounds":
            rounds = int(args[i + 1]); i += 2
        elif args[i] == "--steps":
            steps = int(args[i + 1]); i += 2
        elif args[i] == "--sample":
            sample = True; i += 1
        else:
            variants.append(args[i]); i += 1
    for r in range(rounds):
        for v in variants:
            env = dict(os.environ)
            for kv in v.split():
                if "=" in kv:
                    k, val = kv.split("=", 1)
                    env[k] = val
            res = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", str(steps), "1" if sample else "0"],
                                 env=env, capture_output=True, text=True, cwd=ROOT)
            last = res.stdout.strip().splitlines()[-1] if res.stdout.strip() else "FAILED: " + res.stderr[-400:]
            print(f"[round {r}] {v or '(default)':40s} {last}", flush=True)
