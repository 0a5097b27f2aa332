"""What bounds the GroupNorm apply pass?  Times adm_gn_apply with the activation and the dropout hash switched on and off,
the cluster kernels (statistics + apply, and the backward pair), and a plain torch copy of the same bytes as the roofline.
CUDA-graph of 10 launches each over rotating buffers larger than L2 (no host launch gaps)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from adm_b200 import ops


def graph_time(fn, nbuf, reps=10):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in range(nbuf):
            fn(i)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(reps):
            fn(i % nbuf)
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (5 * reps) * 1000


def main():
    dev = "cuda"
    n = 128
    for (hw, c) in [(32, 192), (16, 384), (16, 768), (8, 384), (4, 384)]:
        elems = n * hw * hw * c
        nbuf = max(3, int(400e6 // (elems * 4)) + 1)
        xs = [torch.randn(n, hw, hw, c, device=dev).bfloat16() for _ in range(nbuf)]
        dys = [torch.randn(n, hw, hw, c, device=dev).bfloat16() for _ in range(nbuf)]
        ys = [torch.empty_like(x) for x in xs]
        coef = torch.randn(n, c, 4, device=dev)
        gamma, beta = torch.ones(c, device=dev), torch.zeros(c, device=dev)
        params = 0.1 * torch.randn(n, 2 * c, device=dev)
        dg, db, dp = torch.zeros(c, device=dev), torch.zeros(c, device=dev), torch.zeros(n, 2 * c, device=dev)
        g = min(32, c // 4)
        mb = elems * 4 / 1e6
        row = [f"[{n},{hw},{hw},{c}] {mb:6.1f} MB r+w:"]
        t = graph_time(lambda i: ys[i].copy_(xs[i]), nbuf)
        row.append(f"torch copy {t:5.1f} us ({mb / t:.2f} TB/s)")
        for act, dp_ in ((False, 0.0), (True, 0.0), (True, 0.1)):
            t = graph_time(lambda i: ops.gn_apply(xs[i], None, coef, act=act, drop_p=dp_, seed=i), nbuf)
            row.append(f"apply act={int(act)} drop={dp_}: {t:5.1f} us ({mb / t:.2f})")
        t = graph_time(lambda i: ops.gn_forward(xs[i], None, gamma, beta, g, 1e-5, params=params, act=True, drop_p=0.0), nbuf)
        row.append(f"cluster fwd nodrop {t:5.1f}")
        t = graph_time(lambda i: ops.gn_forward(xs[i], None, gamma, beta, g, 1e-5, params=params, act=True, drop_p=0.1, seed=i), nbuf)
        row.append(f"cluster fwd drop {t:5.1f}")
        cf, _ = ops.gn_forward(xs[0], None, gamma, beta, g, 1e-5, params=params, act=True)
        for scratch in (False, True):
            t = graph_time(lambda i: ops.gn_bwd(dys[i], xs[i], None, cf, gamma, beta, g, params=params, act=True, drop_p=0.1,
                                                seed=i, dgamma=dg, dbeta=db, dparams=dp, dy_scratch=scratch), nbuf)
            row.append(f"cluster bwd drop scratch={int(scratch)} {t:5.1f}")
        print("  ".join(row), flush=True)


if __name__ == "__main__":
    main()
