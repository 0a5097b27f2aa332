"""Discriminating micro-benchmarks for the conv / GEMM engine: plain K-major GEMM vs implicit-GEMM conv of the same
FLOPs, L2-resident vs rotating (cold) operands."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from adm_b200 import ops
from tools.bench_convs_lib import timeit

N = 128
for cin, cout, res in [(384, 384, 16), (192, 192, 32), (768, 384, 16), (384, 384, 8), (256, 256, 16), (128, 128, 32)]:
    flops = 2.0 * N * res * res * cin * cout * 9
    w = ops.pack_conv_weight(torch.randn(cout, cin, 3, 3, device="cuda") / 60)
    nbuf = max(2, int(400e6 // (N * res * res * (cin + cout) * 2)) + 1)
    xs = [torch.randn(N, res, res, cin, device="cuda").bfloat16() for _ in range(nbuf)]
    outs = [torch.empty(N, res, res, cout, device="cuda", dtype=torch.bfloat16) for _ in range(nbuf)]
    t_hot = timeit(lambda: ops.conv_fprop(xs[0], w, out=outs[0]))
    it = [0]
    def cold():
        i = it[0] % nbuf
        it[0] += 1
        ops.conv_fprop(xs[i], w, out=outs[i])
    t_cold = timeit(cold, iters=nbuf)
    # the same FLOPs as a plain GEMM: A [M, 9*cin] K-major, B [cout, 9*cin] K-major
    M = N * res * res
    a = torch.randn(M, 9 * cin, device="cuda").bfloat16()
    b = torch.randn(cout, 9 * cin, device="cuda").bfloat16()
    c = torch.empty(M, cout, device="cuda", dtype=torch.bfloat16)
    t_gemm = timeit(lambda: ops.gemm_nt(a, b, out=c))
    t_cublas = timeit(lambda: torch.matmul(a, b.t(), out=c))
    print(f"[{cin:4d}->{cout:4d} @{res:2d}] conv hot {flops/t_hot/1e9:7.1f} TF/s  conv cold {flops/t_cold/1e9:7.1f} TF/s  "
          f"plain gemm {flops/t_gemm/1e9:7.1f} TF/s  cuBLAS {flops/t_cublas/1e9:7.1f} TF/s", flush=True)
    del xs, outs, a, b, c
