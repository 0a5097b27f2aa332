"""Where the MMA-issuing thread of the conv kernel spends its clocks (wait on TMA data / issue 4 MMAs / commit), per
k-iteration of the first tile of CTA 0.  Needs a library built with -DADM_GEMM_TIMING:

    make -C adm_b200/csrc -B NVCCFLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC --expt-relaxed-constexpr -DADM_GEMM_TIMING"
    python tools/gemm_thread_timing.py
    ADM_GEMM_DEBUG=1|2|3: skip the MMAs / the TMA loads / both (plain tc_gemm_kernel only)

Round-1 result (conv3x3 384->384 @16x16 x128): wait 204 + issue 291 + commit 55 = 550 clocks per k-iteration; with the
TMA loads skipped the same loop takes 425 (= 4 MMAs of 128x192x16 at ~106 clocks each, the tensor pipe's own rate), so
~23 % of the main loop is spent waiting for operand bytes (TMA ingest ~100 GB/s per SM for 40 KB per k-iteration).
"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from adm_b200 import ops
x = torch.randn(128, 16, 16, 384, device="cuda").bfloat16()
w = ops.pack_conv_weight(torch.randn(384, 384, 3, 3, device="cuda") / 60)
out = torch.empty(128, 16, 16, 384, device="cuda", dtype=torch.bfloat16)
for _ in range(2):
    ops.conv_fprop(x, w, out=out)
torch.cuda.synchronize()
