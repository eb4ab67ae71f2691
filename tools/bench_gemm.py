#!/usr/bin/env python
"""Event-timed micro-benchmark of tt_gemm_bf16 on the training step's shapes."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from mrm_b200 import ops  # noqa: E402

T, D, FF = 51200, 256, 1024
dev = "cuda"
bf = dict(device=dev, dtype=torch.bfloat16)
x = torch.randn(T, FF, **bf)
w = torch.randn(FF, FF, **bf) * 0.05
bias = torch.randn(FF, device=dev)
res = torch.randn(T, D, device=dev)
gate = torch.randn(T, FF, **bf)
o32 = torch.empty(T, D, device=dev)
o16 = torch.empty(T, FF, **bf)
g32 = torch.zeros(FF, FF, device=dev)


def t(fn, iters=10):
    """CUDA-graph replay of `iters` back-to-back launches: no host launch overhead in the number."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


cases = [
    ("qkv   fwd bf16 bias          ", T, 768, 256, lambda: ops.gemm(x[:, :256], w[:768, :256], bias=bias, out_bf16=o16[:, :768])),
    ("qkv   fwd bf16 plain         ", T, 768, 256, lambda: ops.gemm(x[:, :256], w[:768, :256], out_bf16=o16[:, :768])),
    ("oproj fwd f32 bias+res       ", T, 256, 256, lambda: ops.gemm(x[:, :256], w[:256, :256], bias=bias, residual=res, out_f32=o32)),
    ("oproj fwd f32 bias+res+drop  ", T, 256, 256, lambda: ops.gemm(x[:, :256], w[:256, :256], bias=bias, residual=res, drop_p=0.1, drop_site=3, out_f32=o32)),
    ("oproj fwd f32 plain          ", T, 256, 256, lambda: ops.gemm(x[:, :256], w[:256, :256], out_f32=o32)),
    ("ffn1  fwd bf16 plain         ", T, 1024, 256, lambda: ops.gemm(x[:, :256], w[:, :256], out_bf16=o16)),
    ("tiny  256x256x256 f32 bias   ", 256, 256, 256, lambda: ops.gemm(x[:256, :256], w[:256, :256], bias=bias, out_f32=o32[:256])),
    ("tiny  256x1024x256 bf16      ", 256, 1024, 256, lambda: ops.gemm(x[:256, :256], w[:, :256], bias=bias, relu=True, out_bf16=o16[:256])),
    ("tiny  256x256x1024 f32       ", 256, 256, 1024, lambda: ops.gemm(x[:256], w[:256], bias=bias, out_f32=o32[:256])),
    ("ffn1  fwd bf16 bias+relu     ", T, 1024, 256, lambda: ops.gemm(x[:, :256], w[:, :256], bias=bias, relu=True, out_bf16=o16)),
    ("ffn1  fwd bf16 +drop         ", T, 1024, 256, lambda: ops.gemm(x[:, :256], w[:, :256], bias=bias, relu=True, drop_p=0.1, drop_site=2, out_bf16=o16)),
    ("ffn2  fwd f32 bias+res       ", T, 256, 1024, lambda: ops.gemm(x, w[:256], bias=bias, residual=res, out_f32=o32)),
    ("dpre  dgrad bf16 gate        ", T, 1024, 256, lambda: ops.gemm(x[:, :256], w[:256], b_mn=True, gate=gate, gate_scale=1.1, out_bf16=o16)),
    ("dh    dgrad f32 K=1024       ", T, 256, 1024, lambda: ops.gemm(x, w[:, :256], b_mn=True, out_f32=o32)),
    ("dctx  dgrad bf16 K=256       ", T, 256, 256, lambda: ops.gemm(x[:, :256], w[:256, :256], b_mn=True, out_bf16=o16[:, :256])),
    ("dW2   wgrad 256x1024         ", 256, 1024, T, lambda: ops.gemm(x[:, :256], x, a_mn=True, b_mn=True, out_f32=g32[:256], accumulate=True)),
    ("dWo   wgrad 256x256          ", 256, 256, T, lambda: ops.gemm(x[:, :256], x[:, :256], a_mn=True, b_mn=True, out_f32=g32[:256, :256], accumulate=True)),
]
for name, M, N, K, fn in cases:
    us = t(fn)
    print(f"{name} M={M:6d} N={N:5d} K={K:6d}  {us:8.1f} us  {2.0 * M * N * K / us / 1e6:8.1f} TFLOP/s")
