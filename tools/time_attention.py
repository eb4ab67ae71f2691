"""Times tt_attn_causal_fwd / tt_attn_causal_bwd alone with CUDA events, H = 4. By default over sequence lengths on
both sides of the kernel switches at L = 256 (forward and backward) and L = 512 (backward), at about the c2 step's
token count (B*L ~ 51200); B and L in the environment time one shape instead. To compare two kernel variants, build
two libraries and run this once with each (TT_B200_LIB selects the library)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mrm_b200 import ops  # noqa: E402

SHAPES = [(256, 200), (200, 256), (160, 320), (100, 512), (80, 640)]   # (B, L)


def main():
    H = 4
    drop = float(os.environ.get("DROP", 0.1))
    shapes = [(int(os.environ.get("B", 256)), int(os.environ["L"]))] if "L" in os.environ else SHAPES
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(fn, iters=20):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        ts.sort()
        return ts[len(ts) // 2]

    for B, L in shapes:
        g = torch.Generator().manual_seed(1)
        qkv = (torch.randn(B * L, 3 * H * 64, generator=g) * 1.0).cuda().bfloat16()
        dctx = torch.randn(B * L, H * 64, generator=g).cuda().bfloat16()
        ctx = torch.empty((B * L, H * 64), device="cuda", dtype=torch.bfloat16)
        lse = torch.empty(B, H, L, device="cuda")
        dqkv = torch.empty((B * L, 3 * H * 64), device="cuda", dtype=torch.bfloat16)
        t = timed(lambda: ops.attn_fwd(qkv, ctx, lse, B, L, H, drop_p=drop, drop_seed=5, drop_site=1))
        print(f"attn_fwd  B={B} L={L}: {t:7.1f} us")
        t = timed(lambda: ops.attn_bwd(qkv, ctx, dctx, lse, dqkv, B, L, H, drop_p=drop, drop_seed=5, drop_site=1))
        print(f"attn_bwd  B={B} L={L}: {t:7.1f} us")


if __name__ == "__main__":
    main()
