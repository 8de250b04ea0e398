"""Device-timed fused attention forward/backward at the phase-1 / phase-2 shapes."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bert_pytorch_b200.ops import api as K  # noqa: E402


def timeit(fn, iters=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


for B, S in ((96, 128), (16, 512)):
    h, H = 16, 1024
    qkv = (torch.randn(B, S, 3 * H, device="cuda") * 0.5).bfloat16()
    lens = torch.full((B,), S, device="cuda", dtype=torch.int32)
    ctx, lse = K.attention_fwd(qkv, lens, h, p_drop=0.1, seed=1, stream=1)
    d = torch.randn_like(ctx)
    tf = timeit(lambda: K.attention_fwd(qkv, lens, h, p_drop=0.1, seed=1, stream=1))
    tb = timeit(lambda: K.attention_bwd(qkv, lens, ctx, d, lse, h, p_drop=0.1, seed=1, stream=1))
    flops = 4.0 * B * h * S * S * 64
    row = {"B": B, "S": S, "fwd_ms": round(tf, 4), "bwd_ms": round(tb, 4),
           "fwd_tflops": round(flops / tf / 1e9, 1), "bwd_tflops": round(2.5 * flops / tb / 1e9, 1)}
    print(json.dumps(row), flush=True)
