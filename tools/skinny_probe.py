"""GPU probe: the skinny (decode) GEMM at the 1.3B shapes, timed inside a CUDA graph (no host launch overhead), cycling
through enough weight copies to defeat the 126 MB L2.  Env YMP_SKINNY_UNROLL / YMP_SKINNY_KSPLIT select variants."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "youku-mplug_b200"))
import torch  # noqa: E402
from ymp import lib, ops  # noqa: E402

dev, bf16, rows = torch.device("cuda"), torch.bfloat16, int(os.environ.get("ROWS", "5"))
# up to 8 rows: ymp_gemm_skinny (one beam search); 9-64 rows: ymp_gemm_skinny_batch (a batch of beam searches)
skinny = ops.gemm_skinny if rows <= ops.SKINNY_MAX_ROWS else ops.gemm_skinny_batch
for name, N, K, kw in (("qkv", 6144, 2048, {}), ("dense", 2048, 2048, dict(res=True)), ("fc1", 8192, 2048, dict(act=2)),
                       ("fc2", 2048, 8192, dict(res=True)), ("lm_head", 51200, 2048, dict(f32=True))):
    copies = max(4, int(600e6 // (N * K * 2)))
    ws = [(torch.randn(N, K, device=dev) * 0.02).to(bf16) for _ in range(copies)]
    x = torch.randn(rows, K, device=dev).to(bf16)
    b = torch.randn(N, device=dev).to(bf16)
    r = torch.randn(rows, N, device=dev) if kw.get("res") else None
    od = torch.float32 if (kw.get("res") or kw.get("f32")) else bf16
    out = torch.empty(rows, N, device=dev, dtype=od)
    for w in ws[:2]:
        skinny(x, w, bias=b, residual=r, act=kw.get("act", 0), out=out)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    lib.set_pdl(os.environ.get("PDL", "0") == "1")
    with torch.cuda.graph(g):
        for w in ws:
            skinny(x, w, bias=b, residual=r, act=kw.get("act", 0), out=out)
    lib.set_pdl(0)
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / (reps * copies) * 1e3
    print("SKINNY " + json.dumps(dict(shape=name, N=N, K=K, rows=rows, entry=skinny.__name__, us=round(us, 2), gbs=round(N * K * 2 / us / 1e3, 1),
                                      unroll=os.environ.get("YMP_SKINNY_UNROLL", "4"), pdl=os.environ.get("PDL", "0"), ksplit=os.environ.get("YMP_SKINNY_KSPLIT", "auto"))))
    del ws, g
