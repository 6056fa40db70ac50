"""GPU probe: run each GEMM layout case in its own subprocess (a hung kernel cannot take the
whole call down), print error statistics, then time a few hot-path shapes against torch.matmul."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "youku-mplug_b200"))

CASES = [
    # (a_t, b_t, M, N, K, tile_n)
    (0, 0, 128, 256, 64, 256), (0, 0, 128, 128, 64, 128), (0, 0, 256, 512, 256, 256),
    (0, 1, 128, 256, 64, 256), (1, 0, 128, 256, 64, 256), (1, 1, 128, 256, 64, 256),
    (0, 1, 256, 512, 256, 128), (1, 1, 256, 512, 256, 128),
]


def one(case):
    import torch
    from ymp import ops
    a_t, b_t, M, N, K, tn = case
    torch.manual_seed(0)
    a = torch.randn((K, M) if a_t else (M, K), device="cuda").bfloat16()
    b = torch.randn((K, N) if b_t else (N, K), device="cuda").bfloat16()
    out = ops.gemm(a, b, a_t=bool(a_t), b_t=bool(b_t), tile_n=tn)
    torch.cuda.synchronize()
    A = a.float().t() if a_t else a.float()
    B = b.float() if b_t else b.float().t()
    ref = A @ B
    err = (out.float() - ref).abs()
    bad = (err > 0.05 * ref.abs().max()).nonzero()
    res = dict(case=case, max_err=err.max().item(), ref_max=ref.abs().max().item(),
               n_bad=int(bad.shape[0]), first_bad=bad[:8].tolist(),
               out00=out[:2, :4].float().tolist(), ref00=ref[:2, :4].tolist())
    print("PROBE " + json.dumps(res))


def bench():
    import torch
    from ymp import ops
    shapes = [(8192, 8192, 2048), (8192, 2048, 8192), (8192, 6144, 2048), (50176, 2304, 768),
              (50208, 3072, 768), (50208, 768, 3072), (8192, 51200, 2048)]
    for (M, N, K) in shapes:
        a = torch.randn(M, K, device="cuda").bfloat16()
        b = torch.randn(N, K, device="cuda").bfloat16()
        for name, fn in (("ymp", lambda: ops.gemm(a, b)), ("torch", lambda: a @ b.t())):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n = 10
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / n
            print("BENCH " + json.dumps(dict(impl=name, M=M, N=N, K=K, ms=ms, tflops=2 * M * N * K / ms / 1e9)))


def ncu_shapes():
    """A few hot-path GEMM launches (2 each) for `ncu --set full -k regex:gemm_bf16`."""
    import torch
    from ymp import ops
    dev = "cuda"
    a = torch.randn(50176, 768, device=dev).bfloat16()
    w = torch.randn(2304, 768, device=dev).bfloat16()
    for _ in range(2):
        ops.gemm(a, w)                                         # ViT qkv forward
    dy = torch.randn(50208, 768, device=dev).bfloat16()
    w2 = torch.randn(768, 3072, device=dev).bfloat16()
    pre = torch.randn(50208, 3072, device=dev).bfloat16()
    for _ in range(2):
        ops.gemm(dy, w2, b_t=True, act=1, aux_in=pre)         # fc2 dgrad with GELU'(erf) epilogue
    x = torch.randn(8192, 2048, device=dev).bfloat16()
    w3 = torch.randn(8192, 2048, device=dev).bfloat16()
    for _ in range(2):
        ops.gemm(x, w3)                                        # GPT h->4h
    g = torch.zeros(768, 768, device=dev)
    for _ in range(2):
        ops.gemm(dy[:50176], a, a_t=True, b_t=True, out=g, accumulate=True)   # wgrad, split-K
    torch.cuda.synchronize()


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "case":
        one(CASES[int(sys.argv[2])])
    elif len(sys.argv) > 1 and sys.argv[1] == "bench":
        bench()
    elif len(sys.argv) > 1 and sys.argv[1] == "ncu":
        ncu_shapes()
    else:
        for i in range(len(CASES)):
            try:
                r = subprocess.run([sys.executable, __file__, "case", str(i)], timeout=90,
                                   capture_output=True, text=True)
                print(r.stdout.strip()[-1500:] or ("NOOUT rc=%d " % r.returncode) + r.stderr[-800:])
            except subprocess.TimeoutExpired:
                print("PROBE " + json.dumps(dict(case=CASES[i], hang=True)))
        try:
            r = subprocess.run([sys.executable, __file__, "bench"], timeout=300, capture_output=True, text=True)
            print(r.stdout[-4000:], r.stderr[-1500:])
        except subprocess.TimeoutExpired:
            print("BENCH hang")
