"""GPU parity: tcgen05 GEMM (ymp_gemm) vs an fp32 torch matmul of the same bf16 inputs."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _dact(x, act):
    if act == 1:
        return 0.5 * (1 + torch.erf(x / 2 ** 0.5)) + x * torch.exp(-0.5 * x * x) / (2 * torch.pi) ** 0.5
    if act == 2:
        u = 0.79788456 * x * (1 + 0.044715 * x * x)
        t = torch.tanh(u)
        return 0.5 * (1 + t) + 0.5 * x * (1 - t * t) * 0.79788456 * (1 + 3 * 0.044715 * x * x)
    return torch.ones_like(x)


def _ref(a, b, a_t, b_t, bias=None, residual=None, act=0, aux_in=None, alpha=1.0):
    """Returns (D, aux_out) where aux_out = act'(pre-activation) when act != 0, else the pre-activation."""
    A = a.float().t() if a_t else a.float()
    B = b.float() if b_t else b.float().t()
    v = alpha * (A @ B)
    if bias is not None:
        v = v + bias.float()
    aux = _dact(v, act) if act else v
    if aux_in is not None:
        v = v * aux_in.float()
    elif act == 1:
        v = torch.nn.functional.gelu(v)
    elif act == 2:
        v = torch.nn.functional.gelu(v, approximate="tanh")
    if residual is not None:
        v = v + residual.float()
    return v, aux


def _close(out, ref, tol=2e-2):
    err = (out.float() - ref).abs().max().item()
    scale = ref.abs().max().item() + 1e-6
    assert err / scale < tol, f"max err {err} vs scale {scale}"


@pytest.mark.parametrize("a_t,b_t", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("M,N,K,tile_n", [(256, 256, 128, 256), (384, 512, 192, 128), (200, 328, 72, 0),
                                          (1024, 768, 768, 256), (512, 512, 256, 512), (1024, 768, 768, 512),
                                          (304, 520, 136, 512), (2304, 768, 512, 512)])
def test_gemm_layouts(cuda, a_t, b_t, M, N, K, tile_n):
    from ymp import ops
    torch.manual_seed(0)
    a = torch.randn((K, M) if a_t else (M, K), device=cuda).bfloat16()
    b = torch.randn((K, N) if b_t else (N, K), device=cuda).bfloat16()
    out = ops.gemm(a, b, a_t=a_t, b_t=b_t, tile_n=tile_n)
    ref, _ = _ref(a, b, a_t, b_t)
    _close(out, ref, 1e-2)


@pytest.mark.parametrize("tile_n", [0, 512])
@pytest.mark.parametrize("act", [0, 1, 2])
def test_gemm_epilogue_fwd(cuda, act, tile_n):
    from ymp import ops
    torch.manual_seed(1)
    M, N, K = 512, 768, 256
    a = torch.randn(M, K, device=cuda).bfloat16()
    b = (torch.randn(N, K, device=cuda) * 0.1).bfloat16()
    bias = torch.randn(N, device=cuda).bfloat16()
    res = torch.randn(M, N, device=cuda).bfloat16()
    aux = torch.empty(M, N, device=cuda, dtype=torch.bfloat16)
    out = ops.gemm(a, b, bias=bias, residual=res, act=act, aux_out=aux, tile_n=tile_n)
    ref, pre = _ref(a, b, False, False, bias=bias, residual=res, act=act)
    _close(out, ref)
    _close(aux, pre)


@pytest.mark.parametrize("tile_n", [0, 512])
def test_gemm_epilogue_multiplier(cuda, tile_n):
    """Backward of an activation: D = (dY @ W) * aux_in, aux_in = act'(pre) saved by the forward GEMM."""
    from ymp import ops
    torch.manual_seed(2)
    M, N, K = 256, 512, 320
    a = torch.randn(M, K, device=cuda).bfloat16()
    b = (torch.randn(K, N, device=cuda) * 0.1).bfloat16()
    mul = torch.randn(M, N, device=cuda).bfloat16()
    out = ops.gemm(a, b, b_t=True, act=1, aux_in=mul, tile_n=tile_n)
    ref, _ = _ref(a, b, False, True, aux_in=mul)
    _close(out, ref)


def test_gemm_f32_out_and_splitk(cuda):
    from ymp import ops
    torch.manual_seed(3)
    M, N, K = 768, 768, 4096  # wgrad-like: both operands MN-major, long K
    a = torch.randn(K, M, device=cuda).bfloat16()
    b = torch.randn(K, N, device=cuda).bfloat16()
    ref, _ = _ref(a, b, True, True)
    out = ops.gemm(a, b, a_t=True, b_t=True, out_dtype=torch.float32)
    _close(out, ref, 1e-3)
    acc = torch.ones(M, N, device=cuda, dtype=torch.float32)
    ops.gemm(a, b, a_t=True, b_t=True, out=acc, accumulate=True, split_k=8)
    _close(acc, ref + 1.0, 1e-3)
    acc2 = torch.zeros(M, N, device=cuda, dtype=torch.float32)
    ops.gemm(a, b, a_t=True, b_t=True, out=acc2, accumulate=True, split_k=0)
    _close(acc2, ref, 1e-3)
    acc3 = torch.zeros(M, N, device=cuda, dtype=torch.float32)
    ops.gemm(a, b, a_t=True, b_t=True, out=acc3, accumulate=True, split_k=4, tile_n=512)   # CTA-pair tiles
    _close(acc3, ref, 1e-3)


def test_gemm_large_persistent(cuda):
    """More tiles than SMs: exercises the persistent loop, the smem ring wrap and both TMEM stages."""
    from ymp import ops
    torch.manual_seed(4)
    M, N, K = 4096 + 64, 2048, 1024
    a = torch.randn(M, K, device=cuda).bfloat16()
    b = (torch.randn(N, K, device=cuda) * 0.05).bfloat16()
    out = ops.gemm(a, b)
    ref, _ = _ref(a, b, False, False)
    _close(out, ref, 1e-2)
    out_p = ops.gemm(a, b, tile_n=512)   # CTA pairs: persistent loop + 6-stage ring + both TMEM stages
    _close(out_p, ref, 1e-2)
    big_m = torch.randn(20000, K, device=cuda).bfloat16()   # > 74 pairs: several tiles per pair
    _close(ops.gemm(big_m, b, tile_n=512), big_m.float() @ b.float().t(), 1e-2)
    # strided views (ld > width) as produced by slicing packed QKV buffers
    big = torch.randn(M, 3 * K, device=cuda).bfloat16()
    out2 = ops.gemm(big[:, K:2 * K], b)
    ref2, _ = _ref(big[:, K:2 * K], b, False, False)
    _close(out2, ref2, 1e-2)


@pytest.mark.parametrize("M", [1000, 2560 + 37])
def test_gemm_pair_tile_tma_epilogue_variants(cuda, M):
    """CTA-pair kernel, epilogue staged through swizzled smem and written with bulk tensor stores / reduce-adds:
    ragged M (rows clipped by the tensor map), fp32 residual stream in and out, bf16 + act' pairs, row-strided
    outputs, split-K accumulation into a non-zero buffer, several tiles per CTA pair (staging-buffer reuse)."""
    from ymp import ops
    torch.manual_seed(5)
    N, K = 768, 320
    a = torch.randn(M, K, device=cuda).bfloat16()
    b = (torch.randn(N, K, device=cuda) * 0.1).bfloat16()
    bias = torch.randn(N, device=cuda).bfloat16()
    # fp32 stream: out = x + (a b^T + bias)
    x = torch.randn(M, N, device=cuda)
    out = ops.gemm(a, b, bias=bias, residual=x, out_dtype=torch.float32, tile_n=512)
    ref, _ = _ref(a, b, False, False, bias=bias)
    _close(out, ref + x, 1e-3 * 8)
    # in place on the stream buffer itself (engine: residual and D may alias)
    x2 = x.clone()
    ops.gemm(a, b, bias=bias, residual=x2, out=x2, tile_n=512)
    _close(x2, ref + x, 1e-3 * 8)
    # bf16 + act' into row-strided views of wider buffers
    wide = torch.zeros(M, 2 * N, device=cuda, dtype=torch.bfloat16)
    wide_aux = torch.zeros(M, 2 * N, device=cuda, dtype=torch.bfloat16)
    for act in (1, 2):
        ops.gemm(a, b, bias=bias, act=act, aux_out=wide_aux[:, N:], out=wide[:, N:], tile_n=512)
        r2, pre = _ref(a, b, False, False, bias=bias, act=act)
        _close(wide[:, N:], r2)
        _close(wide_aux[:, N:], pre)
        assert float(wide[:, :N].abs().max()) == 0.0 and float(wide_aux[:, :N].abs().max()) == 0.0
    # activation backward: multiplier read per element
    mul = torch.randn(M, K, device=cuda).bfloat16()
    g = ops.gemm(a.new_empty(M, N).normal_().bfloat16(), b, b_t=True, aux_in=mul, act=1, tile_n=512)
    assert g.shape == (M, K)
    # split-K wgrad: fp32 accumulate into a running buffer (slices added in order by the reduction kernel)
    dy = torch.randn(M, N, device=cuda).bfloat16()
    acc = torch.full((N, K), 0.5, device=cuda)
    ops.gemm(dy, a, a_t=True, b_t=True, out=acc, accumulate=True, split_k=3, tile_n=512)
    _close(acc, dy.float().t() @ a.float() + 0.5, 2e-3)
    # many tiles per pair
    big = torch.randn(40000, K, device=cuda).bfloat16()
    _close(ops.gemm(big, b, bias=bias, tile_n=512), big.float() @ b.float().t() + bias.float(), 1e-2)


@pytest.mark.parametrize("M", [1, 5, 8])
@pytest.mark.parametrize("N,K", [(2048, 2048), (6144, 2048), (8192, 2048), (2048, 8192), (51200, 2048), (50, 64), (130, 2560)])
def test_gemm_skinny_decode_shapes(cuda, M, N, K):
    """ymp_gemm_skinny (single-token decoding linears, csrc/gemv.cu) vs fp32 torch on the same bf16 inputs: every
    K-split the host heuristic picks at the 1.3B / 2.7B shapes, ragged N, all epilogues."""
    from ymp import ops
    torch.manual_seed(M + N)
    x = torch.randn(M, K, device=cuda).bfloat16()
    w = (torch.randn(N, K, device=cuda) * K ** -0.5).bfloat16()
    bias = torch.randn(N, device=cuda).bfloat16()
    res32 = torch.randn(M, N, device=cuda)
    resb = torch.randn(M, N, device=cuda).bfloat16()
    pre = x.float() @ w.float().t()
    _close(ops.gemm_skinny(x, w), pre)
    _close(ops.gemm_skinny(x, w, out_dtype=torch.float32), pre, tol=1e-4)
    _close(ops.gemm_skinny(x, w, bias=bias, act=2), torch.nn.functional.gelu(pre + bias.float(), approximate="tanh"))
    _close(ops.gemm_skinny(x, w, bias=bias, act=1), torch.nn.functional.gelu(pre + bias.float()))
    _close(ops.gemm_skinny(x, w, bias=bias, residual=res32, out_dtype=torch.float32), pre + bias.float() + res32, tol=1e-4)
    _close(ops.gemm_skinny(x, w, bias=bias, residual=resb), pre + bias.float() + resb.float())
    # against the tensor-core GEMM on the same inputs (fp32 accumulation on both sides, different summation order)
    if N % 8 == 0:
        _close(ops.gemm_skinny(x, w, bias=bias, out_dtype=torch.float32), ops.gemm(x, w, bias=bias, out_dtype=torch.float32).float(), tol=1e-4)
    # strided rows: x and y as column slices of wider buffers
    xw = torch.randn(M, K + 64, device=cuda).bfloat16()
    yw = torch.zeros(M, N + 8, device=cuda, dtype=torch.bfloat16)
    ops.gemm_skinny(xw[:, 32:32 + K], w, out=yw[:, :N])
    _close(yw[:, :N], (xw[:, 32:32 + K].float() @ w.float().t()))
    assert float(yw[:, N:].abs().max()) == 0.0


def test_gemm_skinny_rejects_wide_inputs(cuda):
    from ymp import lib, ops
    x = torch.randn(8, 64, device=cuda).bfloat16()
    w = torch.randn(16, 64, device=cuda).bfloat16()
    a = lib.GemmSkinnyArgs()
    a.x, a.w, a.y = x.data_ptr(), w.data_ptr(), torch.empty(9, 16, device=cuda, dtype=torch.bfloat16).data_ptr()
    a.M, a.N, a.K, a.ldx, a.ldw, a.ldy = 9, 16, 64, 64, 64, 16
    import ctypes
    assert lib._gemm_skinny(ctypes.byref(a), lib.cur_stream()) == -1
    with pytest.raises(AssertionError):
        ops.gemm_skinny(torch.randn(9, 64, device=cuda).bfloat16(), w)


@pytest.mark.parametrize("M,N,K", [(5, 2048, 2048), (8, 2048, 8192), (1, 2560, 2560), (3, 72, 64)])
def test_gemm_skinny_fused_layernorm_and_cache_row(cuda, M, N, K):
    """The two fused outputs of the decoding step: LN(y) written by the last CTA (ymp_layernorm_fwd's formula on the same
    y; only the fp32 summation order differs, so results agree to one bf16 ulp; the ticket counter resets itself) and the
    second bf16 copy at a device-side row offset."""
    from ymp import ops
    torch.manual_seed(N + K)
    x = torch.randn(M, K, device=cuda).bfloat16()
    w = (torch.randn(N, K, device=cuda) * K ** -0.5).bfloat16()
    bias = torch.randn(N, device=cuda).bfloat16()
    res = torch.randn(M, N, device=cuda)
    gamma, beta = (1 + 0.1 * torch.randn(N, device=cuda)).bfloat16(), (0.1 * torch.randn(N, device=cuda)).bfloat16()
    ticket = torch.zeros(1, device=cuda, dtype=torch.int32)
    for _ in range(3):
        y, ln_y = ops.gemm_skinny(x, w, bias=bias, residual=res, out_dtype=torch.float32, ln=(gamma, beta, 1e-5, ticket))
        assert int(ticket) == 0
        ref, _, _ = ops.layernorm_fwd(y, gamma, beta, 1e-5, stats=False)
        assert (ln_y.float() - ref.float()).abs().max().item() <= 2 ** -7 * max(1.0, ref.float().abs().max().item())
        assert (ln_y != ref).float().mean().item() < 0.02
        _close(y, x.float() @ w.float().t() + bias.float() + res, tol=1e-4)
    ML = 7
    cache = torch.zeros(M * ML, N, device=cuda, dtype=torch.bfloat16)
    off = torch.tensor([4], device=cuda, dtype=torch.int64)
    st = ops.gemm_skinny(x, w, bias=bias, out2=cache, out2_row_stride=ML, out2_off=off)
    assert torch.equal(cache.view(M, ML, N)[:, 4], st)
    cache.view(M, ML, N)[:, 4] = 0
    assert float(cache.abs().max()) == 0.0
