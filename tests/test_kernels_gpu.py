"""GPU parity tests of the individual CUDA kernels (through the C ABI via tinyrec.ops)
against plain PyTorch fp32 restatements of the same op.  Tolerances are the bf16 bar of
BASELINE.json's north_star (1e-2 relative) unless stated."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

BF = torch.bfloat16


def _ops():
    import tinyrec.ops as ops
    return ops


def _rel_err(got, ref):
    got, ref = got.float(), ref.float()
    return float((got - ref).norm() / (ref.norm() + 1e-12)), float((got - ref).abs().max())


def _randn(*shape, scale=1.0, dtype=BF, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*shape, generator=g, device="cuda") * scale).to(dtype)


# ------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (300, 256, 128), (1000, 768, 768), (257, 2304, 768),
                                   (130, 200, 768), (4096, 3072, 768), (513, 768, 3072), (64, 128, 200)])
def test_gemm_nt_plain(M, N, K):
    ops = _ops()
    a, b = _randn(M, K, seed=1), _randn(N, K, seed=2)
    out = torch.empty(M, N, device="cuda", dtype=BF)
    ops.gemm(a, b, out)
    ref = a.float() @ b.float().t()
    rel, mx = _rel_err(out, ref)
    assert rel < 5e-3, (rel, mx)


def test_gemm_fp32_out_bias_residual():
    ops = _ops()
    M, N, K = 777, 768, 768
    a, b = _randn(M, K, seed=3), _randn(N, K, scale=0.05, seed=4)
    bias = _randn(N, dtype=torch.float32, seed=5)
    res = _randn(M, N, seed=6)
    out = torch.empty(M, N, device="cuda", dtype=torch.float32)
    ops.gemm(a, b, out, bias=bias, residual=res)
    ref = a.float() @ b.float().t() + bias + res.float()
    rel, mx = _rel_err(out, ref)
    assert rel < 1e-4, (rel, mx)       # fp32 accumulate + fp32 store: only summation order differs


def test_gemm_gelu_with_preact_and_tanh():
    ops = _ops()
    M, N, K = 500, 3072, 768
    a, b = _randn(M, K, seed=7), _randn(N, K, scale=0.03, seed=8)
    bias = _randn(N, dtype=torch.float32, scale=0.1, seed=9)
    out = torch.empty(M, N, device="cuda", dtype=BF)
    pre = torch.empty(M, N, device="cuda", dtype=BF)
    ops.gemm(a, b, out, bias=bias, act=ops.ACT_GELU, aux=pre)
    z = a.float() @ b.float().t() + bias
    assert _rel_err(pre, z)[0] < 5e-3
    assert _rel_err(out, torch.nn.functional.gelu(z))[0] < 5e-3
    N2 = 200
    b2 = _randn(N2, K, scale=0.03, seed=10)
    out2 = torch.empty(M, N2, device="cuda", dtype=BF)
    ops.gemm(a, b2, out2, bias=bias[:N2].contiguous(), act=ops.ACT_TANH)
    assert _rel_err(out2, torch.tanh(a.float() @ b2.float().t() + bias[:N2]))[0] < 5e-3


def test_gemm_gelu_epilogue_extreme_preactivations():
    """The epilogue GELU is a fitted sigmoid form (common.cuh): check it against erf-GELU over the
    whole range including |z| far outside the fitted interval."""
    ops = _ops()
    M, N, K = 256, 256, 64
    z = torch.linspace(-40, 40, M * N, device="cuda").reshape(M, N)
    a = torch.zeros(M, K, device="cuda", dtype=BF)
    b = torch.zeros(N, K, device="cuda", dtype=BF)
    a[:, 0] = 1.0
    out = torch.empty(M, N, device="cuda", dtype=BF)
    # pre-activation = 0 + bias is per-column only, so sweep through K=64 one-hot rows instead
    zz = torch.linspace(-40, 40, M, device="cuda")
    a[:, 0] = zz.to(BF)
    b[:, 0] = 1.0
    ops.gemm(a, b, out, act=ops.ACT_GELU)
    ref = torch.nn.functional.gelu(a[:, 0].float())[:, None].expand(M, N)
    assert float((out.float() - ref).abs().max()) <= 0.13              # bf16 rounding of values up to 40
    assert _rel_err(out, ref)[0] < 4e-3
    assert float(out[zz < -9].float().abs().max()) < 1e-6
    dz = torch.empty(M, N, device="cuda", dtype=BF)
    ones = torch.zeros(M, K, device="cuda", dtype=BF)
    ones[:, 0] = 1.0
    w = torch.zeros(K, N, device="cuda", dtype=BF)
    w[0] = 1.0
    aux = a[:, :1].expand(M, N).contiguous()
    ops.gemm(ones, w, dz, b_t=True, act=ops.ACT_DGELU, aux=aux)
    zf = aux.float().requires_grad_(True)
    torch.nn.functional.gelu(zf).sum().backward()
    assert float((dz.float() - zf.grad).abs().max()) < 6e-3


def test_gemm_dgelu_epilogue():
    ops = _ops()
    M, N, K = 384, 3072, 768
    dy, w = _randn(M, K, seed=11), _randn(K, N, scale=0.03, seed=12)      # dgrad through W [out=K, in=N]
    z = _randn(M, N, seed=13)
    out = torch.empty(M, N, device="cuda", dtype=BF)
    cs = torch.zeros(N, device="cuda")
    ops.gemm(dy, w, out, b_t=True, act=ops.ACT_DGELU, aux=z, colsum=cs)       # M = 384: single-CTA kernels
    assert _rel_err(cs, out.float().sum(0))[0] < 1e-5
    zf = z.float().requires_grad_(True)
    torch.nn.functional.gelu(zf).backward(dy.float() @ w.float())
    assert _rel_err(out, zf.grad)[0] < 5e-3


@pytest.mark.parametrize("M,N,K", [(256, 768, 768), (1000, 768, 3072), (300, 3072, 768), (100, 768, 200)])
def test_gemm_b_mn_major(M, N, K):
    """dgrad: dX[M, N] = dY[M, K] @ W[K, N] with W stored [K, N] row-major."""
    ops = _ops()
    a, w = _randn(M, K, seed=14), _randn(K, N, scale=0.05, seed=15)
    out = torch.empty(M, N, device="cuda", dtype=BF)
    ops.gemm(a, w, out, b_t=True)
    rel, mx = _rel_err(out, a.float() @ w.float())
    assert rel < 5e-3, (rel, mx)


@pytest.mark.parametrize("M,N,K,split", [(768, 768, 512, 1), (768, 3072, 1000, 4), (3072, 768, 5280, 8),
                                         (200, 768, 960, 3), (256, 256, 1760, 2), (640, 768, 2000, 5)])
def test_gemm_wgrad_mn_major_splitk(M, N, K, split):
    """wgrad: dW[M, N] = dY[K, M]^T @ X[K, N], both operands MN-major, split-K fp32 atomics."""
    ops = _ops()
    dy, x = _randn(K, M, seed=16), _randn(K, N, seed=17)
    out = torch.zeros(M, N, device="cuda", dtype=torch.float32)
    ops.gemm(dy, x, out, a_t=True, b_t=True, split_k=split, accumulate=True)
    ref = dy.float().t() @ x.float()
    rel, mx = _rel_err(out, ref)
    assert rel < 1e-4, (rel, mx)
    ops.gemm(dy, x, out, a_t=True, b_t=True, split_k=split, accumulate=True)     # accumulates
    assert _rel_err(out, 2 * ref)[0] < 1e-4


# CTA-pair (tcgen05 cta_group::2) kernels take over for M >= 4096, N > 128, bf16 output (gemm_tcgen05.cu).
@pytest.mark.parametrize("M,N,K,b_t", [(4096, 768, 768, False), (4200, 2304, 768, False), (4232, 768, 3072, False),
                                       (4096, 256, 64, False), (5000, 3072, 768, True), (4200, 768, 2304, True),
                                       (4100, 200, 768, False)])
def test_gemm_cta_pair_plain(M, N, K, b_t):
    """Odd numbers of 128-row tiles (the second CTA of the last pair is all padding), ragged M and N,
    K-major and MN-major B."""
    ops = _ops()
    a = _randn(M, K, seed=21)
    blog = _randn(N, K, scale=0.05, seed=22)
    b = blog.t().contiguous() if b_t else blog
    out = torch.full((M, N), float("nan"), device="cuda", dtype=BF)
    ops.gemm(a, b, out, b_t=b_t)
    ref = a.float() @ blog.float().t()
    rel, mx = _rel_err(out, ref)
    assert rel < 5e-3, (rel, mx)
    # every row block matches on its own (a swapped / dropped half tile would hide in a global norm)
    blk = (out.float() - ref).reshape(-1)[: (M // 8) * 8 * N].reshape(M // 8, -1).norm(dim=1)
    refn = ref.reshape(-1)[: (M // 8) * 8 * N].reshape(M // 8, -1).norm(dim=1)
    assert float((blk / (refn + 1e-6)).max()) < 2e-2


def test_gemm_cta_pair_epilogues():
    ops = _ops()
    M, N, K = 4200, 3072, 768
    a, b = _randn(M, K, seed=23), _randn(N, K, scale=0.03, seed=24)
    bias = _randn(N, dtype=torch.float32, scale=0.1, seed=25)
    out = torch.empty(M, N, device="cuda", dtype=BF)
    pre = torch.empty(M, N, device="cuda", dtype=BF)
    ops.gemm(a, b, out, bias=bias, act=ops.ACT_GELU, aux=pre)
    z = a.float() @ b.float().t() + bias
    assert _rel_err(pre, z)[0] < 5e-3
    assert _rel_err(out, torch.nn.functional.gelu(z))[0] < 5e-3
    ops.gemm(a, b, out, bias=bias, act=ops.ACT_GELU)                       # no pre-activation output
    assert _rel_err(out, torch.nn.functional.gelu(z))[0] < 5e-3
    # bias + residual (BertSelfOutput / BertOutput dense)
    N2, K2 = 768, 3072
    a2, b2 = _randn(M, K2, seed=26), _randn(N2, K2, scale=0.03, seed=27)
    res = _randn(M, N2, seed=28)
    out2 = torch.empty(M, N2, device="cuda", dtype=BF)
    ops.gemm(a2, b2, out2, bias=bias[:N2].contiguous(), residual=res)
    assert _rel_err(out2, a2.float() @ b2.float().t() + bias[:N2] + res.float())[0] < 5e-3
    # dgrad + dGELU (MN-major B, pre-activation box prefetched by TMA)
    dy, w = _randn(M, K, seed=29), _randn(K, N, scale=0.03, seed=30)
    zz = _randn(M, N, seed=31)
    dz = torch.empty(M, N, device="cuda", dtype=BF)
    cs = torch.zeros(N, device="cuda")
    ops.gemm(dy, w, dz, b_t=True, act=ops.ACT_DGELU, aux=zz, colsum=cs)
    zf = zz.float().requires_grad_(True)
    torch.nn.functional.gelu(zf).backward(dy.float() @ w.float())
    assert _rel_err(dz, zf.grad)[0] < 5e-3
    assert _rel_err(cs, dz.float().sum(0))[0] < 1e-5                # fused bias gradient = colsum of the bf16 output
    # dgrad + residual
    dx = torch.empty(M, K, device="cuda", dtype=BF)
    w1 = _randn(N, K, scale=0.03, seed=32)
    r2 = _randn(M, K, seed=33)
    ops.gemm(dz, w1, dx, b_t=True, residual=r2)
    assert _rel_err(dx, dz.float() @ w1.float() + r2.float())[0] < 5e-3


def test_gemm_rejects_bad_arguments():
    import tinyrec._lib as L
    ops = _ops()
    a, b = _randn(64, 64), _randn(30, 64)
    with pytest.raises(L.TinyRecError):
        ops.gemm(a, b, torch.empty(64, 30, device="cuda", dtype=BF))      # N % 8 != 0


# ------------------------------------------------------------------ row kernels
def test_embed_ln():
    ops = _ops()
    n, L, E, V = 37, 30, 768, 30522
    g = torch.Generator(device="cuda").manual_seed(0)
    ids = torch.randint(0, V, (n, L), generator=g, device="cuda")
    x = torch.cat([ids, torch.ones_like(ids)], 1)
    word = _randn(V, E, scale=0.02, dtype=torch.float32, seed=1)
    pos, typ = _randn(512, E, scale=0.02, dtype=torch.float32, seed=2), _randn(2, E, scale=0.02, dtype=torch.float32, seed=3)
    gamma, beta = 1 + _randn(E, scale=0.1, dtype=torch.float32, seed=4), _randn(E, scale=0.1, dtype=torch.float32, seed=5)
    ref = torch.nn.functional.layer_norm(word[ids] + pos[:L] + typ[0], (E,), gamma, beta, 1e-12).reshape(n * L, E)
    for table in (word, word.to(BF)):
        out = torch.empty(n * L, E, device="cuda", dtype=BF)
        ops.embed_ln(x, L, table, pos, typ[0].contiguous(), gamma, beta, 1e-12, out)
        ref_t = ref if table.dtype == torch.float32 else torch.nn.functional.layer_norm(
            table.float()[ids] + pos[:L] + typ[0], (E,), gamma, beta, 1e-12).reshape(n * L, E)
        assert (out.float() - ref_t).abs().max() < 0.03      # bf16 output rounding of O(1..4) values
        assert _rel_err(out, ref_t)[0] < 4e-3


def test_layernorm_fwd_bwd():
    ops = _ops()
    rows, E = 1003, 768
    x = _randn(rows, E, seed=1)
    dy = _randn(rows, E, seed=2)
    gamma, beta = 1 + _randn(E, scale=0.1, dtype=torch.float32, seed=3), _randn(E, scale=0.1, dtype=torch.float32, seed=4)
    y = torch.empty_like(x)
    ops.layernorm_fwd(x, gamma, beta, 1e-12, y)
    xf = x.float().requires_grad_(True)
    gf, bf = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    ref = torch.nn.functional.layer_norm(xf, (E,), gf, bf, 1e-12)
    assert _rel_err(y, ref)[0] < 4e-3
    ref.backward(dy.float())
    dx = torch.empty_like(x)
    dg, db = torch.zeros(E, device="cuda"), torch.zeros(E, device="cuda")
    ops.layernorm_bwd(dy, x, gamma, 1e-12, dx, dg, db)
    assert _rel_err(dx, xf.grad)[0] < 5e-3
    assert _rel_err(dg, gf.grad)[0] < 1e-4
    assert _rel_err(db, bf.grad)[0] < 1e-4


def test_colsum():
    ops = _ops()
    x = _randn(5281, 3072, seed=1)
    out = torch.zeros(3072, device="cuda")
    ops.colsum(x, out)
    assert _rel_err(out, x.float().sum(0))[0] < 1e-5
    x2 = _randn(77, 200, seed=2)
    out2 = torch.zeros(200, device="cuda")
    ops.colsum(x2, out2)
    assert _rel_err(out2, x2.float().sum(0))[0] < 1e-5


# ------------------------------------------------------------------ attention
def _rel_matrix(relvec, L):
    """[A, 2L-1] bias vector -> the [A, L, L] matrix the reference adds (entry [i, j] = vec[(j - i) + L - 1])."""
    idx = torch.arange(L, device=relvec.device)
    return relvec[:, (idx[None, :] - idx[:, None]) + L - 1]


def _attn_ref(qkv, mask, relvec, n, L, A):
    relpos = _rel_matrix(relvec, L)
    E = qkv.shape[1] // 3
    q, k, v = [t.reshape(n, L, A, 64).permute(0, 2, 1, 3) for t in qkv.float().split(E, dim=1)]
    s = q @ k.transpose(-1, -2) / 8.0 + (1.0 - mask.float())[:, None, None, :] * -10000.0 + relpos[None]
    return (torch.softmax(s, -1) @ v).permute(0, 2, 1, 3).reshape(n * L, E)


@pytest.mark.parametrize("L", [30, 32, 9, 1])
def test_attention_fwd_bwd(L):
    ops = _ops()
    n, A, E = 11, 12, 768
    qkv = _randn(n * L, 3 * E, seed=1)
    g = torch.Generator(device="cuda").manual_seed(3)
    lens = torch.randint(1, L + 1, (n,), generator=g, device="cuda")
    lens[0] = L
    mask = (torch.arange(L, device="cuda")[None, :] < lens[:, None]).long()
    if n > 2:
        mask[2] = 0                                  # all-pad news
    x = torch.cat([torch.zeros_like(mask), mask], 1)
    relpos = _randn(A, 2 * L - 1, dtype=torch.float32, seed=4)
    ctx = torch.empty(n * L, E, device="cuda", dtype=BF)
    ops.attn_fwd(qkv, x, L, relpos, ctx, A)
    qf = qkv.float().requires_grad_(True)
    ref = _attn_ref(qf, mask, relpos, n, L, A)
    assert _rel_err(ctx, ref)[0] < 5e-3
    dctx = _randn(n * L, E, seed=5)
    ref.backward(dctx.float())
    dqkv = torch.empty_like(qkv)
    dbias = torch.zeros(3 * E, device="cuda")
    ops.attn_bwd(qkv, x, L, relpos, dctx, dqkv, A, dbias=dbias)
    assert _rel_err(dqkv, qf.grad)[0] < 6e-3
    assert _rel_err(dbias, dqkv.float().sum(0))[0] < 1e-5           # fused [bq|bk|bv] gradient = colsum(dqkv)


@pytest.mark.parametrize("L", [33, 64, 100, 180, 512])
def test_attention_long_fwd(L):
    """Streamed-KV kernel for body / abstract lengths (32 < L <= 512): ragged lengths, an all-pad row,
    tail query block and tail key chunk."""
    ops = _ops()
    n, A, E = (5, 12, 768) if L <= 180 else (2, 12, 768)
    qkv = _randn(n * L, 3 * E, seed=1)
    g = torch.Generator(device="cuda").manual_seed(3)
    lens = torch.randint(1, L + 1, (n,), generator=g, device="cuda")
    lens[0] = L
    mask = (torch.arange(L, device="cuda")[None, :] < lens[:, None]).long()
    mask[n - 1] = 0                                  # all-pad news
    x = torch.cat([torch.zeros_like(mask), mask], 1)
    relpos = _randn(A, 2 * L - 1, dtype=torch.float32, seed=4)
    ctx = torch.full((n * L, E), float("nan"), device="cuda", dtype=BF)
    ops.attn_fwd(qkv, x, L, relpos, ctx, A)
    ref = _attn_ref(qkv, mask, relpos, n, L, A)
    assert torch.isfinite(ctx.float()).all()
    assert _rel_err(ctx, ref)[0] < 5e-3
    per_row = (ctx.float() - ref).norm(dim=1) / (ref.norm(dim=1) + 1e-3)
    assert float(per_row.max()) < 3e-2


# ------------------------------------------------------------------ dropout (counter-based masks)
P_DROP = 0.1


def _seed_tensor(seed):
    return torch.tensor([seed], device="cuda", dtype=torch.int64)


def _keep(seed, site, n):
    from oracle.dropout import keep_mask
    return torch.from_numpy(keep_mask(seed, site, n, P_DROP)).cuda()


def test_dropout_mask_matches_oracle_generator():
    ops = _ops()
    for seed, site, n in ((12345, 3, 100003), (2 ** 40 + 17, 77, 4099), (0, 0, 8)):
        st = _seed_tensor(seed)
        got = ops.dropout_mask(ops.make_drop(st, site, P_DROP), n, "cuda").bool()
        want = _keep(seed, site, n)
        assert torch.equal(got, want)
    big = ops.dropout_mask(ops.make_drop(_seed_tensor(99), 5, P_DROP), 1 << 22, "cuda").float()
    assert abs(float(big.mean()) - (1 - P_DROP)) < 1e-3            # keep rate
    a, b = big[:-1], big[1:]
    assert abs(float(((a - a.mean()) * (b - b.mean())).mean())) < 1e-3   # neighbours uncorrelated
    other = ops.dropout_mask(ops.make_drop(_seed_tensor(100), 5, P_DROP), 1 << 22, "cuda").float()
    assert abs(float(((big - big.mean()) * (other - other.mean())).mean())) < 1e-3   # seeds independent


def test_gemm_dropout_epilogue():
    ops = _ops()
    M, N, K = 333, 768, 256
    a, b = _randn(M, K, seed=3), _randn(N, K, scale=0.05, seed=4)
    bias = _randn(N, dtype=torch.float32, seed=5)
    res = _randn(M, N, seed=6)
    st = _seed_tensor(4242)
    out = torch.empty(M, N, device="cuda", dtype=torch.float32)
    ops.gemm(a, b, out, bias=bias, residual=res, drop=ops.make_drop(st, 9, P_DROP))
    keep = _keep(4242, 9, M * N).reshape(M, N).float()
    ref = (a.float() @ b.float().t() + bias) * keep / (1 - P_DROP) + res.float()
    assert _rel_err(out, ref)[0] < 1e-4


def test_embed_ln_dropout_and_layernorm_bwd_drop_output():
    ops = _ops()
    n, L, E, V = 19, 30, 768, 1000
    g = torch.Generator(device="cuda").manual_seed(0)
    ids = torch.randint(0, V, (n, L), generator=g, device="cuda")
    x = torch.cat([ids, torch.ones_like(ids)], 1)
    word = _randn(V, E, scale=0.02, dtype=torch.float32, seed=1)
    pos, typ = _randn(512, E, scale=0.02, dtype=torch.float32, seed=2), _randn(2, E, scale=0.02, dtype=torch.float32, seed=3)
    gamma, beta = 1 + _randn(E, scale=0.1, dtype=torch.float32, seed=4), _randn(E, scale=0.1, dtype=torch.float32, seed=5)
    st = _seed_tensor(777)
    out = torch.empty(n * L, E, device="cuda", dtype=BF)
    ops.embed_ln(x, L, word, pos, typ[0].contiguous(), gamma, beta, 1e-12, out, drop=ops.make_drop(st, 1, P_DROP))
    keep = _keep(777, 1, n * L * E).reshape(n * L, E).float()
    ref = torch.nn.functional.layer_norm(word[ids] + pos[:L] + typ[0], (E,), gamma, beta, 1e-12).reshape(n * L, E)
    assert _rel_err(out, ref * keep / (1 - P_DROP))[0] < 4e-3
    assert torch.equal(out == 0, keep == 0) or float(((out == 0) != (keep == 0)).float().mean()) < 1e-4
    # LayerNorm backward: second output = dx * keep / (1 - p)
    rows = n * L
    xin, dy = _randn(rows, E, seed=6), _randn(rows, E, seed=7)
    dx, dxd = torch.empty_like(xin), torch.empty_like(xin)
    dg, db = torch.zeros(E, device="cuda"), torch.zeros(E, device="cuda")
    dsum = torch.zeros(E, device="cuda")
    ops.layernorm_bwd(dy, xin, gamma, 1e-12, dx, dg, db, dx_drop=dxd, drop=ops.make_drop(st, 1, P_DROP), dsum=dsum)
    assert _rel_err(dxd, dx.float() * keep / (1 - P_DROP))[0] < 4e-3
    assert _rel_err(dsum, (dx.float() * keep / (1 - P_DROP)).sum(0))[0] < 2e-3     # fused bias gradient
    ops.layernorm_bwd(dy, xin, gamma, 1e-12, dx, dg, db, dx_drop=dxd, drop=None)
    assert torch.equal(dxd, dx)


@pytest.mark.parametrize("L", [30, 17])
def test_attention_dropout_fwd_bwd(L):
    from oracle.dropout import attention_keep
    ops = _ops()
    n, A, E = 9, 12, 768
    qkv = _randn(n * L, 3 * E, seed=1)
    mask = torch.ones(n, L, device="cuda", dtype=torch.long)
    mask[1, L // 2:] = 0
    x = torch.cat([torch.zeros_like(mask), mask], 1)
    relpos = _randn(A, 2 * L - 1, dtype=torch.float32, seed=4)
    st = _seed_tensor(31337)
    drop = ops.make_drop(st, 21, P_DROP)
    ctx = torch.empty(n * L, E, device="cuda", dtype=BF)
    ops.attn_fwd(qkv, x, L, relpos, ctx, A, drop=drop)
    keep = torch.from_numpy(attention_keep(31337, 21, n * A, L, P_DROP)).cuda().float().reshape(n, A, L, L)
    qf = qkv.float().requires_grad_(True)
    q, k, v = [t.reshape(n, L, A, 64).permute(0, 2, 1, 3) for t in qf.split(E, dim=1)]
    s = q @ k.transpose(-1, -2) / 8.0 + (1.0 - mask.float())[:, None, None, :] * -10000.0 + _rel_matrix(relpos, L)[None]
    ref = ((torch.softmax(s, -1) * keep / (1 - P_DROP)) @ v).permute(0, 2, 1, 3).reshape(n * L, E)
    assert _rel_err(ctx, ref)[0] < 6e-3
    dctx = _randn(n * L, E, seed=5)
    ref.backward(dctx.float())
    dqkv = torch.empty_like(qkv)
    ops.attn_bwd(qkv, x, L, relpos, dctx, dqkv, A, drop=drop)
    assert _rel_err(dqkv, qf.grad)[0] < 8e-3


# ------------------------------------------------------------------ pooling
def _chk(label, value, bound):
    """assert value < bound, recording the measured value in the test report (tests/conftest.py)."""
    from conftest import report
    report(label, float(value), float(bound))
    assert value < bound, (label, value, bound)


def _row_rel(got, ref):
    """Largest relative error in norm over the rows of ``got`` (float64; absolute for an all-zero reference row)."""
    got, ref = got.double().reshape(got.shape[0], -1), ref.double().reshape(ref.shape[0], -1)
    err, den = (got - ref).norm(dim=1), ref.norm(dim=1)
    return float(torch.where(den > 0, err / den.clamp_min(1e-300), err).max())


# (n, S, C, Q, ldq, mask): S below, at and just past the 6-row cp.async ring, S = POOL_SMAX = 512, every C the kernel
# is instantiated for, score rows inside a wider buffer (ldq > Q), and Q > 256, whose columns past 256 the kernels read
# straight from global memory (with a dw2 atomic per row)
@pytest.mark.parametrize("n,S,C,Q,ldq,with_mask", [
    (23, 30, 768, 200, 200, False), (23, 30, 768, 200, 200, True),
    (7, 1, 768, 200, 200, False),
    (9, 5, 256, 64, 64, False),
    (9, 6, 512, 200, 208, False),
    (9, 7, 768, 200, 256, False),
    (5, 100, 768, 200, 200, False),
    (3, 512, 768, 200, 200, False), (3, 512, 768, 200, 200, True),
    (6, 30, 1024, 264, 272, False),
    (4, 30, 768, 512, 512, False),
])
def test_attnpool_fwd_bwd(n, S, C, Q, ldq, with_mask):
    ops = _ops()
    case = f"n{n}_S{S}_C{C}_Q{Q}_ldq{ldq}" + ("_mask" if with_mask else "")
    x = _randn(n * S, C, seed=1)
    # the padding columns [Q, ldq) of the score rows belong to someone else: NaN there must not reach any output
    e = torch.full((n * S, ldq), float("nan"), device="cuda", dtype=BF)
    e[:, :Q] = torch.tanh(_randn(n * S, Q, seed=2).float()).to(BF)
    w2, b2 = _randn(Q, dtype=torch.float32, scale=0.1, seed=3), _randn(1, dtype=torch.float32, seed=4)
    mask = None
    if with_mask:
        g = torch.Generator(device="cuda").manual_seed(5)
        mask = (torch.rand(n, S, device="cuda", generator=g) > 0.3).float()
        mask[1] = 0
    out = torch.empty(n, C, device="cuda", dtype=BF)
    a = torch.empty(n, S, device="cuda")
    ops.attnpool_fwd(x, e, Q, w2, b2, mask, out, a, n, S)
    xf = x.double().reshape(n, S, C).requires_grad_(True)
    ef = e[:, :Q].double().reshape(n, S, Q).requires_grad_(True)
    w2f, b2f = w2.double().requires_grad_(True), b2.double().requires_grad_(True)
    alpha = torch.exp(ef @ w2f + b2f)
    if mask is not None:
        alpha = alpha * mask
    aref = alpha / (alpha.sum(1, keepdim=True) + 1e-8)
    ref = (aref.unsqueeze(-1) * xf).sum(1)
    assert bool(torch.isfinite(out.float()).all()) and bool(torch.isfinite(a).all())
    _chk(f"attnpool.a_row.{case}", _row_rel(a, aref), 1.2e-6)
    _chk(f"attnpool.out_row.{case}", _row_rel(out, ref), 4e-3)
    if with_mask:
        assert float(out[1].float().abs().max()) == 0.0
    dout = _randn(n, C, dtype=torch.float32, seed=6)
    ref.backward(dout.double())
    dx = torch.empty_like(x)
    sentinel = -3.0
    du = torch.full((n * S, ldq), sentinel, device="cuda", dtype=BF)
    # du, dw2 and db2 all carry dz_s = a_s (da_s - sum_t a_t da_t).  With one word (or one dominant word) the weights
    # cannot move and dz is zero in exact arithmetic up to the 1e-8 in the denominator, so both sides hold rounding
    # noise: measure them against the size of the terms dz is made of, a_s (|da_s| + |sum_t a_t da_t|)
    ad, ed = aref.detach(), ef.detach()
    da = torch.einsum("nsc,nc->ns", xf.detach(), dout.double())
    dz_mag = ad * (da.abs() + (ad * da).sum(1, keepdim=True).abs())
    du_mag = (dz_mag.unsqueeze(-1) * w2f.detach().abs() * (1 - ed ** 2)).reshape(n * S, Q)
    dw2_mag = (dz_mag.unsqueeze(-1) * ed.abs()).sum((0, 1))
    # dw2 / db2 are accumulated into: start from nonzero values below the size of the gradient, compare the increments
    dw2_0 = (torch.linspace(-0.5, 0.5, Q, device="cuda", dtype=torch.float64) * dw2_mag.max()).float()
    db2_0 = (0.25 * dz_mag.sum()).float().reshape(1)
    dw2, db2 = dw2_0.clone(), db2_0.clone()
    ops.attnpool_bwd(x, e, Q, w2, a, dout, dx, du, dw2, db2, n, S)
    assert bool(torch.isfinite(dx.float()).all()) and bool(torch.isfinite(du[:, :Q].float()).all())
    assert torch.equal(du[:, Q:], torch.full_like(du[:, Q:], sentinel)), "du written outside its Q columns"
    # dx_direct = a * dout (the part of dx not flowing through fc1)
    dx_ref = (ad.unsqueeze(-1) * dout.double().unsqueeze(1)).reshape(n * S, C)
    _chk(f"attnpool.dx.{case}", _rel_err(dx, dx_ref)[0], 4e-3)
    du_ref = (ef.grad * (1 - ed ** 2)).reshape(n * S, Q)
    _chk(f"attnpool.du.{case}", float((du[:, :Q].double() - du_ref).norm() / du_mag.norm()), 4e-3)
    _chk(f"attnpool.dw2.{case}", float(((dw2 - dw2_0).double() - w2f.grad).norm() / dw2_mag.norm()), 2e-7)
    _chk(f"attnpool.db2.{case}", float(((db2 - db2_0).double() - b2f.grad).abs().sum() / dz_mag.sum()), 8e-8)


# ------------------------------------------------------------------ fp32 head (TF32 mma path)
def _ue_ref(vecs, mask, pad, W1, b1, w2, b2, use_mask):
    """model_bert.py:155-176 (NAML) + :15-34 in torch fp32."""
    if use_mask:
        v = vecs
    else:
        v = vecs * mask.unsqueeze(-1) + pad.view(1, 1, -1) * (1 - mask.unsqueeze(-1))
    e = torch.tanh(v @ W1.t() + b1)
    alpha = torch.exp(e @ w2 + b2)
    if use_mask:
        alpha = alpha * mask
    a = alpha / (alpha.sum(1, keepdim=True) + 1e-8)
    return (a.unsqueeze(-1) * v).sum(1), a, e


@pytest.mark.parametrize("use_mask", [False, True])
@pytest.mark.parametrize("H,Q", [(50, 200), (13, 64), (64, 256)])
def test_user_encoder_multi_fwd_bwd(use_mask, H, Q):
    ops = _ops()
    B, D, n_enc = 7, 256, 3
    f32 = torch.float32
    mask = (torch.rand(B, H, device="cuda") > 0.3).float()
    mask[1] = 0                                   # all-masked history
    mask[2] = 1
    encs, refs, leaves = [], [], []
    for i in range(n_enc):
        vecs = _randn(B, H, D, dtype=f32, scale=0.5, seed=10 * i + 1)
        pad = _randn(D, dtype=f32, scale=0.5, seed=10 * i + 2)
        W1 = _randn(Q, D, dtype=f32, scale=0.06, seed=10 * i + 3)
        b1, w2, b2 = _randn(Q, dtype=f32, scale=0.1, seed=10 * i + 4), _randn(Q, dtype=f32, scale=0.1, seed=10 * i + 5), _randn(1, dtype=f32, seed=10 * i + 6)
        lv = [t.clone().requires_grad_(True) for t in (vecs, pad, W1, b1, w2, b2)]
        leaves.append(lv)
        refs.append(_ue_ref(lv[0], mask, *lv[1:], use_mask))
        encs.append(dict(vecs=vecs.view(B * H, D), pad_doc=pad, W1=W1, b1=b1, w2=w2, b2=b2,
                         user=torch.empty(B, D, device="cuda"), a=torch.empty(B, H, device="cuda"),
                         e=torch.empty(B, H, Q, device="cuda") if i == 0 else None))
    ops.user_encoder_fwd_multi(encs, mask, use_mask, B, H)
    for enc, (u, a, e) in zip(encs, refs):
        assert _rel_err(enc["user"], u)[0] < 2e-3
        assert _rel_err(enc["a"], a)[0] < 2e-3
        if use_mask:
            assert float(enc["user"][1].abs().max()) == 0.0          # 0 / (0 + 1e-8) -> exact zero
    assert _rel_err(encs[0]["e"], refs[0][2])[0] < 2e-3
    # backward of encoder 0
    d_user = _randn(B, D, dtype=f32, seed=99)
    refs[0][0].backward(d_user)
    v0, pad0, W10, b10, w20, b20 = leaves[0]
    d_vecs = _randn(B * H, D, dtype=f32, seed=98)                   # accumulates into existing gradient
    base = d_vecs.clone()
    dpad, dW1 = torch.zeros(D, device="cuda"), torch.zeros(Q, D, device="cuda")
    db1, dw2, db2 = torch.zeros(Q, device="cuda"), torch.zeros(Q, device="cuda"), torch.zeros(1, device="cuda")
    scratch = torch.empty(B * H * (Q + D), device="cuda")
    e_exact = refs[0][2].detach().contiguous()
    a_exact = refs[0][1].detach().contiguous()
    ops.user_encoder_bwd(encs[0]["vecs"], mask, encs[0]["pad_doc"], encs[0]["W1"], encs[0]["w2"], use_mask, a_exact, e_exact,
                         d_user, d_vecs, dpad, dW1, db1, dw2, db2, scratch, B, H)
    assert _rel_err(d_vecs - base, v0.grad.reshape(B * H, D))[0] < 3e-3
    assert _rel_err(dW1, W10.grad)[0] < 3e-3
    assert _rel_err(db1, b10.grad)[0] < 3e-3
    assert _rel_err(dw2, w20.grad)[0] < 3e-3
    assert _rel_err(db2, b20.grad)[0] < 3e-3 or float(b20.grad.abs().max()) < 1e-4
    if not use_mask:
        assert _rel_err(dpad, pad0.grad)[0] < 3e-3


@pytest.mark.parametrize("M,N,K,batch", [(1792, 256, 256, 4), (100, 72, 40, 1), (65, 200, 256, 2)])
def test_sgemm_nt_tf32(M, N, K, batch):
    ops = _ops()
    f32 = torch.float32
    A, Bm = _randn(batch, M, K, dtype=f32, seed=1), _randn(batch, N, K, dtype=f32, seed=2)
    bias = _randn(batch, N, dtype=f32, seed=3)
    C = torch.empty(batch, M, N, device="cuda")
    ops.sgemm_nt(A, Bm, bias, C, M, N, K, batch, M * K, N * K, N, M * N)
    ref = torch.einsum("bmk,bnk->bmn", A.double(), Bm.double()).float() + bias[:, None, :]
    assert _rel_err(C, ref)[0] < 1e-3                        # TF32 inputs (10-bit mantissa), fp32 accumulate


@pytest.mark.parametrize("R,N1,N2,batch", [(1792, 256, 256, 4), (1600, 200, 256, 1), (37, 64, 72, 2)])
def test_sgemm_tn_acc_tf32(R, N1, N2, batch):
    ops = _ops()
    f32 = torch.float32
    A, Bm = _randn(batch, R, N1, dtype=f32, seed=1), _randn(batch, R, N2, dtype=f32, seed=2)
    C = _randn(batch, N1, N2, dtype=f32, seed=3)
    cb = _randn(batch, N1, dtype=f32, seed=4)
    C0, cb0 = C.clone(), cb.clone()
    ops.sgemm_tn_acc(A, Bm, C, cb, R, N1, N2, batch, R * N1, R * N2, N1 * N2, N1)
    ref = torch.einsum("brm,brn->bmn", A.double(), Bm.double()).float()
    assert _rel_err(C - C0, ref)[0] < 1e-3
    assert _rel_err(cb - cb0, A.sum(1))[0] < 1e-4


@pytest.mark.parametrize("M,N,K,parts", [(1600, 256, 256, 3), (100, 72, 40, 1), (65, 200, 36, 2)])
def test_sgemm_nn_tf32(M, N, K, parts):
    ops = _ops()
    f32 = torch.float32
    A, Bm = _randn(parts, M, K, dtype=f32, seed=1), _randn(parts, K, N, dtype=f32, seed=2)
    C = torch.full((M, N), 7.0, device="cuda")
    ops.sgemm_nn(A, Bm, C, M, N, K, parts, M * K, K * N)
    ref = torch.einsum("pmk,pkn->mn", A.double(), Bm.double()).float()
    assert _rel_err(C, ref)[0] < 1e-3


# ------------------------------------------------------------------ NRMS self-attention (model_bert.py:37-100)
def _nrms_ref(q, k, v, mask, B, H, heads):
    """ScaledDotProductAttention.forward restated: exp (no max subtraction), mask, / (sum + 1e-8)."""
    sp = lambda t: t.view(B, H, heads, 16).transpose(1, 2)     # noqa: E731
    s = torch.exp(sp(q) @ sp(k).transpose(-1, -2) / 4.0)
    if mask is not None:
        s = s * mask[:, None, None, :]
    a = s / (s.sum(-1, keepdim=True) + 1e-8)
    return (a @ sp(v)).transpose(1, 2).reshape(B * H, heads * 16)


@pytest.mark.parametrize("with_mask", [False, True])
@pytest.mark.parametrize("B,H,heads", [(32, 50, 16), (3, 5, 16), (2, 64, 20), (5, 33, 3)])
def test_nrms_attention_fwd_bwd(with_mask, B, H, heads):
    ops = _ops()
    f32 = torch.float32
    Dh = heads * 16
    qkv = _randn(3, B * H, Dh, dtype=f32, seed=1, scale=0.7)
    mask = None
    if with_mask:
        mask = (torch.rand(B, H, generator=torch.Generator().manual_seed(3)) > 0.4).float().cuda()
        mask[0] = 0.0                                            # an all-masked history: ctx exactly 0
    ctx = torch.empty(B * H, Dh, device="cuda")
    ops.nrms_attn_fwd(qkv, mask, ctx, B, H)
    leaf = qkv.clone().requires_grad_(True)
    ref = _nrms_ref(leaf[0], leaf[1], leaf[2], mask, B, H, heads)
    assert _rel_err(ctx, ref.detach())[0] < 1e-5
    if with_mask:
        assert float(ctx[:H].abs().max()) == 0.0
    d_ctx = _randn(B * H, Dh, dtype=f32, seed=5)
    ref.backward(d_ctx)
    dqkv = torch.full_like(qkv, 9.0)
    ops.nrms_attn_bwd(qkv, mask, d_ctx, dqkv, B, H)
    for p, nm in enumerate("qkv"):
        assert _rel_err(dqkv[p], leaf.grad[p])[0] < 2e-5, nm


@pytest.mark.parametrize("use_mask", [False, True])
def test_nrms_blend_fwd_bwd(use_mask):
    ops = _ops()
    f32 = torch.float32
    R, D = 1600, 256
    v, pad = _randn(R, D, dtype=f32, seed=1), _randn(D, dtype=f32, seed=2)
    m = (torch.rand(R, generator=torch.Generator().manual_seed(3)) > 0.3).float().cuda()
    out = torch.empty(R, D, device="cuda")
    ops.nrms_blend_fwd(v, m, pad, out)
    assert torch.equal(out, v * m[:, None] + pad[None, :] * (1 - m[:, None]))
    g = _randn(R, D, dtype=f32, seed=4)
    d_v = _randn(R, D, dtype=f32, seed=5)
    d_v0 = d_v.clone()
    dpad = torch.zeros(D, device="cuda")
    ops.nrms_blend_bwd(g, None if use_mask else m, d_v, dpad)
    if use_mask:
        assert torch.equal(d_v, d_v0 + g) and float(dpad.abs().max()) == 0.0
    else:
        assert torch.equal(d_v, d_v0 + g * m[:, None])
        assert _rel_err(dpad, (g * (1 - m[:, None])).sum(0))[0] < 1e-5


@pytest.mark.parametrize("use_mask", [False, True])
def test_user_encoder_gather_equals_gather_then_encode(use_mask):
    """tnr_user_encoder_fwd_gather == tnr_gather_rows_f32 + tnr_user_encoder_fwd (same arithmetic, rows read from
    the table instead of a gathered copy; the logit partial sums meet in shared-memory atomics, so equality is to
    fp32 rounding, not bit for bit); unknown ids read row 0 (dataloader.py:74)."""
    ops = _ops()
    f32 = torch.float32
    B, H, D, Q, N = 37, 50, 256, 200, 1000
    table = _randn(N, D, dtype=f32, scale=0.5, seed=1)
    idx = torch.randint(0, N, (B, H), generator=torch.Generator().manual_seed(2)).int().cuda()
    idx[0, :3] = torch.tensor([-1, N, N + 5], dtype=torch.int32)
    mask = (torch.rand(B, H, generator=torch.Generator().manual_seed(3)) > 0.3).float().cuda()
    pad, W1 = _randn(D, dtype=f32, scale=0.5, seed=4), _randn(Q, D, dtype=f32, scale=0.06, seed=5)
    b1, w2, b2 = _randn(Q, dtype=f32, scale=0.1, seed=6), _randn(Q, dtype=f32, scale=0.1, seed=7), _randn(1, dtype=f32, seed=8)
    vecs = torch.empty(B * H, D, device="cuda")
    ops.gather_rows_f32(table, idx.reshape(-1), vecs)
    assert torch.equal(vecs[:3], table[0].expand(3, D))
    u0, a0 = torch.empty(B, D, device="cuda"), torch.empty(B, H, device="cuda")
    ops.user_encoder_fwd(vecs, mask, pad, W1, b1, w2, b2, use_mask, u0, a0, None, B, H)
    u1, a1 = torch.empty(B, D, device="cuda"), torch.empty(B, H, device="cuda")
    ops.user_encoder_fwd_gather(table, idx, mask, pad, W1, b1, w2, b2, use_mask, u1, a1)
    assert _rel_err(a1, a0)[0] < 1e-5 and _rel_err(u1, u0)[0] < 1e-5
    u2, a2 = torch.empty(B, D, device="cuda"), torch.empty(B, H, device="cuda")        # the flat scoring path
    ops.user_encoder_score(table, idx, mask, pad, ops.user_encoder_pack_w1(W1, pad, b1, w2), Q, b1, w2, b2, use_mask, u2, a2, B, H)
    # tcgen05 kind::tf32 TRUNCATES the fp32 history rows to TF32 (the per-impression kernel rounds them): 2^-11 per element
    assert _rel_err(a2, a0)[0] < 2e-3 and _rel_err(u2, u0)[0] < 2e-3
    ref_u, _, _ = _ue_ref(vecs.view(B, H, D), mask, pad, W1, b1, w2, b2, use_mask)
    assert _rel_err(u2, ref_u)[0] < 2e-3
    assert _rel_err(u1, ref_u)[0] < 2e-3


@pytest.mark.parametrize("use_mask", [False, True])
@pytest.mark.parametrize("B,H,Q,D", [(300, 50, 200, 256), (65, 7, 64, 256), (64, 64, 208, 256), (200, 50, 200, 64), (70, 20, 100, 128)])
def test_user_encoder_scoring_path_vs_torch(use_mask, B, H, Q, D):
    """Scoring-sized batches (B >= 64) take the flat logits GEMM + pooling kernels (tnr_user_encoder_score): same result as the
    torch fp32 restatement, incl. an all-masked history and a ragged last 64-row tile."""
    ops = _ops()
    f32 = torch.float32
    vecs = _randn(B, H, D, dtype=f32, scale=0.5, seed=1)
    mask = (torch.rand(B, H, generator=torch.Generator().manual_seed(2)) > 0.3).float().cuda()
    mask[1] = 0
    mask[2] = 1
    mask[3, : H // 2] = 0                                  # front-padded history, as the loader builds them
    mask[3, H // 2:] = 1
    mask[4] = 0.25                                         # a fractional mask: weight scaling / linear pad_doc blend
    mask[5, ::2] = 0.5
    pad, W1 = _randn(D, dtype=f32, scale=0.5, seed=4), _randn(Q, D, dtype=f32, scale=0.06, seed=5)
    b1, w2, b2 = _randn(Q, dtype=f32, scale=0.1, seed=6), _randn(Q, dtype=f32, scale=0.1, seed=7), _randn(1, dtype=f32, seed=8)
    user, a = torch.empty(B, D, device="cuda"), torch.empty(B, H, device="cuda")
    assert ops.user_encoder_score_supported(B, H, D, Q)
    ops.user_encoder_score(vecs.view(B * H, D), None, mask, pad, ops.user_encoder_pack_w1(W1, pad, b1, w2), Q, b1, w2, b2, use_mask,
                           user, a, B, H)
    ref_u, ref_a, _ = _ue_ref(vecs, mask, pad, W1, b1, w2, b2, use_mask)
    assert _rel_err(a, ref_a)[0] < 2e-3
    assert _rel_err(user, ref_u)[0] < 2e-3
    if use_mask:
        assert float(user[1].abs().max()) == 0.0


@pytest.mark.parametrize("L", [33, 64, 100, 180, 512])
def test_attention_long_bwd(L):
    """Backward of the streamed-KV attention (32 < L <= 512) against torch autograd on the fp32 restatement: ragged
    lengths (fully masked key chunks are skipped), an all-pad row, tail query / key blocks, fused bias gradient."""
    ops = _ops()
    n, A, E = (5, 12, 768) if L <= 180 else (2, 12, 768)
    qkv = _randn(n * L, 3 * E, seed=1)
    g = torch.Generator(device="cuda").manual_seed(3)
    lens = torch.randint(1, L + 1, (n,), generator=g, device="cuda")
    lens[0] = L
    mask = (torch.arange(L, device="cuda")[None, :] < lens[:, None]).long()
    mask[n - 1] = 0                                  # all-pad news
    x = torch.cat([torch.zeros_like(mask), mask], 1)
    relpos = _randn(A, 2 * L - 1, dtype=torch.float32, seed=4)
    qf = qkv.float().requires_grad_(True)
    ref = _attn_ref(qf, mask, relpos, n, L, A)
    dctx = _randn(n * L, E, seed=5)
    ref.backward(dctx.float())
    dqkv = torch.full_like(qkv, float("nan"))
    dbias = torch.zeros(3 * E, device="cuda")
    ops.attn_bwd(qkv, x, L, relpos, dctx, dqkv, A, dbias=dbias)
    assert torch.isfinite(dqkv.float()).all()
    for part, nm in enumerate("qkv"):
        sl = slice(part * E, (part + 1) * E)
        assert _rel_err(dqkv[:, sl], qf.grad[:, sl])[0] < 8e-3, nm
    assert _rel_err(dbias, dqkv.float().sum(0))[0] < 1e-4


@pytest.mark.parametrize("L", [48, 200])
def test_attention_long_dropout_adjoint(L):
    """With dropout the forward is still linear in V for a fixed seed, and the backward regenerates the same mask:
    <dO, ctx(V)> == <dV, V> (adjoint identity).  For L <= 64 the keep mask is read out of the forward and injected
    into the torch restatement, which pins dQ, dK and dV under dropout."""
    ops = _ops()
    n, A, E = 3, 12, 768
    qkv = _randn(n * L, 3 * E, seed=1, scale=0.5)
    mask = torch.ones(n, L, device="cuda", dtype=torch.long)
    mask[1, L // 2:] = 0
    x = torch.cat([torch.zeros_like(mask), mask], 1)
    relpos = _randn(A, 2 * L - 1, dtype=torch.float32, seed=4, scale=0.3)
    seed = _seed_tensor(77)                                         # must outlive `drop`: the kernels read it from HBM
    drop = ops.make_drop(seed, 5, P_DROP)
    ctx = torch.empty(n * L, E, device="cuda", dtype=BF)
    ops.attn_fwd(qkv, x, L, relpos, ctx, A, drop=drop)
    ctx2 = torch.empty_like(ctx)
    ops.attn_fwd(qkv, x, L, relpos, ctx2, A, drop=drop)
    assert torch.equal(ctx, ctx2)                                   # counter-based: same seed, same mask
    nodrop = torch.empty_like(ctx)
    ops.attn_fwd(qkv, x, L, relpos, nodrop, A)
    assert _rel_err(ctx, nodrop)[0] > 0.05                          # the mask is really applied
    dctx = _randn(n * L, E, seed=5)
    dqkv = torch.empty_like(qkv)
    ops.attn_bwd(qkv, x, L, relpos, dctx, dqkv, A, drop=drop)
    lhs = float((dctx.float() * ctx.float()).sum())
    rhs = float((dqkv[:, 2 * E:].float() * qkv[:, 2 * E:].float()).sum())
    assert abs(lhs - rhs) < 1e-2 * abs(lhs) + 1e-2, (lhs, rhs)
    if L > 64:
        return
    # L <= 64: read the keep mask out of the forward (V = one-hot rows make ctx[i, j] = dropout(P)_ij), inject it
    # into the torch restatement and compare ALL of dQ, dK, dV with autograd
    eye = torch.zeros(L, A, 64, device="cuda")
    eye[torch.arange(L), :, torch.arange(L)] = 1.0
    probe = qkv.clone()
    probe[:, 2 * E:] = eye.reshape(1, L, E).expand(n, L, E).reshape(n * L, E).to(BF)
    pm = torch.empty_like(ctx)
    ops.attn_fwd(probe, x, L, relpos, pm, A, drop=drop)
    keep = (pm.float().reshape(n, L, A, 64)[..., :L] != 0).permute(0, 2, 1, 3)          # [n, A, i, j]
    qf = qkv.float().requires_grad_(True)
    q, k, v = [t.reshape(n, L, A, 64).permute(0, 2, 1, 3) for t in qf.split(E, dim=1)]
    sc = q @ k.transpose(-1, -2) / 8.0 + (1.0 - mask.float())[:, None, None, :] * -10000.0 + _rel_matrix(relpos, L)[None]
    pr = torch.softmax(sc, -1)
    keep = keep | (pr < 1e-30)                                     # an exactly-zero probability reads as "dropped"
    ref = ((pr * keep / (1.0 - P_DROP)) @ v).permute(0, 2, 1, 3).reshape(n * L, E)
    assert _rel_err(ctx, ref.detach())[0] < 6e-3
    ref.backward(dctx.float())
    for part, nm in enumerate("qkv"):
        sl = slice(part * E, (part + 1) * E)
        assert _rel_err(dqkv[:, sl], qf.grad[:, sl])[0] < 8e-3, nm


@pytest.mark.parametrize("M,N", [(500, 3072), (4200, 3072), (4200, 296), (4133, 1000)])
def test_gemm_gelu_daux_and_mulaux(M, N):
    """FFN1 of a trained layer: C = gelu(z), aux = gelu'(z) (ACT_GELU_DAUX); its backward: dz = (dy W2) * aux
    (ACT_MULAUX) with the fused bias column sums.  M = 500: single-CTA kernels, M >= 4 133: CTA-pair kernels (both
    outputs through rotating 32 x 32 half boxes; N = 296 / 1 000 leave a clipped last half box, M = 4 133 ragged rows)."""
    ops = _ops()
    K = 768
    a, b = _randn(M, K, seed=7), _randn(N, K, scale=0.03, seed=8)
    bias = _randn(N, dtype=torch.float32, scale=0.1, seed=9)
    out = torch.empty(M, N, device="cuda", dtype=BF)
    dax = torch.empty(M, N, device="cuda", dtype=BF)
    ops.gemm(a, b, out, bias=bias, act=ops.ACT_GELU_DAUX, aux=dax)
    z = (a.float() @ b.float().t() + bias).requires_grad_(True)
    ref = torch.nn.functional.gelu(z)
    ref.sum().backward()
    assert _rel_err(out, ref.detach())[0] < 5e-3
    assert _rel_err(dax, z.grad)[0] < 5e-3
    assert float((dax.float() - z.grad).abs().max()) < 8e-3
    out2 = torch.empty_like(out)
    ops.gemm(a, b, out2, bias=bias, act=ops.ACT_GELU_DAUX)                 # no aux output: plain GELU
    assert _rel_err(out2, ref.detach())[0] < 5e-3
    dy, w = _randn(M, K, seed=29), _randn(K, N, scale=0.03, seed=30)
    dz = torch.empty(M, N, device="cuda", dtype=BF)
    cs = torch.zeros(N, device="cuda")
    ops.gemm(dy, w, dz, b_t=True, act=ops.ACT_MULAUX, aux=dax, colsum=cs)
    assert _rel_err(dz, (dy.float() @ w.float()) * dax.float())[0] < 5e-3
    assert _rel_err(cs, dz.float().sum(0))[0] < 1e-5
