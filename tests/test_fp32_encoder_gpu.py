"""The fp32 inference mode of the news encoder (``args.precision = 'fp32'``): its kernels against float64 torch, the
whole encoder against the reference's own fixtures and the float64 oracle, the table-build drivers, and the places
that must refuse it.

Bound: the 1e-4 parity level of BASELINE.json north_star, as the max over rows of the row-relative error
||y - ref|| / ||ref||; every measured error is recorded with conftest.report.  The single kernels are held to what
fp32 arithmetic gives (a few 1e-7 .. 1e-6) and the split GEMM to 2e-5."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import report

BOUND = 1e-4
gpu = pytest.mark.gpu


def _rowrel(got, ref):
    got = torch.as_tensor(got).double().cpu().reshape(ref.shape[0], -1)
    ref = torch.as_tensor(ref).double().cpu().reshape(ref.shape[0], -1)
    return float(((got - ref).norm(dim=1) / ref.norm(dim=1).clamp_min(1e-300)).max())


def _chk(label, value, bound):
    report(label, float(value), float(bound))
    assert value < bound, (label, value, bound)


def _sd64(sd):
    return {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}


# ------------------------------------------------------------------------------------------------ CPU-side checks
def test_precision_field_is_validated_on_the_host():
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    from tinyrec._lib import TinyRecError
    assert mb.NewsEncoder(synth.demo_args(num_student_layers=1)).precision == "bf16"          # reference args
    assert mb.NewsEncoder(synth.demo_args(num_student_layers=1, precision="fp32")).precision == "fp32"
    for bad in ("fp16", "FP32", "tf32", None):
        with pytest.raises(TinyRecError):
            mb.NewsEncoder(synth.demo_args(num_student_layers=1, precision=bad))


def test_train_state_refuses_an_fp32_news_encoder():
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    from tinyrec._lib import TinyRecError
    args = synth.demo_args(num_student_layers=1, num_teachers=0, precision="fp32")
    m = mb.ModelBert(args)
    with pytest.raises(TinyRecError, match="fp32"):
        mb.TrainState(m.news_encoder, m.user_encoder, [], [], torch.device("cpu"))


# ------------------------------------------------------------------------------------------------ split
def _split_ref(v):
    hi = v.bfloat16()
    return hi, (v - hi.float()).bfloat16()


def _layout(out, K, weight):
    a, b, c = out[:, :K], out[:, K:2 * K], out[:, 2 * K:]
    if weight:
        assert torch.equal(a, b)
        return a, c
    assert torch.equal(a, c)
    return a, b


@gpu
@pytest.mark.parametrize("rows,K,ld", [(7, 13, 13), (5, 33, 40), (64, 768, 768), (3, 1, 4), (9, 256, 260)])
def test_split_bf16x3_bit_exact(rows, K, ld):
    import tinyrec.ops as ops
    g = torch.Generator().manual_seed(rows * 1000 + K)
    full = torch.randn(rows, ld, generator=g) * torch.logspace(-30, 30, rows * ld).view(rows, ld)[:, torch.randperm(ld, generator=g)]
    full[0, : min(K, 3)] = 0.0
    full[-1, -1] = -3.4e38                                       # above bf16's largest finite: hi = -inf, as in torch
    x = full.cuda()[:, :K]
    for weight in (False, True):
        out = torch.empty(rows, 3 * K, device="cuda", dtype=torch.bfloat16)
        ops.split_bf16x3(x, out, weight=weight)
        hi, lo = _layout(out.cpu(), K, weight)
        rh, rl = _split_ref(full[:, :K])
        assert torch.equal(hi.view(torch.int16), rh.view(torch.int16)), weight
        assert torch.equal(lo.view(torch.int16), rl.view(torch.int16)), weight


@gpu
def test_split_bf16x3_gelu_is_exact_erf_gelu():
    """The split of gelu(x): hi / lo are the split of an fp32 value within a few ulps (plus the conditioning of erfc) of
    the float64 erf-GELU, the negative tail included, where the fp32 form 0.5 x (1 + erf(x / sqrt 2)) cancels."""
    import tinyrec.ops as ops
    g = torch.Generator().manual_seed(3)
    x = torch.cat([(torch.randn(4096, generator=g) * 3).clamp(-12, 12), torch.linspace(-12, 12, 4096)]).view(64, 128)
    out = torch.empty(64, 384, device="cuda", dtype=torch.bfloat16)
    ops.split_bf16x3(x.cuda(), out, gelu=True)
    hi, lo = _layout(out.cpu(), 128, False)
    # float64 erfc form: F.gelu's 1 + erf(x / sqrt 2) cancels to 0 even in float64 below x = -5.9
    g64 = 0.5 * x.double() * torch.special.erfc(-x.double() / 2 ** 0.5)
    assert float((g64 - F.gelu(x.double())).abs().max()) < 1e-14
    g32 = g64.float()
    # a few ulps, plus the conditioning of erfc at the fp32-rounded argument x / sqrt 2: up to x^2 ulps (144 at x = -12)
    window = 8 + x.double() ** 2
    ok = torch.zeros_like(x, dtype=torch.bool)
    for direction in (float("inf"), float("-inf")):
        y = g32.clone()
        for step in range(int(window.max()) + 1):
            rh, rl = _split_ref(y)
            ok |= (rh.view(torch.int16) == hi.view(torch.int16)) & (rl.view(torch.int16) == lo.view(torch.int16)) & (step <= window)
            y = torch.nextafter(y, torch.full_like(y, direction))
    assert bool(ok.all()), int((~ok).sum())
    rec = hi.double() + lo.double()
    # the GEMM epilogue's quintic GELU (2.6e-5 off) would not pass this reconstruction check
    err = float(((rec - g64).abs() / (g64.abs() + 1e-3)).max())
    _chk("fp32.split_gelu.rel", err, 2e-5)


# ------------------------------------------------------------------------------------------------ row kernels
@gpu
@pytest.mark.parametrize("E", [256, 768])
def test_embed_ln_f32_vs_float64(E):
    import tinyrec.ops as ops
    g = torch.Generator().manual_seed(E)
    n, L, vocab = 5, 7, 1000
    word = torch.randn(vocab, E, generator=g) * 0.05
    pos, type0 = torch.randn(64, E, generator=g) * 0.02, torch.randn(E, generator=g) * 0.02
    gamma, beta = 1 + 0.1 * torch.randn(E, generator=g), 0.1 * torch.randn(E, generator=g)
    ids = torch.randint(0, vocab, (n, L), generator=g)
    ids[1, 2], ids[2, 0], ids[3, 6] = -3, vocab, 10 ** 9            # out of vocabulary: clamped like the bf16 kernel
    x = torch.cat([ids, torch.ones(n, L, dtype=torch.int64)], 1)
    out = torch.empty(n * L, E, device="cuda")
    ops.embed_ln_f32(x.cuda(), L, word.cuda(), pos.cuda(), type0.cuda(), gamma.cuda(), beta.cuda(), 1e-12, out)
    cl = ids.clamp(0, vocab - 1)
    e = word.double()[cl] + pos.double()[:L] + type0.double()
    ref = F.layer_norm(e, (E,), gamma.double(), beta.double(), 1e-12).view(n * L, E)
    _chk(f"fp32.embed_ln.E{E}", _rowrel(out, ref), 2e-6)          # a bf16-rounded gather would be ~2e-3 off


@gpu
def test_add_layernorm_f32_vs_float64():
    import tinyrec.ops as ops
    g = torch.Generator().manual_seed(1)
    rows, E = 37, 768
    x, r = torch.randn(rows, E, generator=g) * 3 + 1, torch.randn(rows, E, generator=g)
    gamma, beta = 1 + 0.1 * torch.randn(E, generator=g), 0.1 * torch.randn(E, generator=g)
    out = torch.empty(rows, E, device="cuda")
    ops.add_layernorm_f32(x.cuda(), r.cuda(), gamma.cuda(), beta.cuda(), 1e-12, out)
    ref = F.layer_norm(x.double() + r.double(), (E,), gamma.double(), beta.double(), 1e-12)
    _chk("fp32.add_layernorm", _rowrel(out, ref), 2e-6)


# ------------------------------------------------------------------------------------------------ attention
def _attn_ref(qkv, mask, relpos, L, A, fp32_scores=False):
    """float64 attention.  ``fp32_scores``: the scores are formed as the kernel and the reference's fp32 code form them
    -- an fp32 dot product (sequential FMAs over the 64 dims), then ``+ (1 - mask) * -10000`` and ``+ relbias`` as two
    fp32 additions -- and only the softmax and P V are float64.  Adding -10000 in fp32 rounds a score to 2^-10, so a
    fully padded row is only defined to ~1e-3 by the reference's own arithmetic; this is what the kernel must match."""
    n = mask.shape[0]
    E = 64 * A
    q, k, v = (qkv.view(n, L, 3, A, 64)[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    idx = torch.arange(L)[None, :] - torch.arange(L)[:, None] + L - 1
    ext = ((1.0 - mask.float()) * -10000.0)[:, None, None, :]
    rel = relpos[:, idx][None]
    if fp32_scores:
        dot = torch.zeros(n, A, L, L)
        for d in range(64):             # fmaf: the product of two floats is exact in float64, one rounding to float
            dot = (dot.double() + q[..., d, None].double() * k[..., d][:, :, None, :].double()).float()
        s = ((dot * 0.125 + ext) + rel).double()
    else:
        s = q.double() @ k.double().transpose(-1, -2) / 8 + ext.double() + rel.double()
    return (torch.softmax(s, -1) @ v.double()).permute(0, 2, 1, 3).reshape(n * L, E)


@gpu
@pytest.mark.parametrize("L", [1, 12, 30, 32, 33, 100, 180, 512])
def test_attn_f32_vs_float64(L):
    import tinyrec.ops as ops
    g = torch.Generator().manual_seed(L)
    n, A = 3, 12
    E = 64 * A
    qkv = torch.randn(n * L, 3 * E, generator=g) * 1.5
    relpos = torch.randn(A, 2 * L - 1, generator=g)
    mask = torch.ones(n, L, dtype=torch.int64)
    mask[0] = 0                                                   # all-pad row (the pad news of every table)
    mask[1, max(1, L // 3):] = 0                                  # partial
    x = torch.cat([torch.zeros(n, L, dtype=torch.int64), mask], 1)
    ctx = torch.full((n * L, E), float("nan"), device="cuda")
    ops.attn_fwd_f32(qkv.cuda(), x.cuda(), L, relpos.cuda(), ctx, A)
    ref = _attn_ref(qkv, mask, relpos, L, A)
    ref32 = _attn_ref(qkv, mask, relpos, L, A, fp32_scores=True)
    # rows with an unmasked key against plain float64; every row, the all-pad one included, against fp32 score formation
    _chk(f"fp32.attn.L{L}.unpadded_rows", _rowrel(ctx[L:].view(-1, 64), ref[L:].view(-1, 64)), 1e-5)
    _chk(f"fp32.attn.L{L}.all_pad", _rowrel(ctx[:L].view(L * A, 64), ref32[:L].view(L * A, 64)), 1e-5)
    _chk(f"fp32.attn.L{L}", _rowrel(ctx.view(-1, 64), ref32.view(-1, 64)), 1e-5)
    report(f"fp32.attn.L{L}.all_pad_vs_float64_scores", _rowrel(ctx[:L].view(L * A, 64), ref[:L].view(L * A, 64)), None)


# ------------------------------------------------------------------------------------------------ pooling
@gpu
@pytest.mark.parametrize("S", [1, 30, 180, 512])
def test_attnpool_f32_vs_float64(S):
    import tinyrec.ops as ops
    g = torch.Generator().manual_seed(S)
    n, C, Q, ldq = 4, 768, 200, 208
    x = torch.randn(n * S, C, generator=g)
    u_full = torch.full((n * S, ldq), float("nan"))
    u_full[:, :Q] = torch.randn(n * S, Q, generator=g) * 2
    w2, b2 = torch.randn(Q, generator=g) * 0.1, torch.randn(1, generator=g)
    out = torch.empty(n, C, device="cuda")
    ops.attnpool_fwd_f32(x.cuda(), u_full.cuda()[:, :Q], Q, w2.cuda(), b2.cuda(), out, n, S)
    alpha = torch.exp(torch.tanh(u_full[:, :Q].double()) @ w2.double() + b2.double()).view(n, S)
    alpha = alpha / (alpha.sum(1, keepdim=True) + 1e-8)
    ref = torch.einsum("ns,nsc->nc", alpha, x.double().view(n, S, C))
    _chk(f"fp32.attnpool.S{S}", _rowrel(out, ref), 2e-6)


# ------------------------------------------------------------------------------------------------ split GEMM
@gpu
@pytest.mark.parametrize("K,N", [(768, 2304), (3072, 768), (768, 200)])
def test_bf16x3_gemm_vs_float64(K, N):
    import tinyrec.ops as ops
    g = torch.Generator().manual_seed(K + N)
    M = 1000                                                      # ragged: not a multiple of the 128-row tile
    a, w, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) * 0.02, torch.randn(N, generator=g) * 0.1
    ac, wc = a.cuda(), w.cuda()
    a3 = ops.split_bf16x3(ac, torch.empty(M, 3 * K, device="cuda", dtype=torch.bfloat16))
    w3 = ops.split_bf16x3(wc, torch.empty(N, 3 * K, device="cuda", dtype=torch.bfloat16), weight=True)
    out = torch.empty(M, N, device="cuda")
    ops.gemm(a3, w3, out, bias=b.cuda())
    ref = a.double() @ w.double().T + b.double()
    _chk(f"fp32.gemm_bf16x3.K{K}.N{N}", _rowrel(out, ref), 2e-5)
    plain = torch.empty(M, N, device="cuda")
    ops.gemm(ac.bfloat16(), wc.bfloat16(), plain, bias=b.cuda())
    report(f"fp32.gemm_plain_bf16.K{K}.N{N}", _rowrel(plain, ref), None)


# ------------------------------------------------------------------------------------------------ whole encoder
def _news_encoder(layers, sd, **over):
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    nsd = {k[len("news_encoder."):]: v for k, v in sd.items() if k.startswith("news_encoder.")}
    ne = mb.NewsEncoder(synth.demo_args(num_student_layers=layers, precision="fp32", **over))
    ne.load_state_dict(nsd, strict=True)
    return ne.cuda().eval()


@gpu
def test_news_encoder_fp32_vs_reference_golden(golden):
    import tinyrec.synth as synth
    g = golden("encoder")
    layers = int(g["layers"])
    ne = _news_encoder(layers, synth.model_bert_state("", layers, int(g["seed"]), noisy=True))
    with torch.no_grad():
        vec = ne(torch.from_numpy(g["x"]).cuda())
    _chk("fp32.golden.news_vec", _rowrel(vec, torch.from_numpy(g["news_vec"])), BOUND)


@gpu
@pytest.mark.parametrize("tag,ulm", [("pad", False), ("mask", True)])
def test_model_bert_fp32_vs_reference_golden(golden, tag, ulm):
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    g = golden("modelbert")
    layers = int(g["layers"])
    H = g["history"].shape[1]
    m = mb.ModelBert(synth.demo_args(num_student_layers=layers, user_log_length=H, user_log_mask=ulm, precision="fp32"))
    m.load_state_dict(synth.model_bert_state("", layers, int(g["seed"]), noisy=True), strict=True)
    m.cuda().eval()
    with torch.no_grad():
        score, hv, cv, uv = m(torch.from_numpy(g["history"]).cuda(), torch.from_numpy(g["history_mask"]).cuda(),
                              torch.from_numpy(g["candidate"]).cuda())
    D = hv.shape[-1]
    _chk(f"fp32.golden.hist_{tag}", _rowrel(hv.reshape(-1, D), torch.from_numpy(g[f"hist_{tag}"]).reshape(-1, D)), BOUND)
    _chk(f"fp32.golden.cand_{tag}", _rowrel(cv.reshape(-1, D), torch.from_numpy(g[f"cand_{tag}"]).reshape(-1, D)), BOUND)


@gpu
@pytest.mark.parametrize("L,rows", [(30, 8), (180, 3)])
def test_news_encoder_fp32_vs_float64_oracle_12_layers(L, rows):
    import tinyrec.synth as synth
    from oracle import model as om
    layers = 12
    sd = synth.model_bert_state("", layers, 7, noisy=True)
    news = synth.news_table(rows - 1, L=L, seed=L, mean_len=0.6 * L, std_len=0.2 * L)    # row 0: the all-pad news
    x = torch.from_numpy(news.astype(np.int64))
    ne = _news_encoder(layers, sd)
    with torch.no_grad():
        vec = ne(x.cuda())
        ref = om.news_encoder(_sd64(sd), "news_encoder.", x, layers)
    _chk(f"fp32.oracle64.12L.L{L}", _rowrel(vec, ref), BOUND)
    _chk(f"fp32.oracle64.12L.L{L}.pad_row", _rowrel(vec[:1], ref[:1]), BOUND)


# ------------------------------------------------------------------------------------------------ drivers
@gpu
def test_build_news_table_fp32():
    import tinyrec.run as trun
    import tinyrec.synth as synth
    from oracle import model as om
    layers, L, n_news = 2, 16, 149
    news = synth.news_table(n_news, L=L, seed=9)
    sd = synth.model_bert_state("", layers, 4, noisy=True)
    ne = _news_encoder(layers, sd)
    tab = trun.build_news_table(ne, news, batch_size=64)
    assert tuple(tab.shape) == (n_news + 1, 256) and tab.dtype == torch.float32
    assert torch.equal(tab, trun.build_news_table(ne, news, batch_size=4096))    # batching is invisible, bit for bit
    x = torch.from_numpy(news.astype(np.int64))
    with torch.no_grad():
        row0 = ne(x[:1].cuda())
        ref = om.news_encoder(_sd64(sd), "news_encoder.", x, layers)
    _chk("fp32.build_news_table.row0_vs_per_row", _rowrel(tab[:1], row0), 1e-6)
    _chk("fp32.build_news_table.oracle64", _rowrel(tab, ref), BOUND)


@gpu
def test_get_teacher_emb_fp32(tmp_path):
    import tinyrec.checkpoint as ckpt
    import tinyrec.model_bert_2 as mb2
    import tinyrec.run as trun
    import tinyrec.synth as synth
    from oracle import model as om
    layers, L = 2, 12
    news = synth.news_table(99, L=L, seed=2)
    args = synth.demo_args(num_hidden_layers=layers, batch_size=1, enable_hvd=False, precision="fp32")
    sd = synth.model_bert_state("", layers, 31, noisy=True)
    m = mb2.ModelBert(args)
    m.load_state_dict(sd, strict=True)
    p, out = str(tmp_path / "teacher.pt"), str(tmp_path / "teacher.pkl")
    ckpt.save_checkpoint(p, m)
    args.teacher_ckpts, args.teacher_emb_paths = [p], [out]
    tables = trun.get_teacher_emb(args, None, news)
    arr = ckpt.load_teacher_table(out)
    assert arr.dtype == np.float32 and arr.shape == (100, 256) and np.array_equal(arr, tables[0])
    with torch.no_grad():
        ref = om.news_encoder(_sd64(sd), "news_encoder.", torch.from_numpy(news.astype(np.int64)), layers)
    _chk("fp32.get_teacher_emb.oracle64", _rowrel(torch.from_numpy(arr), ref), BOUND)


# ------------------------------------------------------------------------------------------------ refusals
@gpu
def test_fp32_refuses_training_mode_and_the_train_step():
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    from tinyrec._lib import TinyRecError
    layers, B, H, K, L = 1, 2, 3, 2, 8
    args = synth.demo_args(num_student_layers=layers, num_teachers=0, user_log_length=H, precision="fp32")
    model = mb.Model(args).cuda()
    x = torch.from_numpy(synth.news_table(5, L=L, seed=1).astype(np.int64)).cuda()
    with pytest.raises(TinyRecError, match="eval"):
        model.student.news_encoder(x)                       # a freshly built module is in training mode
    model.eval()
    assert model.student.news_encoder(x).shape == (6, 256)
    hist, cand = x[1:].view(1, 5, -1)[:, :H].expand(B, H, -1), x[1:3].view(1, K, -1).expand(B, K, -1)
    with torch.no_grad(), pytest.raises(TinyRecError, match="fp32"):
        model(hist, torch.ones(B, H, device="cuda"), cand, torch.zeros(B, dtype=torch.int64, device="cuda"), [], [])
