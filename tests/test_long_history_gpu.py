"""User histories longer than 64 clicks (64 < user_log_length <= 512): the chunked NAML user-encoder kernels, the
scoring path's pooling kernel, the per-head NRMS self-attention kernels, the rejections at H = 0 and H = 513, and the
model / drivers at long H against the CPU oracle.

Bounds are those of the H <= 64 tests: 2e-3 for user / a / e through TF32, 3e-3 for the user-encoder gradients, 1e-5 /
2e-5 for the NRMS forward / backward, SCORE_TOL and GRAD_TOL for the model.  A softmax over more rows needs no looser
bound: every output is a convex combination, and the relative error of each weight does not grow with H."""
import numpy as np
import pytest
import torch

from conftest import report

pytestmark = pytest.mark.gpu

F32, F64 = torch.float32, torch.float64
SCORE_TOL = 1e-2
GRAD_TOL = 3e-2


def _ops():
    import tinyrec.ops as ops
    return ops


def _chk(label, value, bound):
    report(label, float(value), float(bound))
    assert value < bound, (label, value, bound)


def _rel(got, ref):
    got, ref = torch.as_tensor(got).double().cpu(), torch.as_tensor(ref).double().cpu()
    return float((got - ref).norm() / (ref.norm() + 1e-30))


def _randn(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(*shape, generator=g, device="cuda") * scale


def _ue_ref(vecs, mask, pad, W1, b1, w2, b2, use_mask):
    """model_bert.py:155-176 (NAML) + :15-34, in float64."""
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


def _long_mask(B, H, seed):
    """Front-padded random histories plus the edges of the chunked kernels: an all-masked history, a full one, one
    whose only live rows are in the last 64-row chunk, a single live row at h = H - 1 and fractional masks."""
    g = torch.Generator().manual_seed(seed)
    mask = (torch.rand(B, H, generator=g) > 0.3).float()
    mask[1] = 0
    mask[2] = 1
    c0 = (H - 1) // 64 * 64
    mask[3, :c0] = 0
    mask[3, c0:] = 1
    mask[4] = 0
    mask[4, H - 1] = 1
    mask[5] = 0.25
    mask[6, ::2] = 0.5
    return mask.cuda()


# ------------------------------------------------------------------ NAML user encoder, forward + backward
@pytest.mark.parametrize("use_mask", [False, True])
@pytest.mark.parametrize("H", [65, 100, 128, 200, 512])
def test_user_encoder_long_fwd_bwd(use_mask, H):
    ops = _ops()
    B, D, Q, n_enc, N = 7, 256, 200, 3, 3000
    case = f"H{H}_mask{int(use_mask)}"
    mask = _long_mask(B, H, seed=H)
    encs, refs, leaves = [], [], []
    for i in range(n_enc):
        vecs = _randn(B, H, D, scale=0.5, seed=10 * i + 1)
        pad = _randn(D, scale=0.5, seed=10 * i + 2)
        W1 = _randn(Q, D, scale=0.06, seed=10 * i + 3)
        b1, w2, b2 = _randn(Q, scale=0.1, seed=10 * i + 4), _randn(Q, scale=0.1, seed=10 * i + 5), _randn(1, seed=10 * i + 6)
        lv = [t.double().requires_grad_(True) for t in (vecs, pad, W1, b1, w2, b2)]
        leaves.append(lv)
        refs.append(_ue_ref(lv[0], mask.double(), *lv[1:], use_mask))
        encs.append(dict(vecs=vecs.view(B * H, D), pad_doc=pad, W1=W1, b1=b1, w2=w2, b2=b2,
                         user=torch.empty(B, D, device="cuda"), a=torch.empty(B, H, device="cuda"),
                         e=torch.empty(B, H, Q, device="cuda") if i == 0 else None))
    ops.user_encoder_fwd_multi(encs, mask, use_mask, B, H)
    for i, (enc, (u, a, e)) in enumerate(zip(encs, refs)):
        _chk(f"long_ue.multi.user.{case}.enc{i}", _rel(enc["user"], u.detach()), 2e-3)
        _chk(f"long_ue.multi.a.{case}.enc{i}", _rel(enc["a"], a.detach()), 2e-3)
        if use_mask:
            assert float(enc["user"][1].abs().max()) == 0.0          # all-masked history: 0 / (0 + 1e-8) -> exact zero
    _chk(f"long_ue.multi.e.{case}", _rel(encs[0]["e"], refs[0][2].detach()), 2e-3)
    # plain form: the same kernel as encoder 1 of the multi launch
    e1 = encs[1]
    u, a = torch.empty(B, D, device="cuda"), torch.empty(B, H, device="cuda")
    ops.user_encoder_fwd(e1["vecs"], mask, e1["pad_doc"], e1["W1"], e1["b1"], e1["w2"], e1["b2"], use_mask, u, a, None, B, H)
    _chk(f"long_ue.plain.user.{case}", _rel(u, refs[1][0].detach()), 2e-3)
    _chk(f"long_ue.plain.a.{case}", _rel(a, refs[1][1].detach()), 2e-3)
    # gather form, with out-of-range ids (they read row 0)
    table = _randn(N, D, scale=0.5, seed=77)
    idx = torch.randint(0, N, (B, H), generator=torch.Generator().manual_seed(H)).int()
    idx[0, :3] = torch.tensor([-1, N, N + 5], dtype=torch.int32)
    idx[2, H - 2:] = torch.tensor([-7, N], dtype=torch.int32)
    idx = idx.cuda()
    ug, ag = torch.empty(B, D, device="cuda"), torch.empty(B, H, device="cuda")
    ops.user_encoder_fwd_gather(table, idx, mask, e1["pad_doc"], e1["W1"], e1["b1"], e1["w2"], e1["b2"], use_mask, ug, ag)
    safe = torch.where((idx >= 0) & (idx < N), idx, torch.zeros_like(idx)).long()
    rg, ra, _ = _ue_ref(table.double()[safe], mask.double(), *[t.detach() for t in leaves[1][1:]], use_mask)
    _chk(f"long_ue.gather.user.{case}", _rel(ug, rg), 2e-3)
    _chk(f"long_ue.gather.a.{case}", _rel(ag, ra), 2e-3)
    # backward of encoder 0 (exact a and e in, as the train step feeds its own forward's)
    d_user = _randn(B, D, seed=99)
    refs[0][0].backward(d_user.double())
    v0, pad0, W10, b10, w20, b20 = leaves[0]
    d_vecs = _randn(B * H, D, seed=98)                               # accumulates into an existing gradient
    base = d_vecs.clone()
    dpad, dW1 = torch.zeros(D, device="cuda"), torch.zeros(Q, D, device="cuda")
    db1, dw2, db2 = torch.zeros(Q, device="cuda"), torch.zeros(Q, device="cuda"), torch.zeros(1, device="cuda")
    scratch = torch.empty(B * H * (Q + D), device="cuda")
    ops.user_encoder_bwd(encs[0]["vecs"], mask, encs[0]["pad_doc"], encs[0]["W1"], encs[0]["w2"], use_mask,
                         refs[0][1].detach().float().contiguous(), refs[0][2].detach().float().contiguous(),
                         d_user, d_vecs, dpad, dW1, db1, dw2, db2, scratch, B, H)
    _chk(f"long_ue.bwd.d_vecs.{case}", _rel(d_vecs - base, v0.grad.reshape(B * H, D)), 3e-3)
    _chk(f"long_ue.bwd.dW1.{case}", _rel(dW1, W10.grad), 3e-3)
    _chk(f"long_ue.bwd.db1.{case}", _rel(db1, b10.grad), 3e-3)
    _chk(f"long_ue.bwd.dw2.{case}", _rel(dw2, w20.grad), 3e-3)
    # d loss / d b2 is zero up to the 1e-8 in the denominator: measure against the dw2 scale
    _chk(f"long_ue.bwd.db2.{case}", float((db2.double().cpu() - b20.grad.cpu()).abs().max() / w20.grad.norm().cpu()), 3e-3)
    if not use_mask:
        _chk(f"long_ue.bwd.dpad.{case}", _rel(dpad, pad0.grad), 3e-3)


# ------------------------------------------------------------------ scoring path (flat logits GEMM + pooling)
@pytest.mark.parametrize("use_mask", [False, True])
@pytest.mark.parametrize("H,D", [(65, 256), (128, 256), (512, 256), (65, 64), (128, 64), (512, 64)])
def test_user_encoder_score_long(use_mask, H, D):
    ops = _ops()
    B, Q, N = 70, 200, 5000
    case = f"H{H}_D{D}_mask{int(use_mask)}"
    mask = _long_mask(B, H, seed=H + 1)
    table = _randn(N, D, scale=0.5, seed=1)
    idx = torch.randint(0, N, (B, H), generator=torch.Generator().manual_seed(2)).int()
    idx[0, :3] = torch.tensor([-1, N, N + 5], dtype=torch.int32)
    idx = idx.cuda()
    pad, W1 = _randn(D, scale=0.5, seed=4), _randn(Q, D, scale=0.06, seed=5)
    b1, w2, b2 = _randn(Q, scale=0.1, seed=6), _randn(Q, scale=0.1, seed=7), _randn(1, seed=8)
    assert ops.user_encoder_score_supported(B, H, D, Q)
    user, a = torch.empty(B, D, device="cuda"), torch.empty(B, H, device="cuda")
    ops.user_encoder_score(table, idx, mask, pad, ops.user_encoder_pack_w1(W1, pad, b1, w2), Q, b1, w2, b2, use_mask, user, a, B, H)
    safe = torch.where((idx >= 0) & (idx < N), idx, torch.zeros_like(idx)).long()
    ref_u, ref_a, _ = _ue_ref(table.double()[safe], mask.double(), pad.double(), W1.double(), b1.double(), w2.double(),
                              b2.double(), use_mask)
    _chk(f"long_score.user.{case}", _rel(user, ref_u), 2e-3)
    _chk(f"long_score.a.{case}", _rel(a, ref_a), 2e-3)
    if use_mask:
        assert float(user[1].abs().max()) == 0.0
    # against the per-impression kernel (it rounds the rows to TF32, the tcgen05 GEMM truncates them)
    u1, a1 = torch.empty(B, D, device="cuda"), torch.empty(B, H, device="cuda")
    ops.user_encoder_fwd_gather(table, idx, mask, pad, W1, b1, w2, b2, use_mask, u1, a1)
    _chk(f"long_score.vs_per_impression.user.{case}", _rel(user, u1), 2e-3)
    _chk(f"long_score.vs_per_impression.a.{case}", _rel(a, a1), 2e-3)


# ------------------------------------------------------------------ NRMS self-attention
def _nrms_ref(q, k, v, mask, B, H, heads):
    """ScaledDotProductAttention.forward restated: exp (no max subtraction), mask, / (sum + 1e-8)."""
    sp = lambda t: t.view(B, H, heads, 16).transpose(1, 2)     # noqa: E731
    s = torch.exp(sp(q) @ sp(k).transpose(-1, -2) / 4.0)
    if mask is not None:
        s = s * mask[:, None, None, :]
    a = s / (s.sum(-1, keepdim=True) + 1e-8)
    return (a @ sp(v)).transpose(1, 2).reshape(B * H, heads * 16)


@pytest.mark.parametrize("with_mask", [False, True])
@pytest.mark.parametrize("H", [65, 100, 256, 512])
def test_nrms_attention_long_fwd_bwd(with_mask, H):
    ops = _ops()
    B, heads = 3, 16
    Dh = heads * 16
    case = f"H{H}_mask{int(with_mask)}"
    qkv = _randn(3, B * H, Dh, seed=1, scale=0.7)
    mask = None
    if with_mask:
        mask = (torch.rand(B, H, generator=torch.Generator().manual_seed(3)) > 0.4).float().cuda()
        mask[0] = 0.0                                            # an all-masked history: ctx exactly 0
        mask[2, :H - 1] = 0.0                                    # one live key, the last one
    ctx = torch.full((B * H, Dh), float("nan"), device="cuda")
    ops.nrms_attn_fwd(qkv, mask, ctx, B, H)
    leaf = qkv.double().requires_grad_(True)
    ref = _nrms_ref(leaf[0], leaf[1], leaf[2], None if mask is None else mask.double(), B, H, heads)
    _chk(f"long_nrms.ctx.{case}", _rel(ctx, ref.detach()), 1e-5)
    if with_mask:
        assert float(ctx[:H].abs().max()) == 0.0
    d_ctx = _randn(B * H, Dh, seed=5)
    ref.backward(d_ctx.double())
    dqkv = torch.full_like(qkv, float("nan"))                   # unwritten entries show as NaN
    ops.nrms_attn_bwd(qkv, mask, d_ctx, dqkv, B, H)
    assert bool(torch.isfinite(dqkv).all())
    for p, nm in enumerate("qkv"):
        _chk(f"long_nrms.d{nm}.{case}", _rel(dqkv[p], leaf.grad[p]), 2e-5)


# ------------------------------------------------------------------ rejections
@pytest.mark.parametrize("H", [0, 513])
def test_history_length_rejected(H):
    from tinyrec._lib import TinyRecError
    import tinyrec.run as trun
    ops = _ops()
    B, D, Q, N = 64, 256, 200, 100
    z = lambda *s: torch.zeros(*s, device="cuda")          # noqa: E731
    vecs, mask, pad, W1, b1, w2, b2 = z(B * H, D), z(B, H), z(D), z(Q, D), z(Q), z(Q), z(1)
    user, a, e = z(B, D), z(B, H), z(B, H, Q)
    idx = torch.zeros(B, H, device="cuda", dtype=torch.int32)
    msg = "history length"
    with pytest.raises(TinyRecError, match=msg):
        ops.user_encoder_fwd(vecs, mask, pad, W1, b1, w2, b2, True, user, a, e, B, H)
    with pytest.raises(TinyRecError, match=msg):
        ops.user_encoder_fwd_multi([dict(vecs=vecs, pad_doc=pad, W1=W1, b1=b1, w2=w2, b2=b2, user=user, a=a, e=None)],
                                   mask, True, B, H)
    with pytest.raises(TinyRecError, match=msg + "|idx and a non-empty table"):        # H = 0: no ids at all
        ops.user_encoder_fwd_gather(z(N, D), idx, mask, pad, W1, b1, w2, b2, True, user, a)
    with pytest.raises(TinyRecError, match=msg):
        ops.user_encoder_bwd(vecs, mask, pad, W1, w2, True, a, e, user, z(B * H, D), z(D), z(Q, D), z(Q), z(Q), z(1),
                             z(max(B * H * (Q + D), 4)), B, H)
    with pytest.raises(TinyRecError, match=msg):
        ops.user_encoder_score(z(N, D), idx, mask, pad, ops.user_encoder_pack_w1(W1, pad, b1, w2), Q, b1, w2, b2, True,
                               user, a, B, H)
    assert not ops.user_encoder_score_supported(B, 513, D, Q)
    qkv = z(3, B * H, 64)
    with pytest.raises(TinyRecError, match=msg):
        ops.nrms_attn_fwd(qkv, mask, z(B * H, 64), B, H)
    with pytest.raises(TinyRecError, match=msg):
        ops.nrms_attn_bwd(qkv, mask, z(B * H, 64), z(3, B * H, 64), B, H)
    # the drivers refuse before staging anything
    hist = np.zeros((4, H), dtype=np.int32)
    with pytest.raises(TinyRecError, match="user_log_length"):
        trun.evaluate(None, z(N, D), hist, hist.astype(np.float32), np.arange(5, dtype=np.int64), np.zeros(4, np.int32),
                      np.zeros(4, np.int8))


# ------------------------------------------------------------------ model and drivers against the oracle
def _grad_err(name, got, ref, named):
    """As tests/test_model_gpu.py: gradients that are zero up to rounding (key / W_K biases, att_fc2.bias, the NRMS
    pooling parameters) are measured against the scale of their neighbours."""
    got, ref = torch.as_tensor(got).float().cpu(), torch.as_tensor(ref).float().cpu()
    if name.endswith("attention.self.key.bias"):
        scale = named[name.replace("key.bias", "query.bias")].grad.float().norm().cpu()
        return float((got - ref).norm() / (scale + 1e-12))
    if name.endswith("multi_head_self_attn.W_K.bias"):
        scale = named[name.replace("W_K.bias", "W_Q.bias")].grad.float().norm().cpu()
        return float((got - ref).norm() / (scale + 1e-12))
    if ".user_encoder.attn." in name and name.replace("attn." + name.split("attn.")[1], "multi_head_self_attn.W_V.weight") in named:
        wv = named[name.replace("attn." + name.split("attn.")[1], "multi_head_self_attn.W_V.weight")].grad
        return float((got - ref).norm() / (max(float(ref.norm()), float(wv.float().norm().cpu())) + 1e-12))
    if name.endswith("attn.att_fc2.bias"):
        scale = named[name.replace("att_fc2.bias", "att_fc2.weight")].grad.float().norm().cpu()
        return float((got - ref).norm() / (scale + 1e-12))
    return float((got - ref).norm() / (ref.norm() + 1e-12))


def _apply_freeze(model, trainable_layers):
    """run.py:101-112: teachers frozen, the student's BERT trainable in ``trainable_layers`` only."""
    for p in model.teachers.parameters():
        p.requires_grad = False
    bm = model.student.news_encoder.bert_model
    for p in bm.parameters():
        p.requires_grad = False
    for i, layer in enumerate(bm.bert.encoder.layer):
        if i in trainable_layers:
            for p in layer.parameters():
                p.requires_grad = True


def _long_impressions(B, N, H, K, seed):
    """train_impressions with the first impression's history full: the rest are front-padded geometric lengths."""
    import tinyrec.synth as synth
    hist_idx, hmask, cand_idx, label = synth.train_impressions(B, N, H, K, seed=seed)
    hist_idx[0] = np.random.default_rng(seed).integers(1, N + 1, size=H)
    hmask[0] = 1.0
    return hist_idx, hmask, cand_idx, label


@pytest.mark.parametrize("model", ["NAML", "NRMS"])
@pytest.mark.parametrize("H", [100, 200])
def test_kd_step_long_history_vs_oracle(model, H):
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    from oracle import model as om
    B, K, L, M, layers, N = 4, 5, 12, 2, 1, 1000
    news = synth.news_table(N, L=L, seed=1)
    hist_idx, hmask, cand_idx, label = _long_impressions(B, N, H, K, seed=H)
    tables = synth.teacher_tables(N, M, 256, seed=3)
    history = torch.from_numpy(news[hist_idx].astype(np.int64))
    candidate = torch.from_numpy(news[cand_idx].astype(np.int64))
    th = [torch.from_numpy(t[hist_idx]) for t in tables]
    tc = [torch.from_numpy(t[cand_idx]) for t in tables]
    extra = dict(model="NRMS", n_heads=16) if model == "NRMS" else {}
    sd = synth.kd_model_state(layers, M, 5, noisy=True, **extra)
    for ulm in (False, True):
        case = f"{model}.H{H}.ulm{int(ulm)}"
        args = synth.demo_args(num_student_layers=layers, num_teachers=M, user_log_length=H, model=model, user_log_mask=ulm)
        m = mb.Model(args)
        m.load_state_dict(sd, strict=True)
        m.cuda().eval()
        _apply_freeze(m, [0])
        res = m(history.cuda(), torch.from_numpy(hmask).cuda(), candidate.cuda(), torch.from_numpy(label).cuda(),
                [t.cuda() for t in th], [t.cuda() for t in tc])
        res[0].backward()
        osd = {k: v.clone() for k, v in sd.items()}
        names = [k for k, p in m.named_parameters() if p.requires_grad]
        for k in names:
            osd[k].requires_grad_(True)
        ref = om.kd_model_forward(osd, history, torch.from_numpy(hmask), candidate, torch.from_numpy(label), th, tc,
                                  layers, ulm, args.temperature, args.coef)
        ref[0].backward()
        for v, r, nm in zip(res[:4], ref[:4], ("total", "distill", "emb", "target")):
            assert abs(float(v) - float(r)) < 1e-2 * abs(float(r)) + 1e-4, (case, nm, float(v), float(r))
        _chk(f"long_kd.score.{case}", _rel(res[4], ref[4].detach()), SCORE_TOL)
        named = dict(m.named_parameters())
        for k in names:
            if osd[k].grad is None:                 # pad_doc in the user_log_mask branch
                assert float(named[k].grad.abs().max()) == 0.0, k
                continue
            _chk(f"long_kd.grad.{case}.{k}", _grad_err(k, named[k].grad, osd[k].grad, named), GRAD_TOL)


def test_model_bert_forward_long_history():
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    from oracle import model as om
    B, H, K, L, layers, N = 3, 150, 5, 12, 1, 1000
    news = synth.news_table(N, L=L, seed=4)
    hist_idx, hmask, cand_idx, _ = _long_impressions(B, N, H, K, seed=6)
    hmask[1] = 0.0                                  # an empty history
    history = torch.from_numpy(news[hist_idx].astype(np.int64))
    candidate = torch.from_numpy(news[cand_idx].astype(np.int64))
    sd = synth.model_bert_state("", layers, 7, noisy=True)
    for ulm in (False, True):
        m = mb.ModelBert(synth.demo_args(num_student_layers=layers, user_log_length=H, user_log_mask=ulm))
        m.load_state_dict(sd, strict=True)
        m.cuda().eval()
        with torch.no_grad():
            score, hv, cv, uv = m(history.cuda(), torch.from_numpy(hmask).cuda(), candidate.cuda())
            o_score, o_hv, o_cv, o_uv = om.model_bert_forward(sd, "", history, torch.from_numpy(hmask), candidate, layers, ulm)
        _chk(f"long_modelbert.user.ulm{int(ulm)}", _rel(uv, o_uv), SCORE_TOL)
        _chk(f"long_modelbert.score.ulm{int(ulm)}", _rel(score, o_score), SCORE_TOL)
        if ulm:
            assert float(uv[1].abs().max()) == 0.0


@pytest.mark.parametrize("ulm", [False, True])
@pytest.mark.parametrize("H", [100, 300])
def test_evaluate_long_history_vs_oracle_loop(H, ulm):
    """run.evaluate at long H against the reference's per-impression loop (run.py:335-379), in ragged batches that
    take both the scoring path (B >= 64) and the per-impression kernel (the last 44 impressions)."""
    import tinyrec.model_bert as mb
    import tinyrec.run as trun
    import tinyrec.synth as synth
    from oracle import metrics as omet, model as om
    from test_drivers_gpu import _eval_problem
    D = 256
    hist, hmask, ptr, cand, lab, kinds, table = _eval_problem(n_imp=300, H=H, D=D)
    n = hist.shape[0]
    args = synth.demo_args(user_log_mask=ulm, user_log_length=H)
    sd = synth.user_encoder_state("", D, args.user_query_vector_dim, 3)
    ue = mb.UserEncoder(args)
    ue.load_state_dict(sd, strict=True)
    ue.cuda().eval()
    tab_d = table.cuda()
    mean, total, per = trun.evaluate(ue, tab_d, hist, hmask, ptr, cand, lab, batch_size=128, return_per_impression=True)
    assert total == n
    per = per.cpu().numpy()
    with torch.no_grad():
        user = ue.forward_gather(tab_d, torch.from_numpy(hist).cuda(), torch.from_numpy(hmask).cuda())
        osd = {"user_encoder." + k: v for k, v in sd.items()}
        o_user = om.user_encoder(osd, "user_encoder.", table[torch.from_numpy(hist.astype(np.int64))], torch.from_numpy(hmask),
                                 ulm).numpy()
    _chk(f"long_evaluate.user_vec.H{H}.ulm{int(ulm)}", _rel(user, o_user), 1e-2)
    if ulm:
        assert float(user[5].abs().max()) == 0.0
    tab_np = table.numpy()
    o_per = []
    for i in range(n):
        seg = slice(int(ptr[i]), int(ptr[i + 1]))
        o_per.append(omet.impression_metrics(lab[seg], tab_np[cand[seg]] @ o_user[i]))
    keep = kinds != 3                                    # pos / neg ties: argsort order unspecified (test_drivers_gpu.py)
    o_mean_all, _ = omet.eval_reduce(o_per, n)
    o_mean, _ = omet.eval_reduce([m for m, k in zip(o_per, keep) if k], n)
    g_mean = per[keep, :4].sum(0) / n
    _chk(f"long_evaluate.mean_auc.H{H}.ulm{int(ulm)}", abs(float(mean[0]) - float(o_mean_all[0])), 1e-3)
    for j, nm in ((1, "mrr"), (2, "ndcg5"), (3, "ndcg10")):
        _chk(f"long_evaluate.mean_{nm}.H{H}.ulm{int(ulm)}", abs(float(g_mean[j]) - float(o_mean[j])), 1e-3)


def test_graphed_train_step_long_history_matches_eager_loop():
    """GraphedTrainStep at H = 100 against the eager loop on the same batches: the same losses step by step, and
    parameters within the spread of the split-K fp32 atomics (not bitwise)."""
    import tinyrec.model_bert as mb
    import tinyrec.optim as topt
    import tinyrec.run as trun
    import tinyrec.synth as synth
    B, H, K, L, M, layers, N = 4, 100, 3, 12, 2, 2, 600
    news = synth.news_table(N, L=L, seed=1)
    tables = synth.teacher_tables(N, M, 256, seed=3)
    batches = []
    for s in range(3):
        hist_idx, hmask, cand_idx, label = _long_impressions(B, N, H, K, seed=10 + s)
        batches.append((torch.from_numpy(news[hist_idx].astype(np.int64)).cuda(), torch.from_numpy(hmask).cuda(),
                        torch.from_numpy(news[cand_idx].astype(np.int64)).cuda(), torch.from_numpy(label).cuda(),
                        [torch.from_numpy(t[hist_idx]).cuda() for t in tables], [torch.from_numpy(t[cand_idx]).cuda() for t in tables]))
    sd = synth.kd_model_state(layers, M, 5, noisy=True)
    runs = []
    for graphed in (False, True):
        m = mb.Model(synth.demo_args(num_student_layers=layers, num_teachers=M, user_log_length=H))
        m.load_state_dict(sd, strict=True)
        m.cuda().eval()
        _apply_freeze(m, [1])
        opt = topt.Adam(m, lr=1e-4)
        losses = []
        if graphed:
            step = trun.GraphedTrainStep(m, opt, batches[0])
            for b in batches:
                losses.append(float(step(*b)[0]))
        else:
            for b in batches:
                opt.zero_grad()
                out = m(*b)
                out[0].backward()
                opt.step()
                losses.append(float(out[0]))
        runs.append((losses, {k: v.detach().clone() for k, v in m.named_parameters() if v.requires_grad}))
    (l0, p0), (l1, p1) = runs
    assert l0[0] != l0[1]
    for a, b in zip(l0, l1):
        assert abs(a - b) < 5e-3 * abs(a) + 1e-5, (l0, l1)
    for k in p0:
        if k.endswith(("key.bias", "att_fc2.bias")):
            continue
        assert _rel(p1[k], p0[k]) < 2e-3, k
