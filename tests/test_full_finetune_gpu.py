"""Full-encoder fine-tuning: the embedding block (word / position / token-type tables and embeddings.LayerNorm) and the
shared rel-pos bias table trained like every other parameter.

- tnr_embed_ln_bwd against a float64 autograd restatement of the forward (same bf16 dy and bf16 word rows): repeated
  ids, [CLS] / [SEP] in every row, an all-pad row, dropout on and off, accumulation into non-zero buffers, untouched
  rows exact, reruns bit-identical.
- tnr_attn_relpos_bwd_drel against float64 autograd over the bucket table, dqkv bit-identical to tnr_attn_relpos_bwd.
- The KD Model / DistillModel train steps against the CPU oracle with autograd, the fused-Adam update seen by the next
  forward, CUDA-graph replay and the dead pooler / classifier parameters.
Every measured error is recorded with conftest.report; bounds are about twice the worst value measured on a B200."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
P_DROP = 0.1
GRAD_TOL = 3e-2           # as tests/test_model_gpu.py: bf16 activations and activation gradients
GRAD_TOL_LONG = 6e-2      # 100-token rows
SCORE_TOL = 1e-2
EMB_TOL = 5e-7            # embedding backward, fp32 sums against float64: worst measured 2.4e-7 (dtype, L = 100)
DREL_TOL = 4e-4           # rel-pos bias table gradient, dS summed in fp32 before its bf16 staging: worst 1.8e-4 (L = 7);
                          # 1e-2 would be the bound for sums of the bf16-staged dS


def _chk(label, value, bound):
    from conftest import report
    report(label, float(value), float(bound))
    assert value < bound, (label, value, bound)


def _rel(got, ref):
    got = torch.as_tensor(got).double().cpu()
    ref = torch.as_tensor(ref).double().cpu()
    return float((got - ref).norm() / (ref.norm() + 1e-300))


def _ops():
    import tinyrec.ops as ops
    return ops


def _seed_tensor(seed):
    return torch.tensor([seed], device="cuda", dtype=torch.int64)


def _diag_buckets(L):
    from tinyrec.engine import rel_pos_bucket_table
    tab = rel_pos_bucket_table(L)
    return torch.cat([tab[1:, 0].flip(0), tab[0, :]])


# ------------------------------------------------------------------ embedding backward
def _embed_ids(n, L, vocab, g):
    """[CLS] ... [SEP] rows of random ids drawn from a small pool (repeats), pad tails, row 1 all pad."""
    ids = torch.zeros(n, L, dtype=torch.int64)
    lens = torch.randint(1, L + 1, (n,), generator=g)
    lens[0] = L
    for r in range(n):
        k = int(lens[r])
        row = torch.randint(103, min(vocab, 400), (k,), generator=g)
        row[0] = 101
        if k > 1:
            row[k - 1] = 102
        ids[r, :k] = row
    ids[1] = 0
    mask = (ids != 0).long()
    return torch.cat([ids, mask], 1)


@pytest.mark.parametrize("L", [1, 7, 30, 100])
@pytest.mark.parametrize("dropout", [False, True])
def test_embed_ln_bwd_vs_float64(L, dropout):
    ops = _ops()
    E, vocab, maxpos = 768, 1000, 512
    n = 80 if L <= 30 else 24
    g = torch.Generator().manual_seed(L + 7 * dropout)
    x = _embed_ids(n, L, vocab, g).cuda()
    word = (torch.randn(vocab, E, generator=g) * 0.5).to(BF).cuda()
    pos = (torch.randn(maxpos, E, generator=g) * 0.3).cuda()
    typ = (torch.randn(2, E, generator=g) * 0.3).cuda()
    gamma = (1 + 0.1 * torch.randn(E, generator=g)).cuda()
    beta = (0.1 * torch.randn(E, generator=g)).cuda()
    dy = torch.randn(n * L, E, generator=g).to(BF).cuda()
    seed = _seed_tensor(4242)
    drop = ops.make_drop(seed, 0, P_DROP) if dropout else None
    # non-zero starting buffers: the kernel accumulates
    init = dict(dword=torch.randn(vocab, E, generator=g).cuda(), dpos=torch.randn(maxpos, E, generator=g).cuda(),
                dtype=torch.randn(2, E, generator=g).cuda(), dgamma=torch.randn(E, generator=g).cuda(),
                dbeta=torch.randn(E, generator=g).cuda())

    def run():
        b = {k: v.clone() for k, v in init.items()}
        ops.embed_ln_bwd(x, L, word, pos, typ[0], gamma, 1e-12, dy, dword=b["dword"], dpos=b["dpos"], dtype0=b["dtype"][0],
                         dgamma=b["dgamma"], dbeta=b["dbeta"], drop=drop)
        return b

    got = run()
    again = run()
    for k in got:
        assert torch.equal(got[k], again[k]), k                    # bit-identical rerun
    # float64 reference from the same bf16 word rows and bf16 dy
    ids = x[:, :L]
    w64 = word.double().requires_grad_(True)
    p64 = pos.double().requires_grad_(True)
    t64 = typ.double().requires_grad_(True)
    g64, b64 = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    h = w64[ids] + p64[:L][None] + t64[0]
    y = torch.nn.functional.layer_norm(h, (E,), g64, b64, 1e-12).reshape(n * L, E)
    if dropout:
        keep = ops.dropout_mask(drop, n * L * E, "cuda").reshape(n * L, E).double()
        y = y * keep / (1.0 - P_DROP)
    (y * dy.double()).sum().backward()
    ref_word = w64.grad.clone()
    ref_word[0] = 0                                                # padding_idx = 0
    tag = f"L{L}_{'drop' if dropout else 'nodrop'}"
    d = {k: got[k].double() - init[k].double() for k in got}
    _chk(f"test_embed_ln_bwd_vs_float64.dword.{tag}", _rel(d["dword"], ref_word), EMB_TOL)
    _chk(f"test_embed_ln_bwd_vs_float64.dpos.{tag}", _rel(d["dpos"][:L], p64.grad[:L]), EMB_TOL)
    _chk(f"test_embed_ln_bwd_vs_float64.dtype.{tag}", _rel(d["dtype"][0], t64.grad[0]), EMB_TOL)
    _chk(f"test_embed_ln_bwd_vs_float64.dgamma.{tag}", _rel(d["dgamma"], g64.grad), EMB_TOL)
    _chk(f"test_embed_ln_bwd_vs_float64.dbeta.{tag}", _rel(d["dbeta"], b64.grad), EMB_TOL)
    # untouched rows stay bit-exact: row 0, ids that never occur, positions >= L, token type 1
    seen = torch.zeros(vocab, dtype=torch.bool)
    seen[ids.reshape(-1).cpu()] = True
    seen[0] = False
    assert torch.equal(got["dword"][~seen.cuda()], init["dword"][~seen.cuda()])
    assert torch.equal(got["dpos"][L:], init["dpos"][L:])
    assert torch.equal(got["dtype"][1], init["dtype"][1])
    assert bool(seen[101]) and (L == 1 or bool(seen[102]))


# ------------------------------------------------------------------ rel-pos bias gradient of the attention backward
def _drop_keep(ops, qkv, x, L, A, n, drop):
    """[n, A, L, L] keep flags of the attention dropout, read out of the forward: V rows one-hot within a 64-key block
    make ctx[i, c] = dropout(P)[i, 64 b + c]."""
    E = A * 64
    keep = torch.zeros(n, A, L, L, dtype=torch.bool, device="cuda")
    relz = torch.zeros(A, 2 * L - 1, device="cuda")
    for b in range((L + 63) // 64):
        probe = qkv.clone()
        v = torch.zeros(L, A, 64, device="cuda")
        r = torch.arange(64 * b, min(L, 64 * b + 64), device="cuda")
        v[r, :, r - 64 * b] = 1.0
        probe[:, 2 * E:] = v.reshape(1, L, E).expand(n, L, E).reshape(n * L, E).to(BF)
        ctx = torch.empty(n * L, E, device="cuda", dtype=BF)
        ops.attn_fwd(probe, x, L, relz, ctx, A, drop=drop)
        blk = ctx.float().reshape(n, L, A, 64)[..., :len(r)].permute(0, 2, 1, 3)
        keep[..., 64 * b:64 * b + len(r)] = blk != 0
    return keep


@pytest.mark.parametrize("L", [1, 7, 30, 32, 33, 100, 512])
@pytest.mark.parametrize("dropout", [False, True])
def test_attn_bwd_drel_vs_float64(L, dropout):
    ops = _ops()
    n, A = (5, 4) if L <= 100 else (2, 4)
    E, NB = A * 64, 32
    g = torch.Generator().manual_seed(100 + L + dropout)
    qkv = (torch.randn(n * L, 3 * E, generator=g) * 0.5).to(BF).cuda()
    lens = torch.randint(1, L + 1, (n,), generator=g)
    lens[0] = L
    mask = (torch.arange(L)[None, :] < lens[:, None]).long()
    if n > 2:
        mask[2] = 0                                                # all-pad news
    mask = mask.cuda()
    x = torch.cat([torch.zeros_like(mask), mask], 1)
    table = (torch.randn(A, NB, generator=g) * 0.5).cuda()
    bvec = _diag_buckets(L).cuda()
    relpos = table[:, bvec].contiguous()
    bucket = bvec.to(torch.int32)
    dctx = torch.randn(n * L, E, generator=g).to(BF).cuda()
    seed = _seed_tensor(99)
    drop = ops.make_drop(seed, 13, P_DROP) if dropout else None
    dq_ref = torch.empty_like(qkv)
    ops.attn_bwd(qkv, x, L, relpos, dctx, dq_ref, A, drop=drop)
    init = torch.randn(A, NB, generator=g).cuda()
    outs = []
    for _ in range(2):
        dqkv = torch.empty_like(qkv)
        drel = init.clone()
        ops.attn_bwd_drel(qkv, x, L, relpos, dctx, dqkv, A, bucket, drel, drop=drop)
        outs.append((dqkv, drel))
    assert torch.equal(outs[0][0], dq_ref)                         # dqkv bit-identical to tnr_attn_relpos_bwd
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    # float64 autograd over the bucket table
    t64 = table.double().requires_grad_(True)
    q, k, v = [t.reshape(n, L, A, 64).permute(0, 2, 1, 3) for t in qkv.double().split(E, dim=1)]
    idx = torch.arange(L, device="cuda")
    rel = t64[:, bvec][:, (idx[None, :] - idx[:, None]) + L - 1]          # [A, L, L]
    sc = q @ k.transpose(-1, -2) / 8.0 + (1.0 - mask.double())[:, None, None, :] * -10000.0 + rel[None]
    pr = torch.softmax(sc, -1)
    if dropout:
        keep = _drop_keep(ops, qkv, x, L, A, n, drop)
        keep = keep | (pr.detach() < 1e-30)                        # an exactly-zero probability reads as "dropped"
        pr = pr * keep / (1.0 - P_DROP)
    ctx = (pr @ v).permute(0, 2, 1, 3).reshape(n * L, E)
    (ctx * dctx.double()).sum().backward()
    if L == 1:
        # one key: the softmax is constant and its score gradient zero; both sides hold rounding noise (the kernel's
        # probability is 1 to an ulp), measured against the size of the dP = dO . V it is formed from
        scale = float((dctx.double().reshape(n, A, 64) * v.reshape(n, A, 64)).abs().sum())
        _chk("test_attn_bwd_drel_vs_float64.drel_noise_over_dP.L1_" + ("drop" if dropout else "nodrop"),
             float((outs[0][1].double() - init.double()).abs().max()) / scale, 5e-9)     # worst measured 2.4e-9
        assert float(t64.grad.abs().max()) < 1e-12 * scale
        return
    err = _rel(outs[0][1].double() - init.double(), t64.grad)
    _chk(f"test_attn_bwd_drel_vs_float64.drel.L{L}_{'drop' if dropout else 'nodrop'}", err, DREL_TOL)


# ------------------------------------------------------------------ model level against the CPU oracle
def _set_trainable(m, student_ne, what, layers):
    """what: 'all' (the whole student encoder, PyTorch's default flags), 'bottom' (embedding block + rel_pos_bias, all
    layers frozen), 'rel' (rel_pos_bias only); the pooling head / dense / user encoder / transform train as in run.py."""
    if hasattr(m, "teachers"):
        for p in m.teachers.parameters():
            p.requires_grad = False
    bm = student_ne.bert_model
    for p in bm.parameters():
        p.requires_grad = what == "all"
    if what == "bottom":
        for p in bm.bert.embeddings.parameters():
            p.requires_grad = True
    if what in ("bottom", "rel"):
        bm.bert.rel_pos_bias.weight.requires_grad = True


def _dead_names(named):
    return [k for k in named if ".bert.pooler." in k or ".bert_model.classifier." in k]


def _compare_grads(label, m, osd, tol):
    named = dict(m.named_parameters())
    dead = set(_dead_names(named))
    names = [k for k, p in named.items() if p.requires_grad and k not in dead]
    word = [k for k in names if k.endswith("word_embeddings.weight")]
    for k in word:
        osd[k].grad[0] = 0                                         # nn.Embedding(padding_idx=0)
        assert float(named[k].grad[0].abs().max()) == 0.0
    for k in dead:
        assert named[k].grad is None, k
    for k in names:
        gref, got = osd[k].grad, named[k].grad
        if k.endswith("attention.self.key.bias"):                  # identically zero: against the query-bias scale
            err = float((got.double().cpu() - gref.double()).norm() / (osd[k.replace("key.bias", "query.bias")].grad.double().norm()))
        elif k.endswith("attn.att_fc2.bias"):                      # shift invariant as well
            err = float((got.double().cpu() - gref.double()).norm() / (osd[k.replace("att_fc2.bias", "att_fc2.weight")].grad.double().norm()))
        else:
            err = _rel(got, gref)
        _chk(f"{label}.grad.{k}", err, tol)
    return names


def _kd_inputs(B, H, K, L, M, N, seeds=(3, 4, 5)):
    import tinyrec.synth as synth
    news = synth.news_table(N, L=L, seed=seeds[0])
    hist_idx, hmask, cand_idx, label = synth.train_impressions(B, N, H, K, seed=seeds[1])
    tables = synth.teacher_tables(N, M, 256, seed=seeds[2])
    history = torch.from_numpy(news[hist_idx].astype(np.int64))
    candidate = torch.from_numpy(news[cand_idx].astype(np.int64))
    th = [torch.from_numpy(t[hist_idx]) for t in tables]
    tc = [torch.from_numpy(t[cand_idx]) for t in tables]
    return history, torch.from_numpy(hmask), candidate, torch.from_numpy(label), th, tc


def _kd_case(what, B, H, K, L, M, N, layers, tol, label, train_mode=False):
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    from oracle import model as om
    history, hmask, candidate, lab, th, tc = _kd_inputs(B, H, K, L, M, N)
    sd = synth.kd_model_state(layers, M, 11, noisy=True)
    args = synth.demo_args(num_student_layers=layers, num_teachers=M, user_log_length=H)
    m = mb.Model(args)
    m.load_state_dict(sd, strict=True)
    m.cuda().eval()
    _set_trainable(m, m.student.news_encoder, what, layers)
    gpu_in = (history.cuda(), hmask.cuda(), candidate.cuda(), lab.cuda(), [t.cuda() for t in th], [t.cuda() for t in tc])
    res = m(*gpu_in)
    res[0].backward()
    st = m.train_state()
    osd = {k: v.clone() for k, v in sd.items()}
    named = dict(m.named_parameters())
    for k, p in named.items():
        if p.requires_grad:
            osd[k].requires_grad_(True)
    ref = om.kd_model_forward(osd, history, hmask, candidate, lab, th, tc, layers, False, args.temperature, args.coef)
    ref[0].backward()
    for v, r, nm in zip(res[:4], ref[:4], ("total", "distill", "emb", "target")):
        assert abs(float(v) - float(r)) < 1e-2 * abs(float(r)) + 1e-4, (nm, float(v), float(r))
    _chk(f"{label}.score", _rel(res[4], ref[4].detach()), SCORE_TOL)
    _compare_grads(label, m, osd, tol)
    return m, st, gpu_in


@pytest.mark.parametrize("what", ["all", "bottom", "rel"])
def test_kd_step_full_finetune_vs_oracle(what):
    """KD Model, 2 layers, B 4, H 50, K 5, L 30, M 4."""
    m, st, gpu_in = _kd_case(what, 4, 50, 5, 30, 4, 500, 2, GRAD_TOL, f"test_kd_step_full_finetune_vs_oracle.{what}")
    if what == "all":
        # dead parameters: accepted, grad stays None, and the train state is not rebuilt by the next call
        named = dict(m.named_parameters())
        dead = _dead_names(named)
        assert dead and all(named[k].requires_grad for k in dead)
        m(*gpu_in)[0].backward()
        assert m.train_state() is st
        assert all(named[k].grad is None for k in dead)


def test_kd_step_full_finetune_long_rows_vs_oracle():
    _kd_case("all", 2, 4, 3, 100, 2, 120, 2, GRAD_TOL_LONG, "test_kd_step_full_finetune_long_rows_vs_oracle")


def test_distill_model_full_finetune_vs_oracle():
    """Two saved passes per step (12-token titles, a 72-token body) accumulating into one gradient."""
    from types import SimpleNamespace
    import tinyrec.post_train as pt
    import tinyrec.synth as synth
    from oracle import model as om
    B, K1, Lt, Lb, M, layers, D = 3, 4, 12, 72, 2, 2, 256
    rng = np.random.default_rng(5)
    title = torch.from_numpy(synth.news_table(B * K1 - 1, L=Lt, seed=1).astype(np.int64)).reshape(B, K1, 2 * Lt)
    body = torch.from_numpy(synth.news_table(B - 1, L=Lb, seed=2).astype(np.int64))
    labels = torch.tensor([0, 2, 1])
    tt = [torch.from_numpy(rng.standard_normal((B, K1, D)).astype(np.float32) * 0.3) for _ in range(M)]
    tb = [torch.from_numpy(rng.standard_normal((B, D)).astype(np.float32) * 0.3) for _ in range(M)]
    args = SimpleNamespace(news_query_vector_dim=200, news_dim=D, num_hidden_layers=layers, num_teachers=M)
    m = pt.DistillModel(args)
    full = synth.kd_model_state(layers, M, 7, noisy=True)
    sd = {k: v for k, v in full.items() if k.startswith(("student.news_encoder.", "transform_matrix."))}
    m.load_state_dict(sd, strict=True)
    m.cuda().eval()
    _set_trainable(m, m.student.news_encoder, "all", layers)
    res = m(title.cuda(), body.cuda(), labels.cuda(), [t.cuda() for t in tt], [t.cuda() for t in tb])
    res[0].backward()
    osd = {k: v.clone() for k, v in sd.items()}
    for k, p in m.named_parameters():
        if p.requires_grad:
            osd[k].requires_grad_(True)
    ref = om.post_train_distill_forward(osd, title, body, labels, tt, tb, layers)
    ref[0].backward()
    for got, want in zip(res[:4], ref[:4]):
        assert abs(float(got) - float(want)) < 1e-2 * abs(float(want)) + 1e-4, (float(got), float(want))
    _chk("test_distill_model_full_finetune_vs_oracle.score", _rel(res[4], ref[4].detach()), SCORE_TOL)
    _compare_grads("test_distill_model_full_finetune_vs_oracle", m, osd, GRAD_TOL)


def test_forward_follows_fused_adam_update():
    """After a fused-Adam step the next forward reads the updated word table (bf16 shadow) and rel-pos table (gathered
    on the device every forward): it matches a fresh model loaded with the updated state_dict."""
    import tinyrec.model_bert as mb
    import tinyrec.optim as topt
    import tinyrec.synth as synth
    B, H, K, L, M, N, layers = 4, 10, 3, 12, 2, 300, 2
    history, hmask, candidate, lab, th, tc = _kd_inputs(B, H, K, L, M, N, seeds=(1, 2, 3))
    gpu_in = (history.cuda(), hmask.cuda(), candidate.cuda(), lab.cuda(), [t.cuda() for t in th], [t.cuda() for t in tc])
    sd = synth.kd_model_state(layers, M, 5, noisy=True)
    args = synth.demo_args(num_student_layers=layers, num_teachers=M, user_log_length=H)

    def fresh(state):
        m = mb.Model(args)
        m.load_state_dict(state, strict=True)
        m.cuda().eval()
        _set_trainable(m, m.student.news_encoder, "bottom", layers)
        return m

    m = fresh(sd)
    opt = topt.Adam(m, lr=1e-2)
    with torch.no_grad():
        s0 = m(*gpu_in)[4].clone()
    opt.zero_grad()
    m(*gpu_in)[0].backward()
    opt.step()
    with torch.no_grad():
        s1 = m(*gpu_in)[4].clone()
        s2 = fresh({k: v.detach().cpu().clone() for k, v in m.state_dict().items()})(*gpu_in)[4]
    moved = _rel(s1, s0)
    assert moved > 1e-3, moved                                   # the step changed the scores
    _chk("test_forward_follows_fused_adam_update.score_vs_fresh_model", _rel(s1, s2), 1e-5)


def test_graphed_train_step_full_finetune_matches_eager_loop():
    """GraphedTrainStep with everything in the student encoder trainable against the eager loop, step by step."""
    import tinyrec.model_bert as mb
    import tinyrec.optim as topt
    import tinyrec.run as trun
    import tinyrec.synth as synth
    B, H, K, L, M, layers, N = 4, 10, 3, 12, 2, 2, 300
    news = synth.news_table(N, L=L, seed=1)
    tables = synth.teacher_tables(N, M, 256, seed=3)
    batches = []
    for s in range(3):
        hist_idx, hmask, cand_idx, label = synth.train_impressions(B, N, H, K, seed=10 + s)
        batches.append((torch.from_numpy(news[hist_idx].astype(np.int64)).cuda(), torch.from_numpy(hmask).cuda(),
                        torch.from_numpy(news[cand_idx].astype(np.int64)).cuda(), torch.from_numpy(label).cuda(),
                        [torch.from_numpy(t[hist_idx]).cuda() for t in tables], [torch.from_numpy(t[cand_idx]).cuda() for t in tables]))
    sd = synth.kd_model_state(layers, M, 5, noisy=True)
    runs = []
    for graphed in (False, True):
        m = mb.Model(synth.demo_args(num_student_layers=layers, num_teachers=M, user_log_length=H))
        m.load_state_dict(sd, strict=True)
        m.cuda().eval()
        _set_trainable(m, m.student.news_encoder, "all", layers)
        opt = topt.Adam(m, lr=1e-4)
        losses = []
        if graphed:
            step = trun.GraphedTrainStep(m, opt, batches[0])
            for b in batches:
                losses.append(float(step(*b)[0]))
            assert opt.steps_done() == len(batches)
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
        if k.endswith(("key.bias", "att_fc2.bias")) or ".bert.pooler." in k or ".classifier." in k:
            continue
        _chk(f"test_graphed_train_step_full_finetune_matches_eager_loop.param.{k}", _rel(p1[k], p0[k]), 2e-3)
