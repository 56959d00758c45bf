"""Direct tests of the fp32 head kernels against float64 restatements of the same operations: the click-score / CE /
multi-teacher KD loss head (tnr_kd_loss_fwdbwd) and the eval scoring and ranking kernels (tnr_eval_metrics), at the
shapes and edges the whole-model tests do not reach -- batches of more than 32 impressions, the M = 8 / K = 32 limits
of the loss head's shared arrays, K = 1, D not a multiple of 32, empty impressions inside a CSR batch, every
instantiated D and the shared-memory fallbacks of the rank kernel.

Every measured error goes to the test report (tests/conftest.py: report); each bound is about twice the worst value
measured on a B200."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import metrics as omet, model as om

F64 = torch.float64
DEV = "cuda"


def _ops():
    import tinyrec.ops as ops
    return ops


def _chk(label, value, bound):
    """assert value < bound, recording the measured value in the test report."""
    from conftest import report
    report(label, float(value), float(bound))
    assert value < bound, (label, value, bound)


def _group_rel(got, ref):
    """Error in norm of each leading-index group (one impression) of ``got`` against ``ref``, relative to the group's
    own norm -- an error a swapped or skipped row cannot hide in, as it would in one global norm.  The denominator is
    floored at a tenth of the median group norm: an impression whose loss or gradient nearly cancels in exact
    arithmetic (a saturated softmax, distillation and CE pulling against each other) is judged on the scale of its
    batch, not on its fp32 rounding noise.  Absolute where the reference is zero throughout."""
    got = got.detach().to(F64).reshape(got.shape[0], -1)
    ref = ref.detach().to(F64).reshape(ref.shape[0], -1)
    err = (got - ref).norm(dim=1)
    den = ref.norm(dim=1)
    den = torch.maximum(den, 0.1 * den.median())
    return torch.where(den > 0, err / den.clamp_min(1e-300), err)


def _bits(t):
    return t.contiguous().view(torch.int32)


# ------------------------------------------------------------------------------------------------ KD loss head
def _kd_head_ref(s_news, s_user, label, T_ext, TP_ext, M, B, H, K, D, tau, coef):
    """Model.forward from the encoder outputs on (oracle/model.py: kd_model_forward, the reference's
    model_bert.py:262-306), term by term, on the loss head's row layout (include/tinyrec.h): s_news [R, D] with
    R = B*(H+K), history row (b, h) at b*H + h and candidate row (b, k) at B*H + b*K + k; s_user [B, D]; T_ext / TP_ext
    [M, R + B, D], the raw / transformed teacher vectors in the same layout with teacher user vector b at row R + b.
    Returns the scores [B, K], the batch losses distill / emb / target / total and ``per`` [B, 4], the
    (distill, emb, target, total) terms of each impression."""
    R = B * (H + K)
    s_hist = s_news[:B * H].reshape(B, H, D)
    s_cand = s_news[B * H:R].reshape(B, K, D)
    score = torch.bmm(s_cand, s_user.unsqueeze(-1)).squeeze(-1)
    target = F.cross_entropy(score, label)                                               # :271
    target_b = F.cross_entropy(score, label, reduction="none")
    distill = emb = score.new_zeros(())
    distill_b = emb_b = score.new_zeros(B)
    if M > 0:
        s_cat = torch.cat([s_hist, s_cand], dim=1)
        t_scores, t_losses, ne, ue = [], [], [], []
        for i in range(M):
            t_news = torch.cat([TP_ext[i, :B * H].reshape(B, H, D), TP_ext[i, B * H:R].reshape(B, K, D)], dim=1)
            ne.append(((s_cat - t_news) ** 2).mean(-1).mean(-1))                     # :279-280
            ue.append(((s_user - TP_ext[i, R:]) ** 2).mean(-1))                      # :283-284
            sc = torch.bmm(T_ext[i, B * H:R].reshape(B, K, D), T_ext[i, R:].unsqueeze(-1)).squeeze(-1)   # :286-287
            t_scores.append(sc)
            t_losses.append(F.cross_entropy(sc, label, reduction="none"))             # :288
        w = torch.softmax(-torch.stack(t_losses, -1), dim=-1)                          # :292-293
        t_score = torch.bmm(torch.stack(t_scores, -1), w.unsqueeze(-1)).squeeze(-1)   # :295-297
        distill = om.kd_ce_loss(score, t_score, tau)                                   # :298
        distill_b = torch.stack([om.kd_ce_loss(score[b:b + 1], t_score[b:b + 1], tau) for b in range(B)])
        ne_w, ue_w = (torch.stack(ne, -1) * w).sum(-1), (torch.stack(ue, -1) * w).sum(-1)
        emb = ne_w.mean() + ue_w.mean()                                                # :300-303
        emb_b = ne_w + ue_w
    total = distill + coef * target + emb                                              # :305
    per = torch.stack([distill_b, emb_b, target_b, distill_b + coef * target_b + emb_b], -1)
    return dict(score=score, distill=distill, emb=emb, target=target, total=total, per=per)


def test_kd_head_ref_matches_reference_golden(golden):
    """The reference above, fed with the oracle's encoder outputs laid out as the kernel expects, reproduces the real
    reference model's losses and scores (tests/golden/kd.npz): this pins the row layout conventions of the GPU tests
    below.  CPU only."""
    import tinyrec.synth as synth
    g = golden("kd")
    layers, M = int(g["layers"]), int(g["M"])
    tau, coef = float(g["temperature"]), float(g["coef"])
    sd = synth.kd_model_state(layers, M, int(g["seed"]), noisy=True)
    history, hmask = torch.from_numpy(g["history"]), torch.from_numpy(g["history_mask"])
    candidate, label = torch.from_numpy(g["candidate"]), torch.from_numpy(g["label"])
    th = [torch.from_numpy(g[f"th{i}"]) for i in range(M)]
    tc = [torch.from_numpy(g[f"tc{i}"]) for i in range(M)]
    B, H, K, D = history.shape[0], history.shape[1], candidate.shape[1], th[0].shape[-1]
    threads = torch.get_num_threads()
    torch.set_num_threads(8)            # the thread count the fixture was recorded with (tests/test_oracle_golden.py)
    try:
        for tag, ulm in (("pad", False), ("mask", True)):
            with torch.no_grad():
                _, s_hist, s_cand, s_user = om.model_bert_forward(sd, "student.", history, hmask, candidate, layers, ulm)
                t_user = [om.user_encoder(sd, f"teachers.{i}.", th[i], hmask, ulm) for i in range(M)]
                s_news = torch.cat([s_hist.reshape(B * H, D), s_cand.reshape(B * K, D)])
                T = torch.stack([torch.cat([th[i].reshape(B * H, D), tc[i].reshape(B * K, D), t_user[i]]) for i in range(M)])
                TP = torch.stack([F.linear(T[i], sd[f"transform_matrix.{i}.weight"], sd[f"transform_matrix.{i}.bias"])
                                  for i in range(M)])
            ref = _kd_head_ref(s_news.double(), s_user.double(), label, T.double(), TP.double(), M, B, H, K, D, tau, coef)
            for nm in ("total", "distill", "emb", "target"):
                np.testing.assert_allclose(float(ref[nm]), float(g[f"{nm}_{tag}"]), rtol=2e-5, err_msg=f"{nm}_{tag}")
            np.testing.assert_allclose(ref["score"].numpy(), g[f"score_{tag}"], rtol=2e-5, err_msg=f"score_{tag}")
            batch = torch.stack([ref[nm] for nm in ("distill", "emb", "target", "total")])
            np.testing.assert_allclose(ref["per"].mean(0).numpy(), batch.numpy(), rtol=1e-12)
    finally:
        torch.set_num_threads(threads)


def _kd_problem(M, B, H, K, D, big, seed):
    """Student and teacher vectors in the kernel's layout, float64 on the host.  Candidate rows are built so that
    their scores are level + spread * N(0, 1) (level 10..60 as behind a trained 12-layer encoder, or 200..400 with
    ``big``) plus a component orthogonal to the user vector; the teacher projections sit near the student vectors
    (MSE ~0.1), so the CE, distillation and embedding terms all carry weight.  With ``big`` the teacher scores spread
    by ~60, so the teacher CE losses exceed what exp(-loss) can hold in fp32 and only the min-subtracted weights
    stay finite."""
    g = torch.Generator().manual_seed(seed)

    def rn(*shape):
        return torch.randn(*shape, generator=g, dtype=F64)

    lo, hi, s_spread, t_spread = (200.0, 400.0, 8.0, 60.0) if big else (10.0, 60.0, 2.0, 2.0)

    def cands(user, spread):
        want = lo + (hi - lo) * torch.rand(B, 1, generator=g, dtype=F64) + spread * rn(B, K)
        u = user / (user * user).sum(-1, keepdim=True)
        noise = rn(B, K, D)
        noise = noise - (noise * user[:, None]).sum(-1, keepdim=True) * u[:, None]
        return want[..., None] * u[:, None] + noise

    R = B * (H + K)
    s_user = rn(B, D)
    s_news = torch.cat([rn(B * H, D), cands(s_user, s_spread).reshape(B * K, D)])
    label = torch.randint(0, K, (B,), generator=g)
    T = TP = None
    if M > 0:
        T = torch.empty(M, R + B, D, dtype=F64)
        for i in range(M):
            t_user = rn(B, D)
            T[i] = torch.cat([rn(B * H, D), cands(t_user, t_spread).reshape(B * K, D), t_user])
        TP = torch.cat([s_news, s_user]).unsqueeze(0) + 0.3 * rn(M, R + B, D)
    return s_news, s_user, label, T, TP


# (M, B, H, K, D, tau, coef, big, tol): tol bounds the per-impression losses and all gradients.  It is larger where
# softmaxes saturate -- two candidates, or scores in the hundreds: a CE, distillation or gradient term that nearly
# cancels is judged against a tenth of its batch's median, and what it then shows is the fp32 spacing of the scores
# it comes from (4e-6 at 60, 3e-5 at 300).
KD_CASES = [
    (0, 5, 50, 5, 256, 1.0, 1.0, False, 6e-6),       # PLM-NR: CE only, with gradients
    (4, 32, 50, 5, 256, 1.0, 0.2, False, 2e-5),      # the benchmark step
    (8, 33, 50, 32, 256, 0.5, 0.2, False, 1.5e-5),   # M and K at the shared-array limits; B > 32
    (3, 70, 0, 8, 256, 1.0, 1.0, False, 1.5e-5),     # post-training layout (H = 0); three impressions per reducing lane
    (2, 1, 1, 1, 100, 4.0, 0.3, False, 1e-7),        # K = 1, B = 1, D not a multiple of 32
    (5, 40, 64, 2, 64, 2.0, 0.2, False, 1.1e-4),     # small D
    (4, 36, 20, 6, 128, 1.0, 0.2, True, 6e-4),       # scores in the hundreds
]


@pytest.mark.gpu
@pytest.mark.parametrize("M,B,H,K,D,tau,coef,big,tol", KD_CASES)
def test_kd_loss_vs_float64_reference(M, B, H, K, D, tau, coef, big, tol):
    ops = _ops()
    case = f"M{M}_B{B}_H{H}_K{K}_D{D}" + ("_big" if big else "")
    s_news, s_user, label, T, TP = _kd_problem(M, B, H, K, D, big, seed=100 + M * 7 + B)
    R = B * (H + K)
    nan = float("nan")
    s_news_d, s_user_d, label_d = s_news.float().to(DEV), s_user.float().to(DEV), label.to(DEV)
    T_d = T.float().to(DEV) if M else None
    TP_d = TP.float().to(DEV) if M else None

    def launch(want_grad):
        score = torch.full((B, K), nan, device=DEV)
        losses = torch.full((4 + 4 * B + 1,), 7.0, device=DEV)          # the kernel assigns, it does not accumulate
        losses[-1] = 0.0                                                # the ticket word starts at zero
        d_news = torch.full((R, D), nan, device=DEV)
        d_user = torch.full((B, D), nan, device=DEV)
        G = torch.full((M, R + B, D), nan, device=DEV) if M else None
        ops.kd_loss(s_news_d, s_user_d, label_d, T_d, TP_d, M, B, H, K, D, tau, coef, want_grad, score, losses,
                    d_news, d_user, G)
        return score, losses, d_news, d_user, G

    score, losses, d_news, d_user, G = launch(True)
    torch.cuda.synchronize()

    # float64 reference on the fp32 inputs the kernel saw, gradients by autograd of the total loss
    sn = s_news_d.to(F64).requires_grad_(True)
    su = s_user_d.to(F64).requires_grad_(True)
    tp = TP_d.to(F64).requires_grad_(True) if M else None
    ref = _kd_head_ref(sn, su, label_d, T_d.to(F64) if M else None, tp, M, B, H, K, D, tau, coef)
    ref["total"].backward()

    _chk(f"kd.score.{case}", float(_group_rel(score, ref["score"]).max()), 3e-7)
    got_batch = losses[:4].to(F64)
    ref_batch = torch.stack([ref[nm] for nm in ("distill", "emb", "target", "total")]).detach()
    _chk(f"kd.batch_losses.{case}", float(_group_rel(got_batch.reshape(4, 1), ref_batch.reshape(4, 1)).max()), 8e-7)
    got_per = losses[4:4 + 4 * B].reshape(B, 4)
    per_err = max(float(_group_rel(got_per[:, c:c + 1], ref["per"][:, c:c + 1]).max()) for c in range(4))
    _chk(f"kd.impression_losses.{case}", per_err, tol)
    assert int(_bits(losses[4 + 4 * B:])[0]) == 0, "ticket word not reset"

    hist_rows = (torch.arange(B)[:, None] * H + torch.arange(H)[None, :]).to(DEV)             # [B, H]
    cand_rows = (B * H + torch.arange(B)[:, None] * K + torch.arange(K)[None, :]).to(DEV)     # [B, K]
    _chk(f"kd.d_news_hist.{case}", float(_group_rel(d_news[hist_rows], sn.grad[hist_rows]).max()) if H else 0.0, tol)
    _chk(f"kd.d_news_cand.{case}", float(_group_rel(d_news[cand_rows], sn.grad[cand_rows]).max()), tol)
    _chk(f"kd.d_user.{case}", float(_group_rel(d_user, su.grad).max()), tol)
    if M:
        # impression b's rows of all teachers together: a teacher whose weight underflows fp32 leaves a block that is
        # zero in the kernel and ~1e-40 in float64
        rows = torch.cat([hist_rows, cand_rows, R + torch.arange(B, device=DEV)[:, None]], 1)
        _chk(f"kd.G_ext.{case}", float(_group_rel(G[:, rows].transpose(0, 1), tp.grad[:, rows].transpose(0, 1)).max()), tol)

    # two more launches on the same buffers: bitwise the same outputs, the ticket back at zero after each
    first = [t.clone() for t in (score, losses, d_news, d_user) + ((G,) if M else ())]
    for _ in range(2):
        ops.kd_loss(s_news_d, s_user_d, label_d, T_d, TP_d, M, B, H, K, D, tau, coef, True, score, losses, d_news, d_user, G)
        torch.cuda.synchronize()
        assert int(_bits(losses[4 + 4 * B:])[0]) == 0, "ticket word not reset"
        for a, b in zip(first, (score, losses, d_news, d_user) + ((G,) if M else ())):
            assert torch.equal(_bits(a), _bits(b)), "repeat launch changed an output"

    # forward only: the gradient buffers stay untouched, scores and losses are those of the gradient run
    score0, losses0, d_news0, d_user0, G0 = launch(False)
    torch.cuda.synchronize()
    assert torch.equal(_bits(score0), _bits(first[0])) and torch.equal(_bits(losses0), _bits(first[1]))
    nan_bits = int(_bits(torch.tensor([nan]))[0])
    for t in (d_news0, d_user0) + ((G0,) if M else ()):
        assert bool((_bits(t) == nan_bits).all()), "want_grad = 0 wrote a gradient buffer"


@pytest.mark.gpu
def test_kd_loss_rejects_sizes_beyond_its_shared_arrays():
    """M > 8 teachers, K = 0 and K > 32 candidates are refused on the host; nothing is launched."""
    ops = _ops()
    from tinyrec._lib import TinyRecError
    for M, K in ((9, 5), (0, 0), (2, 33)):
        B, H, D = 2, 3, 64
        R = B * (H + K)
        s_news = torch.zeros(max(R, 1), D, device=DEV)
        s_user = torch.zeros(B, D, device=DEV)
        label = torch.zeros(B, dtype=torch.int64, device=DEV)
        T = torch.zeros(max(M, 1), R + B, D, device=DEV)
        score = torch.full((B, max(K, 1)), 3.0, device=DEV)
        losses = torch.zeros(4 + 4 * B + 1, device=DEV)
        with pytest.raises(TinyRecError):
            ops.kd_loss(s_news, s_user, label, T, T, M, B, H, K, D, 1.0, 1.0, True, score, losses,
                        torch.zeros_like(s_news), torch.zeros_like(s_user), torch.zeros_like(T))
        torch.cuda.synchronize()
        assert bool((score == 3.0).all()) and not bool(losses.any())


# ------------------------------------------------------------------------------------------------ eval metrics
def _eval_batch(D, big, seed):
    """A CSR batch of ~300 impressions: random candidate counts with 0 (twice in the middle of the index, once right
    after another), 1, 2, 3, 37, 65 and 301 among them; all-positive and all-negative impressions; impressions with
    more than 64 positives; out-of-range ids; the same news clicked and not clicked; with ``big`` one impression of
    that many candidates (~10 % positive: tens of positive rounds)."""
    rng = np.random.default_rng(seed)
    sizes = rng.integers(2, 80, size=300)
    for i, c in ((10, 0), (11, 1), (12, 2), (13, 3), (20, 37), (30, 65), (40, 301), (41, 200), (50, 20), (51, 20),
                 (60, 12), (70, 9), (150, 0), (151, 0)):
        sizes[i] = c
    if big:
        sizes[200] = big
    n_rows = max(4096, int(sizes.max()) + 1)
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    cand = np.concatenate([rng.choice(n_rows, size=c, replace=False) for c in sizes]).astype(np.int32)
    lab = (rng.random(int(ptr[-1])) < 0.15).astype(np.int8)

    def seg(i):
        return slice(int(ptr[i]), int(ptr[i + 1]))
    for i in range(len(sizes)):                      # mostly two-sided impressions; the planted ones below are not
        if sizes[i] >= 2 and lab[seg(i)].min() == lab[seg(i)].max():
            lab[ptr[i]], lab[ptr[i] + 1] = 1, 0
    lab[seg(13)] = [0, 1, 0]
    lab[seg(40)] = (rng.random(301) < 0.5)           # ~150 positives: five rounds of 32
    lab[seg(41)] = 1
    lab[seg(41)][::3] = 0                            # 133 positives
    lab[seg(50)] = 1                                 # all positive: skipped
    lab[seg(51)] = 0                                 # all negative: skipped
    p0 = int(ptr[60])
    cand[p0:p0 + 4] = [-1, n_rows, 2 ** 31 - 1, 0]   # unknown ids read row 0: four candidates that tie
    lab[p0:p0 + 4] = [1, 0, 0, 1]
    p0 = int(ptr[70])
    cand[p0 + 1] = cand[p0]                          # the same news once clicked, once not
    lab[p0:p0 + 2] = [1, 0]
    if big:
        lab[seg(200)] = rng.random(big) < 0.1
    return n_rows, ptr, cand, lab


# (D, candidates of the one large impression; 0 = none)
EVAL_CASES = [(32, 0), (64, 0), (128, 0), (256, 0), (512, 0),
              (256, 4544),                           # largest impression the rank kernel runs at 4 warps per block
              (256, 4545),                           # 2 warps per block
              (256, 22752)]                          # 1 warp per block, 199.97 KB of shared memory


@pytest.mark.gpu
@pytest.mark.parametrize("D,big", EVAL_CASES)
def test_eval_metrics_vs_float64_scores_and_oracle_metrics(D, big):
    ops = _ops()
    case = f"D{D}" + (f"_c{big}" if big else "")
    n_rows, ptr, cand, lab = _eval_batch(D, big, seed=D + big)
    n_imp, nnz = len(ptr) - 1, len(cand)
    sizes = np.diff(ptr)
    g = torch.Generator().manual_seed(7 + D)
    table = torch.randn(n_rows, D, generator=g) / D ** 0.5
    user = torch.randn(n_imp, D, generator=g)
    table_d, user_d = table.to(DEV), user.to(DEV)
    per = torch.full((n_imp, 5), float("nan"), dtype=F64, device=DEV)
    prefill = torch.tensor([0.5, -1.25, 2.0, 3.5, 11.0], dtype=F64)
    sums = prefill.clone().to(DEV)
    scores = torch.full((nnz,), float("nan"), device=DEV)
    ops.eval_metrics(table_d, user_d, torch.from_numpy(ptr).to(DEV), torch.from_numpy(cand).to(DEV),
                     torch.from_numpy(lab).to(DEV), int(sizes.max()), per, sums, scores)
    per = per.cpu().numpy()
    sums = sums.cpu().numpy()
    scores = scores.cpu().numpy()

    rows = np.where((cand >= 0) & (cand < n_rows), cand, 0)
    tab64, user64 = table.double().numpy(), user.double().numpy()
    worst, bad_auc, bad_rank, bad_skip, n_rank = 0.0, [], [], [], 0
    for i in range(n_imp):
        seg = slice(int(ptr[i]), int(ptr[i + 1]))
        y, s = lab[seg], scores[seg]
        if sizes[i]:
            ref = tab64[rows[seg]] @ user64[i]
            worst = max(worst, float(np.abs(s - ref).max() / np.abs(ref).max()))
        m = omet.impression_metrics(y, s) if sizes[i] else None
        if m is None:                                # empty or constant labels: zeros, not valid
            if np.any(per[i] != 0.0):
                bad_skip.append(i)
            continue
        if per[i, 4] != 1.0 or abs(per[i, 0] - m[0]) >= 1e-12:
            bad_auc.append(i)
        if not set(s[y == 1].tolist()) & set(s[y == 0].tolist()):   # a positive tying a negative: argsort order
            n_rank += 1                                            # of the oracle is unspecified
            if np.any(np.abs(per[i, 1:4] - np.array(m[1:4])) >= 1e-12):
                bad_rank.append(i)
    _chk(f"eval.score_max_rel.{case}", worst, 1e-6)
    assert not bad_skip, ("skipped impressions with nonzero output", bad_skip[:10])
    assert not bad_auc, ("AUC / valid differs from the oracle", bad_auc[:10])
    assert not bad_rank, ("MRR / nDCG differ from the oracle", bad_rank[:10])
    assert n_rank > 0.9 * n_imp - 10
    assert np.isnan(per).sum() == 0
    np.testing.assert_allclose(sums[:4] - prefill.numpy()[:4], per[:, :4].sum(0), rtol=1e-12, atol=1e-12)
    assert sums[4] - prefill[4].item() == float((per[:, 4] == 1.0).sum())


@pytest.mark.gpu
def test_eval_metrics_rejects_unsupported_d_and_oversized_impressions():
    ops = _ops()
    from tinyrec._lib import TinyRecError
    ptr = torch.tensor([0, 3, 5], dtype=torch.int64, device=DEV)
    cand = torch.tensor([1, 2, 3, 4, 5], dtype=torch.int32, device=DEV)
    label = torch.tensor([1, 0, 0, 0, 1], dtype=torch.int8, device=DEV)
    user_d = {D: torch.ones(2, D, device=DEV) for D in (96, 544, 256)}
    for D in (96, 544):
        per = torch.full((2, 5), 5.0, dtype=F64, device=DEV)
        with pytest.raises(TinyRecError):
            ops.eval_metrics(torch.ones(8, D, device=DEV), user_d[D], ptr, cand, label, 3, per, None,
                             torch.zeros(5, device=DEV))
        torch.cuda.synchronize()
        assert bool((per == 5.0).all())
    per = torch.zeros(2, 5, dtype=F64, device=DEV)
    with pytest.raises(TinyRecError):
        ops.eval_metrics(torch.ones(8, 256, device=DEV), user_d[256], ptr, cand, label, 22753, per, None,
                         torch.zeros(5, device=DEV))
