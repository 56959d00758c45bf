"""Filtered top-k recommendation (``run.recommend`` / ``ops.recommend_topk`` with a candidate pool, per-user exclusions
and per-user categories): the result must be the exact top k of each user's eligible rows under the eval scores -- the
scores ``ops.eval_metrics`` gives every row as a candidate of an impression of the user -- ordered by (score desc, row
asc), with row indices equal and scores equal bit for bit.  The reference scores every (user, row) pair through
``eval_metrics(score_out=...)``, applies the eligibility rules in numpy and sorts."""
import numpy as np
import pytest
import torch

from conftest import report

gpu = pytest.mark.gpu

N_NEWS, D = 20000, 256                       # table rows 0..N_NEWS (row 0 = pad news)


def _eval_scores(table, user):
    """fp32 [n, N+1]: eval_metrics' score of every row as a candidate of user b's impression."""
    import tinyrec.ops as ops
    n, N = user.shape[0], table.shape[0]
    dev = table.device
    ptr = torch.arange(n + 1, device=dev, dtype=torch.int64) * N
    cand = torch.arange(N, device=dev, dtype=torch.int32).repeat(n)
    label = torch.zeros(n * N, device=dev, dtype=torch.int8)
    label[::2] = 1
    per = torch.empty(n, 5, device=dev, dtype=torch.float64)
    score = torch.empty(n * N, device=dev, dtype=torch.float32)
    ops.eval_metrics(table, user, ptr, cand, label, N, per, score_out=score)
    return score.view(n, N).cpu().numpy()


def _reference(scores, hist_idx, hist_mask, k, exclude_history=True, candidates=None, exclude=None, news_category=None,
               user_categories=None):
    n, N = scores.shape
    idx = np.full((n, k), -1, dtype=np.int32)
    sc = np.full((n, k), -np.inf, dtype=np.float32)
    for b in range(n):
        ok = np.ones(N, dtype=bool) if candidates is None else np.asarray(candidates, dtype=bool).copy()
        ok[0] = False
        if exclude_history:
            h = hist_idx[b][(hist_mask[b] != 0) & (hist_idx[b] != 0)].astype(np.int64)
            h[(h < 0) | (h >= N)] = 0
            ok[h] = False
        if exclude is not None:
            e = exclude[b].astype(np.int64)
            ok[e[(e > 0) & (e < N)]] = False
        if news_category is not None:
            ok &= user_categories[b][news_category]
        rows = np.nonzero(ok)[0]
        order = np.lexsort((rows, -scores[b, rows]))[:k]     # score desc (-0 == +0), then row asc
        idx[b, :len(order)] = rows[order]
        sc[b, :len(order)] = scores[b, rows[order]]
    return idx, sc


def _assert_exact(label, got_idx, got_score, ref_idx, ref_score):
    gi, gs = got_idx.cpu().numpy(), got_score.cpu().numpy()
    bad = np.nonzero((gi != ref_idx).any(1) | (gs.view(np.int32) != ref_score.view(np.int32)).any(1))[0]
    assert len(bad) == 0, f"{label}: {len(bad)} users differ, first {bad[0]}: {gi[bad[0]][:8]} vs {ref_idx[bad[0]][:8]}"


def _assert_same(label, a, b):
    assert torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32)), label


def _table(seed=1, n=N_NEWS):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n + 1, D, generator=g) * 0.1


def _histories(n, H, seed):
    import tinyrec.synth as synth
    hist, mask, _, _, _ = synth.eval_impressions(n, N_NEWS, H, seed=seed)
    hist, mask = hist.copy(), mask.copy()
    mask[0] = 0                                  # empty history
    mask[1] = 1                                  # full history
    hist[2, -3:] = [N_NEWS + 5, -7, 0]           # out-of-range ids are row 0; a live id 0
    mask[2, -3:] = 1
    return hist, mask


def _user_encoder(model, ulm, H):
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    args = synth.demo_args(user_log_mask=ulm, user_log_length=H, model=model)
    ue = mb.UserEncoder(args)
    ue.load_state_dict(synth.user_encoder_state("", D, args.user_query_vector_dim, 3, model=model), strict=True)
    return ue.cuda().eval()


def _user_vectors(ue, table, hist, mask):
    with torch.no_grad():
        return ue.forward_gather(table, torch.from_numpy(hist).cuda(), torch.from_numpy(mask).cuda())


def _exclusions(rng, n, E, hist, mask, outside=None):
    """[n, E] ids: random rows, with duplicates, 0 / negative / out-of-range ids, live history rows and (``outside``)
    rows outside the pool mixed in."""
    ex = rng.integers(1, N_NEWS + 1, size=(n, E)).astype(np.int64)
    if E >= 20:
        ex[:, 0] = ex[:, 1]                      # duplicates
        ex[:, 2], ex[:, 3], ex[:, 4], ex[:, 5] = 0, -3, N_NEWS + 1, 2 ** 40     # ignored ids
        live = (mask != 0) & (hist != 0)
        for b in range(n):                       # overlap with the live history
            h = hist[b][live[b]]
            if len(h):
                ex[b, 6:10] = h[:4] if len(h) >= 4 else h[0]
        if outside is not None:
            ex[:, 10:14] = outside[rng.integers(0, len(outside), size=(n, 4))]
    return ex


def _categories(rng, n, C):
    """news_category int [N+1] (category C - 1 is rare: 30 rows) and user_categories bool [n, C]: users allowed
    everything, nothing, only the rare category, or a random subset."""
    cat = rng.integers(0, C - 1, size=N_NEWS + 1)
    cat[rng.choice(np.arange(1, N_NEWS + 1), 30, replace=False)] = C - 1
    uc = rng.random((n, C)) < 0.3
    uc[0::4] = True
    uc[1::4] = False
    uc[2::4] = False
    uc[2::4, C - 1] = True
    return cat, uc


@gpu
@pytest.mark.parametrize("ulm", [True, False])
@pytest.mark.parametrize("model", ["NAML", "NRMS"])
def test_filtered_recommend_exact_under_eval_scores(model, ulm):
    import tinyrec.run as trun
    n, H = 300, 50
    rng = np.random.default_rng(21)
    table = _table().cuda()
    hist, mask = _histories(n, H, seed=17)
    ue = _user_encoder(model, ulm, H)
    scores = _eval_scores(table, _user_vectors(ue, table, hist, mask))
    N1 = N_NEWS + 1
    rand10 = rng.random(N1) < 0.1
    window = np.zeros(N1, dtype=bool)
    window[7000:7900] = True
    single = np.zeros(N1, dtype=bool)
    single[12345] = True
    row0 = np.zeros(N1, dtype=bool)
    row0[0] = True
    tiny = np.zeros(N1, dtype=bool)
    tiny[[0, 3, 18000, 19999, 20000]] = True    # 4 eligible rows: fewer than k pads
    pools = {"rand10": rand10, "window": window, "single": single, "row0": row0, "tiny": tiny}
    outside = np.nonzero(~rand10)[0]
    cat18, uc18 = _categories(rng, n, 18)
    cat64, uc64 = _categories(rng, n, 64)
    case = f"{model}.ulm{int(ulm)}"
    for k in (1, 10, 64):
        base = trun.recommend(ue, table, hist, mask, k)
        configs = {f"pool.{name}": dict(candidates=c) for name, c in pools.items()}
        configs["pool.dev_tensor"] = dict(candidates=torch.from_numpy(rand10).cuda())
        for E in (0, 20, 512):
            configs[f"exclude.E{E}"] = dict(exclude=_exclusions(rng, n, E, hist, mask))
        configs["exclude.in_pool"] = dict(candidates=rand10, exclude=_exclusions(rng, n, 40, hist, mask, outside))
        configs["cat.C18"] = dict(news_category=cat18, user_categories=uc18)
        configs["cat.C64"] = dict(news_category=cat64, user_categories=uc64)
        configs["all_three"] = dict(candidates=rand10, exclude=_exclusions(rng, n, 100, hist, mask, outside),
                                    news_category=cat18, user_categories=uc18)
        configs["all_three.no_history"] = dict(configs["all_three"], exclude_history=False)
        for name, kw in configs.items():
            idx, sc = trun.recommend(ue, table, hist, mask, k, **kw)
            ref_kw = dict(kw)
            if isinstance(ref_kw.get("candidates"), torch.Tensor):
                ref_kw["candidates"] = ref_kw["candidates"].cpu().numpy()
            ref_idx, ref_sc = _reference(scores, hist, mask, k, **ref_kw)
            _assert_exact(f"{case}.k{k}.{name}", idx, sc, ref_idx, ref_sc)
        # filters that filter nothing return the unfiltered result bit for bit
        _assert_same(f"{case}.k{k}.all_true_pool", trun.recommend(ue, table, hist, mask, k, candidates=np.ones(N1, bool)),
                     base)
        _assert_same(f"{case}.k{k}.all_true_categories",
                     trun.recommend(ue, table, hist, mask, k, news_category=cat18, user_categories=np.ones((n, 18), bool)),
                     base)
        idx, sc = trun.recommend(ue, table, hist, mask, k, candidates=row0)
        assert (idx == -1).all() and torch.isinf(sc).all()


@gpu
def test_filtered_ties_inside_a_pool_go_to_lower_rows():
    import tinyrec.ops as ops
    table = _table(seed=3)
    g = torch.Generator().manual_seed(4)
    top = torch.randn(D, generator=g) * 0.3
    copies = [17, 4000, 4001, 9000, 12345, 19999, 20000, 3, 7777, 15000, 11, 2500]
    table[copies] = top                          # 12 identical rows, best for every user: ties straddle k = 5 and 10
    table = table.cuda()
    n = 96
    user = (top.unsqueeze(0) + 0.02 * torch.randn(n, D, generator=g)).cuda()
    hist = np.zeros((n, 4), dtype=np.int32)
    mask = np.zeros((n, 4), dtype=np.float32)
    scores = _eval_scores(table, user)
    rng = np.random.default_rng(5)
    cand = rng.random(N_NEWS + 1) < 0.2
    cand[copies] = True
    cand[4001] = False                           # one copy outside the pool
    excl = np.full((n, 3), 7777, dtype=np.int32)  # and one excluded for every user
    excl[:, 1:] = rng.integers(1, N_NEWS + 1, size=(n, 2))
    pool = ops.recommend_pool(table, cand)
    kept = np.sort([c for c in copies if c not in (4001, 7777)])
    for k in (5, 10, 64):
        idx, sc, _ = ops.recommend_topk(table, user, torch.from_numpy(hist).cuda(), torch.from_numpy(mask).cuda(), k,
                                        pool=pool, exclude=torch.from_numpy(excl).cuda())
        ref_idx, ref_sc = _reference(scores, hist, mask, k, candidates=cand, exclude=excl)
        _assert_exact(f"ties.pool.k{k}", idx, sc, ref_idx, ref_sc)
        m = min(k, len(kept))
        assert (idx[:, :m].cpu().numpy() == kept[:m]).all()


@gpu
def test_long_histories_and_exclusions_stay_off_the_exact_pass():
    """H = 512 live clicks and E = 512 exclusions at k = 64: excluded rows leave the candidate lists instead of raising
    the list threshold, so no user takes the exact pass."""
    import tinyrec.ops as ops
    n, H, E, k = 300, 512, 512, 64
    rng = np.random.default_rng(31)
    table = _table(seed=8).cuda()
    hist = rng.integers(1, N_NEWS + 1, size=(n, H)).astype(np.int32)
    mask = np.ones((n, H), dtype=np.float32)
    excl = rng.integers(1, N_NEWS + 1, size=(n, E)).astype(np.int32)
    ue = _user_encoder("NAML", True, H)
    user = _user_vectors(ue, table, hist, mask)
    scores = _eval_scores(table, user)
    hi_t, hm_t = torch.from_numpy(hist).cuda(), torch.from_numpy(mask).cuda()
    idx, sc, info = ops.recommend_topk(table, user, hi_t, hm_t, k, exclude=torch.from_numpy(excl).cuda())
    ref_idx, ref_sc = _reference(scores, hist, mask, k, exclude=excl)
    _assert_exact("cliff.H512.E512", idx, sc, ref_idx, ref_sc)
    info = info.cpu().numpy()
    report("recommend_filter.cliff.exact_pass_users", int(info[0]))
    report("recommend_filter.cliff.candidates_per_user.mean", float(info[1:].mean()))
    report("recommend_filter.cliff.candidates_per_user.max", int(info[1:].max()))
    assert int(info[0]) == 0
    idx, sc, info = ops.recommend_topk(table, user, hi_t, hm_t, k)          # the history alone
    ref_idx, ref_sc = _reference(scores, hist, mask, k)
    _assert_exact("cliff.H512", idx, sc, ref_idx, ref_sc)
    assert int(info[0]) == 0


@gpu
def test_filtered_overflowing_lists_take_the_exact_pass():
    import tinyrec.ops as ops
    table = _table(seed=6)
    g = torch.Generator().manual_seed(7)
    top = torch.randn(D, generator=g) * 0.3
    table[1:801] = top + 1e-6 * torch.randn(800, D, generator=g)   # 800 rows within a few eps of each other
    table = table.cuda()
    n = 200
    user = (top.unsqueeze(0) + 0.05 * torch.randn(n, D, generator=g)).cuda()
    rng = np.random.default_rng(8)
    hist = rng.integers(1, N_NEWS, size=(n, 20)).astype(np.int32)
    mask = np.ones((n, 20), dtype=np.float32)
    cand = rng.random(N_NEWS + 1) < 0.9          # a large pool: its slices hold more rows than a list (duplicates share one)
    cand[1:801] = True
    excl = rng.integers(1, 801, size=(n, 50)).astype(np.int32)
    cat, uc = _categories(rng, n, 18)
    uc[1::4] = True                              # no user without categories: every user has candidates
    scores = _eval_scores(table, user)
    pool = ops.recommend_pool(table, cand, cat)
    masks = torch.from_numpy(ops.category_masks(uc)).cuda()
    for k in (10, 64):
        idx, sc, info = ops.recommend_topk(table, user, torch.from_numpy(hist).cuda(), torch.from_numpy(mask).cuda(), k,
                                           pool=pool, exclude=torch.from_numpy(excl).cuda(), user_categories=masks)
        ref_idx, ref_sc = _reference(scores, hist, mask, k, candidates=cand, exclude=excl, news_category=cat,
                                     user_categories=uc)
        _assert_exact(f"overflow.filtered.k{k}", idx, sc, ref_idx, ref_sc)
        report(f"recommend_filter.overflow.exact_pass_users.k{k}", int(info[0]))
        assert int(info[0]) > 0 and int(info[0]) == int((info[1:] < 0).sum())


@gpu
def test_filtered_recommend_batch_and_repeat_invariance():
    import tinyrec.run as trun
    H, n = 50, 300
    rng = np.random.default_rng(41)
    table = _table(seed=2).cuda()
    hist, mask = _histories(n, H, seed=9)
    ue = _user_encoder("NAML", True, H)
    cand = rng.random(N_NEWS + 1) < 0.3
    cat, uc = _categories(rng, n, 18)
    kw = dict(candidates=cand, exclude=_exclusions(rng, n, 64, hist, mask, np.nonzero(~cand)[0]), news_category=cat,
              user_categories=uc)
    base = trun.recommend(ue, table, hist, mask, 64, **kw)
    for bs in (77, 128, 64):                     # ragged last batches of 69, 44 (padded to 64) and 44 users
        _assert_same(f"bs{bs}", trun.recommend(ue, table, hist, mask, 64, batch_size=bs, **kw), base)
    _assert_same("again", trun.recommend(ue, table, hist, mask, 64, **kw), base)


@gpu
def test_malformed_filters_raise_through_recommend():
    import tinyrec._lib as L
    import tinyrec.run as trun
    n, H = 70, 8
    table = _table(seed=2, n=500).cuda()
    hist = np.ones((n, H), dtype=np.int32)
    mask = np.ones((n, H), dtype=np.float32)
    for kw in _bad_filters(table.shape[0], n):
        with pytest.raises(L.TinyRecError):
            trun.recommend(None, table, hist, mask, 10, **kw)        # raises before the user encoder is called


# ------------------------------------------------------------------------------------------------ host side (no GPU)
def _bad_filters(N, n):
    ok_cat, ok_uc = np.zeros(N, dtype=np.int64), np.ones((n, 4), dtype=bool)
    return [
        dict(candidates=np.ones(N - 1, dtype=bool)),                         # length
        dict(candidates=np.ones(N, dtype=np.int32)),                         # dtype
        dict(candidates=np.ones((N, 1), dtype=bool)),                        # rank
        dict(candidates=torch.ones(N + 1, dtype=torch.bool)),                # length (torch)
        dict(exclude=np.ones((n, 513), dtype=np.int32)),                     # E > 512
        dict(exclude=np.ones((n + 1, 4), dtype=np.int32)),                   # one row per user
        dict(exclude=np.ones((n, 4), dtype=np.float32)),                     # dtype
        dict(exclude=np.ones(n, dtype=np.int32)),                            # rank
        dict(news_category=ok_cat),                                          # one without the other
        dict(user_categories=ok_uc),
        dict(news_category=ok_cat, user_categories=np.ones((n, 65), dtype=bool)),   # C > 64
        dict(news_category=ok_cat + 4, user_categories=ok_uc),               # category >= C
        dict(news_category=ok_cat - 1, user_categories=ok_uc),               # negative category
        dict(news_category=ok_cat[:-1], user_categories=ok_uc),              # length
        dict(news_category=ok_cat.astype(np.float32), user_categories=ok_uc),  # dtype
        dict(news_category=ok_cat, user_categories=ok_uc.astype(np.int32)),  # dtype
        dict(news_category=ok_cat, user_categories=ok_uc[:-1]),              # one row per user
        dict(news_category=ok_cat, user_categories=ok_uc[:, 0]),             # rank
    ]


def test_malformed_filters_are_rejected_before_staging():
    import tinyrec._lib as L
    import tinyrec.ops as ops
    N, n = 500, 70
    ops.check_recommend_filters(N, n)
    ops.check_recommend_filters(N, n, np.ones(N, dtype=bool), np.ones((n, 512), dtype=np.int64),
                                np.arange(N) % 64, np.ones((n, 64), dtype=bool))
    ops.check_recommend_filters(N, n, torch.zeros(N, dtype=torch.bool), torch.zeros(n, 0, dtype=torch.int32))
    for kw in _bad_filters(N, n):
        with pytest.raises(L.TinyRecError):
            ops.check_recommend_filters(N, n, **kw)
    with pytest.raises(L.TinyRecError):                  # CPU table
        ops.recommend_pool(torch.zeros(N, 64), np.ones(N, dtype=bool))


def test_category_masks():
    import tinyrec.ops as ops
    uc = np.zeros((3, 64), dtype=bool)
    uc[0, [0, 5, 63]] = True
    uc[2] = True
    m = ops.category_masks(uc).view(np.uint64)
    assert m[0] == (1 | 32 | (1 << 63)) and m[1] == 0 and m[2] == np.uint64(2 ** 64 - 1)
