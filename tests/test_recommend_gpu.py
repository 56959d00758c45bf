"""Top-k recommendation over the whole news table (``run.recommend`` / ``ops.recommend_topk``): the result must be the
exact top k of the eligible rows under the eval scores -- the scores ``ops.eval_metrics`` gives every row as a candidate
of an impression of the user -- ordered by (score desc, row asc), with row indices equal and scores equal bit for bit.
The reference scores every (user, row) pair through ``eval_metrics(score_out=...)`` and sorts in numpy."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from conftest import report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
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


def _reference(scores, hist_idx, hist_mask, k, exclude):
    n, N = scores.shape
    idx = np.full((n, k), -1, dtype=np.int32)
    sc = np.full((n, k), -np.inf, dtype=np.float32)
    for b in range(n):
        ok = np.ones(N, dtype=bool)
        ok[0] = False
        if exclude:
            h = hist_idx[b][(hist_mask[b] != 0) & (hist_idx[b] != 0)].astype(np.int64)
            h[(h < 0) | (h >= N)] = 0
            ok[h] = False
        rows = np.nonzero(ok)[0]
        order = np.lexsort((rows, -scores[b, rows]))[:k]     # score desc (-0 == +0), then row asc
        idx[b, :len(order)] = rows[order]
        sc[b, :len(order)] = scores[b, rows[order]]
    return idx, sc


def _assert_exact(label, got_idx, got_score, ref_idx, ref_score):
    gi, gs = got_idx.cpu().numpy(), got_score.cpu().numpy()
    bad = np.nonzero((gi != ref_idx).any(1) | (gs.view(np.int32) != ref_score.view(np.int32)).any(1))[0]
    assert len(bad) == 0, f"{label}: {len(bad)} users differ, first {bad[0]}: {gi[bad[0]][:8]} vs {ref_idx[bad[0]][:8]}"


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


@gpu
@pytest.mark.parametrize("H", [50, 300])
@pytest.mark.parametrize("ulm", [True, False])
@pytest.mark.parametrize("model", ["NAML", "NRMS"])
def test_recommend_exact_under_eval_scores(model, ulm, H):
    import tinyrec.run as trun
    n = 300
    table = _table().cuda()
    hist, mask = _histories(n, H, seed=5 + H)
    ue = _user_encoder(model, ulm, H)
    with torch.no_grad():
        user = ue.forward_gather(table, torch.from_numpy(hist).cuda(), torch.from_numpy(mask).cuda())
    scores = _eval_scores(table, user)
    case = f"{model}.ulm{int(ulm)}.H{H}"
    for k in (1, 10, 64):
        for exclude in (True, False):
            idx, sc = trun.recommend(ue, table, hist, mask, k, exclude_history=exclude)
            ref_idx, ref_sc = _reference(scores, hist, mask, k, exclude)
            _assert_exact(f"{case}.k{k}.ex{int(exclude)}", idx, sc, ref_idx, ref_sc)
    # sanity of the eval scores themselves against float64
    t64, u64 = table.double().cpu(), user.double().cpu()
    rows = idx.long().cpu().clamp(min=0)
    s64 = torch.einsum("bkd,bd->bk", t64[rows], u64)
    bound = (t64[rows].norm(dim=-1) * u64.norm(dim=-1, keepdim=True)).clamp(min=1e-30)
    err = float(((sc.double().cpu() - s64).abs() / bound).max())
    report(f"recommend.score_vs_fp64.{case}", err, 1e-5)
    assert err < 1e-5


@gpu
def test_recommend_candidates_and_batch_invariance():
    import tinyrec.ops as ops
    import tinyrec.run as trun
    H, n = 50, 300
    table = _table(seed=2).cuda()
    hist, mask = _histories(n, H, seed=9)
    ue = _user_encoder("NAML", True, H)
    base = trun.recommend(ue, table, hist, mask, 64)
    for bs in (77, 128, 64):                     # ragged last batches of 69, 44 (padded to 64) and 44 users
        got = trun.recommend(ue, table, hist, mask, 64, batch_size=bs)
        assert torch.equal(got[0], base[0]) and torch.equal(got[1].view(torch.int32), base[1].view(torch.int32)), bs
    with torch.no_grad():
        user = ue.forward_gather(table, torch.from_numpy(hist).cuda(), torch.from_numpy(mask).cuda())
    hi_t, hm_t = torch.from_numpy(hist).cuda(), torch.from_numpy(mask).cuda()
    for k in (10, 64):
        idx, sc, info = ops.recommend_topk(table, user, hi_t, hm_t, k)
        again = ops.recommend_topk(table, user, hi_t, hm_t, k)
        assert torch.equal(idx, again[0]) and torch.equal(sc.view(torch.int32), again[1].view(torch.int32))
        info = info.cpu().numpy()
        cand = info[1:][info[1:] >= 0]
        report(f"recommend.candidates_per_user.k{k}.mean", float(cand.mean()))
        report(f"recommend.candidates_per_user.k{k}.max", int(cand.max()))
        report(f"recommend.exact_pass_users.k{k}", int(info[0]))


@gpu
def test_recommend_ties_go_to_lower_rows():
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
    for k in (5, 10, 64):
        idx, sc, _ = ops.recommend_topk(table, user, torch.from_numpy(hist).cuda(), torch.from_numpy(mask).cuda(), k)
        ref_idx, ref_sc = _reference(scores, hist, mask, k, True)
        _assert_exact(f"ties.k{k}", idx, sc, ref_idx, ref_sc)
        assert (idx[:, :min(k, 12)].cpu().numpy() == np.sort(copies)[:min(k, 12)]).all()


@gpu
def test_recommend_overflowing_lists_take_the_exact_pass():
    import tinyrec.ops as ops
    table = _table(seed=6)
    g = torch.Generator().manual_seed(7)
    top = torch.randn(D, generator=g) * 0.3
    table[1:801] = top + 1e-6 * torch.randn(800, D, generator=g)   # 800 rows within a few eps of each other, in one slice
    table = table.cuda()
    n = 200
    user = (top.unsqueeze(0) + 0.05 * torch.randn(n, D, generator=g)).cuda()
    hist = np.random.default_rng(8).integers(1, N_NEWS, size=(n, 20)).astype(np.int32)
    mask = np.ones((n, 20), dtype=np.float32)
    scores = _eval_scores(table, user)
    for k in (10, 64):
        idx, sc, info = ops.recommend_topk(table, user, torch.from_numpy(hist).cuda(), torch.from_numpy(mask).cuda(), k)
        ref_idx, ref_sc = _reference(scores, hist, mask, k, True)
        _assert_exact(f"overflow.k{k}", idx, sc, ref_idx, ref_sc)
        report(f"recommend.overflow.exact_pass_users.k{k}", int(info[0]))
        assert int(info[0]) > 0 and int(info[0]) == int((info[1:] < 0).sum())


@gpu
def test_recommend_small_table_pads():
    import tinyrec.ops as ops
    table = _table(seed=10, n=6).cuda()          # rows 1..6 eligible
    n = 70
    user = torch.randn(n, D, generator=torch.Generator().manual_seed(11)).cuda()
    hist = np.tile(np.array([[0, 2, 9]], dtype=np.int32), (n, 1))
    mask = np.ones((n, 3), dtype=np.float32)
    scores = _eval_scores(table, user)
    for exclude, n_ok in ((True, 5), (False, 6)):
        idx, sc, _ = ops.recommend_topk(table, user, torch.from_numpy(hist).cuda(), torch.from_numpy(mask).cuda(), 10,
                                        exclude_history=exclude)
        ref_idx, ref_sc = _reference(scores, hist, mask, 10, exclude)
        _assert_exact(f"small.ex{int(exclude)}", idx, sc, ref_idx, ref_sc)
        assert (idx[:, n_ok:] == -1).all() and torch.isinf(sc[:, n_ok:]).all() and (idx[:, :n_ok] >= 1).all()


# ------------------------------------------------------------------------------------------------ host side (no GPU)
def test_recommend_rejects_bad_shapes_before_staging():
    import tinyrec._lib as L
    import tinyrec.ops as ops
    import tinyrec.run as trun
    ops.check_recommend(64, 256, 512)
    for k, d, h in ((0, 256, 50), (65, 256, 50), (10, 48, 50), (10, 512, 50), (10, 256, 0), (10, 256, 513)):
        with pytest.raises(L.TinyRecError):
            ops.check_recommend(k, d, h)
    t = torch.zeros(8, 64)
    u = torch.zeros(2, 64)
    hi, hm = torch.zeros(2, 5, dtype=torch.int32), torch.zeros(2, 5)
    with pytest.raises(L.TinyRecError):                  # CPU tensors
        ops.recommend_topk(t, u, hi, hm, 4)
    with pytest.raises(L.TinyRecError):                  # dtype
        ops.recommend_topk(t.double(), u, hi, hm, 4)
    with pytest.raises(L.TinyRecError):
        trun.recommend(None, t, hi.numpy(), hm.numpy(), 4)


def test_recommend_sass_is_blackwell_native():
    import tinyrec._lib as L
    if not os.path.exists(L.LIB_PATH):
        import __graft_entry__ as ge
        ge.build()
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", L.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = {}
    for blk in re.split(r"\n\s*Function : ", sass)[1:]:
        name, _, body = blk.partition("\n")
        funcs[name.strip()] = body
    sel = [b for n, b in funcs.items() if "rec_select_kernel" in n]
    assert len(sel) == 1
    assert "UTCHMMA.2CTA" in sel[0] and "LDTM" in sel[0] and "UTMALDG" in sel[0] and "R2UR.BROADCAST" not in sel[0]
    assert len([n for n in funcs if "rec_merge_kernel" in n]) == 4 and len([n for n in funcs if "rec_exact_kernel" in n]) == 4
