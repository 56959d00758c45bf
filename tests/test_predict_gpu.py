"""Prediction files for unlabeled impressions (``run.predict`` / ``run.write_prediction`` / ``run.predict_test``,
``ops.predict_ranks`` / ``ops.format_prediction``, ``dataloader.parse_test_line``):

  * scores bit for bit what ``ops.eval_metrics(score_out=...)`` writes for the same user vectors;
  * ranks equal to numpy's ``np.argsort(keys, kind="stable")[::-1]`` order over the order keys (-0 == +0);
  * MRR and nDCG@5/10 from the ranks equal to ``evaluate``'s per-impression values;
  * results independent of the batch size and of repeated calls;
  * the file byte-equal to a Python formatter, and ``predict_test`` writing what ``write_prediction(predict(...))``
    writes.
Host-side validation, the parser and a static SASS check run without a GPU."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

N_NEWS = 5000


def _table(D, seed=1, n=N_NEWS):
    g = torch.Generator().manual_seed(seed)
    t = torch.randn(n + 1, D, generator=g) * 0.1
    t[0] = 0.0
    return t


def _user_encoder(model, ulm, H, D, precision="bf16"):
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    heads = dict(num_attention_heads=D // 16) if model == "NRMS" else {}      # NRMS: 16 dims per head
    args = synth.demo_args(user_log_mask=ulm, user_log_length=H, model=model, precision=precision, news_dim=D, **heads)
    ue = mb.UserEncoder(args)
    ue.load_state_dict(synth.user_encoder_state("", D, args.user_query_vector_dim, 3, model=model, n_heads=D // 16),
                       strict=True)
    return ue.cuda().eval()


def _impressions(n, H, seed, n_news=N_NEWS):
    """Dev-shaped impressions (C in 2..300) with an empty and a full history, unknown candidate ids, an impression of
    one candidate and one of 300."""
    import tinyrec.synth as synth
    hist, mask, ptr, cand, lab = synth.eval_impressions(n, n_news, H, seed=seed)
    hist, mask, cand = hist.copy(), mask.copy(), cand.copy()
    mask[0], hist[0] = 0, 0                                   # empty history
    mask[1] = 1                                               # full history
    C = np.diff(ptr)
    C[2], C[3] = 1, 300
    ptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(C, out=ptr[1:])
    rng = np.random.default_rng(seed)
    cand = rng.integers(1, n_news + 1, size=int(ptr[-1])).astype(np.int32)
    lab = (rng.random(int(ptr[-1])) < 0.15).astype(np.int8)
    cand[ptr[4]:ptr[4] + 3] = [-5, n_news + 10, 0]            # unknown ids score as row 0
    return hist, mask, ptr, cand, lab


def _user(ue, table, hist, mask):
    with torch.no_grad():
        return ue.forward_gather(table, torch.from_numpy(hist).cuda(), torch.from_numpy(mask).cuda())


def _eval_scores(table, user, ptr, cand):
    import tinyrec.ops as ops
    n = len(ptr) - 1
    per = torch.empty(n, 5, device="cuda", dtype=torch.float64)
    score = torch.empty(max(len(cand), 1), device="cuda", dtype=torch.float32)
    label = torch.zeros(len(cand), device="cuda", dtype=torch.int8)
    ops.eval_metrics(table, user, torch.from_numpy(ptr).cuda(), torch.from_numpy(cand).cuda(), label,
                     int(np.diff(ptr).max()), per, score_out=score)
    return score[:len(cand)].cpu().numpy()


def _ref_ranks(score, ptr):
    """numpy reference: rank of candidate i = its position in np.argsort(keys, kind="stable")[::-1], keys with -0 == +0."""
    keys = score.astype(np.float64) + 0.0
    rank = np.empty(len(score), dtype=np.int32)
    for b in range(len(ptr) - 1):
        p0, p1 = int(ptr[b]), int(ptr[b + 1])
        order = np.argsort(keys[p0:p1], kind="stable")[::-1]
        r = np.empty(p1 - p0, dtype=np.int32)
        r[order] = np.arange(1, p1 - p0 + 1, dtype=np.int32)
        rank[p0:p1] = r
    return rank


def _bits(x):
    return np.asarray(x).view(np.int32)


def _check(label, got, ref_score, ptr):
    score, rank = got[0].cpu().numpy(), got[1].cpu().numpy()
    assert np.array_equal(_bits(score), _bits(ref_score)), f"{label}: scores differ"
    ref = _ref_ranks(ref_score, ptr)
    bad = np.nonzero(rank != ref)[0]
    assert len(bad) == 0, f"{label}: {len(bad)} ranks differ, first at {bad[0]}: {rank[bad[0]]} vs {ref[bad[0]]}"


def _same(label, a, b):
    assert torch.equal(a[1], b[1]) and torch.equal(a[0].view(torch.int32), b[0].view(torch.int32)), label


# ------------------------------------------------------------------------------------------------ scores and ranks
@gpu
@pytest.mark.parametrize("H,D", [(50, 256), (512, 64)])
@pytest.mark.parametrize("ulm", [True, False])
@pytest.mark.parametrize("model", ["NAML", "NRMS"])
def test_predict_scores_and_ranks(model, ulm, H, D):
    import tinyrec.run as trun
    n = 400
    table = _table(D).cuda()
    hist, mask, ptr, cand, _ = _impressions(n, H, seed=11)
    ue = _user_encoder(model, ulm, H, D)
    ref = _eval_scores(table, _user(ue, table, hist, mask), ptr, cand)
    _check(f"{model}.ulm{int(ulm)}.H{H}.D{D}", trun.predict(ue, table, hist, mask, ptr, cand), ref, ptr)


@gpu
@pytest.mark.parametrize("model", ["NAML", "NRMS"])
def test_predict_fp32_user_encoder(model):
    """The fp32 user encoder adds its attention logits with shared-memory atomics, so two ``forward_gather`` calls may
    differ in the last bits: the bitwise check runs on one set of user vectors through ``ops.predict_ranks``, and
    ``predict``'s ranks are checked against its own scores."""
    import tinyrec.ops as ops
    import tinyrec.run as trun
    H, D, n = 50, 256, 300
    table = _table(D, seed=2).cuda()
    hist, mask, ptr, cand, _ = _impressions(n, H, seed=12)
    ue = _user_encoder(model, True, H, D, precision="fp32")
    user = _user(ue, table, hist, mask)
    ref = _eval_scores(table, user, ptr, cand)
    got = (torch.empty(len(cand), device="cuda"), torch.empty(len(cand), device="cuda", dtype=torch.int32))
    ops.predict_ranks(table, user, torch.from_numpy(ptr).cuda(), torch.from_numpy(cand).cuda(), int(np.diff(ptr).max()),
                      *got)
    _check(f"fp32.{model}.ops", got, ref, ptr)
    score, rank = trun.predict(ue, table, hist, mask, ptr, cand)
    score = score.cpu().numpy()
    assert np.abs(score - ref).max() <= 1e-5 * np.abs(ref).max()
    assert np.array_equal(rank.cpu().numpy(), _ref_ranks(score, ptr))


@gpu
def test_predict_ties_duplicates_and_long_impressions():
    """All-duplicate candidates rank C..1 by position; zero rows stored as +0 and -0 tie; impressions of 5 000 and
    20 000 candidates (the second needs more than 48 KB of shared memory per block)."""
    import tinyrec.run as trun
    H, D = 50, 256
    table = _table(D, seed=3)
    table[10] = 0.0
    table[11] = -0.0
    table[12] = torch.where(torch.arange(D) % 2 == 0, torch.tensor(0.0), torch.tensor(-0.0))
    table[13:20] = table[20]                                  # 8 identical rows
    table = table.cuda()
    sizes = [1, 2, 300, 37, 40, 5000, 20000, 64, 33, 65] + [40] * 60
    n = len(sizes)
    ptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(sizes, out=ptr[1:])
    rng = np.random.default_rng(4)
    cand = rng.integers(1, N_NEWS + 1, size=int(ptr[-1])).astype(np.int32)
    cand[ptr[3]:ptr[4]] = 777                                 # one news repeated 37 times
    cand[ptr[4]:ptr[5]] = rng.choice([10, 11, 12, 0, -3, 13, 14, 15, 20], size=40)   # zero scores and duplicates
    cand[ptr[8]:ptr[9]] = 0                                   # every candidate is the pad row
    hist = rng.integers(1, N_NEWS + 1, size=(n, H)).astype(np.int32)
    mask = np.ones((n, H), dtype=np.float32)
    hist[5:7], mask[5:7] = 0, 0                               # empty histories on the long impressions
    ue = _user_encoder("NAML", True, H, D)
    ref = _eval_scores(table, _user(ue, table, hist, mask), ptr, cand)
    got = trun.predict(ue, table, hist, mask, ptr, cand)
    _check("ties", got, ref, ptr)
    rank = got[1].cpu().numpy()
    assert np.array_equal(rank[ptr[3]:ptr[4]], np.arange(37, 0, -1))
    assert np.array_equal(rank[ptr[8]:ptr[9]], np.arange(33, 0, -1))
    assert rank[ptr[0]] == 1
    for b in range(n):
        assert np.array_equal(np.sort(rank[ptr[b]:ptr[b + 1]]), np.arange(1, sizes[b] + 1))


def _metrics_from_ranks(rank, lab, ptr):
    """host MRR, nDCG@5, nDCG@10 (metrics.py:5-23 with binary labels) from the ranks; NaN where evaluate skips."""
    out = np.full((len(ptr) - 1, 3), np.nan)
    for b in range(len(ptr) - 1):
        p0, p1 = int(ptr[b]), int(ptr[b + 1])
        y, r = lab[p0:p1], rank[p0:p1].astype(np.float64)
        P = int(y.sum())
        if P == 0 or P == p1 - p0:
            continue
        rp = r[y == 1]
        out[b, 0] = np.mean(1.0 / rp)
        for j, k in enumerate((5, 10)):
            dcg = np.sum(1.0 / np.log2(rp[rp <= k] + 1))
            idcg = np.sum(1.0 / np.log2(np.arange(1, min(k, P) + 1) + 1))
            out[b, 1 + j] = dcg / idcg
    return out


@gpu
@pytest.mark.parametrize("model", ["NAML", "NRMS"])
def test_predict_agrees_with_evaluate(model):
    import tinyrec.run as trun
    H, D, n = 50, 256, 500
    table = _table(D, seed=5)
    table[30:34] = table[35]                                  # tied scores
    table = table.cuda()
    hist, mask, ptr, cand, lab = _impressions(n, H, seed=13)
    for b in range(20, 60):                                   # duplicates and ties with either label
        p0, c = int(ptr[b]), int(ptr[b + 1] - ptr[b])
        if c >= 4:
            cand[p0:p0 + 4] = [cand[p0], cand[p0], 30, 31]
            lab[p0:p0 + 4] = [b % 2, 1 - b % 2, 1, 0]
    ue = _user_encoder(model, True, H, D)
    _, _, per = trun.evaluate(ue, table, hist, mask, ptr, cand, lab, batch_size=n, return_per_impression=True)
    score, rank = trun.predict(ue, table, hist, mask, ptr, cand)
    ref = _eval_scores(table, _user(ue, table, hist, mask), ptr, cand)
    assert np.array_equal(_bits(score.cpu().numpy()), _bits(ref))      # evaluate's one batch of 500 scores these
    mine = _metrics_from_ranks(rank.cpu().numpy(), lab, ptr)
    per = per.cpu().numpy()
    valid = per[:, 4] != 0
    assert valid.sum() > 400 and np.array_equal(valid, ~np.isnan(mine[:, 0]))
    err = np.abs(mine[valid] - per[valid, 1:4]).max()
    assert err <= 1e-12, err


@gpu
def test_predict_batch_and_repeat_invariance():
    import tinyrec.run as trun
    H, D, n = 50, 256, 300
    table = _table(D, seed=6).cuda()
    hist, mask, ptr, cand, _ = _impressions(n, H, seed=14)
    ue = _user_encoder("NAML", False, H, D)
    base = trun.predict(ue, table, hist, mask, ptr, cand)
    for bs in (77, 128, 64, 30, 1):                           # ragged last batches; batches under 64 impressions
        _same(f"bs{bs}", trun.predict(ue, table, hist, mask, ptr, cand, batch_size=bs), base)
    _same("again", trun.predict(ue, table, hist, mask, ptr, cand), base)


# ------------------------------------------------------------------------------------------------ the file
def _py_format(imp_ids, ptr, rank):
    return "".join(f"{i} [{','.join(map(str, rank[ptr[b]:ptr[b + 1]]))}]\n"
                   for b, i in enumerate(imp_ids.tolist())).encode()


def _parse(text):
    out = []
    for line in text.decode().splitlines():
        m = re.fullmatch(r"(\d+) \[([0-9,]*)\]", line)
        assert m, line
        out.append((int(m.group(1)), [int(x) for x in m.group(2).split(",")] if m.group(2) else []))
    return out


@gpu
def test_write_prediction_matches_python_formatter(tmp_path):
    import tinyrec.run as trun
    H, D, n = 50, 256, 1000
    table = _table(D, seed=7).cuda()
    hist, mask, ptr, cand, _ = _impressions(n, H, seed=15)
    ue = _user_encoder("NRMS", True, H, D)
    _, rank = trun.predict(ue, table, hist, mask, ptr, cand)
    rng = np.random.default_rng(8)
    imp_ids = rng.integers(0, 2 ** 63 - 1, size=n, dtype=np.int64) >> rng.integers(0, 63, size=n)
    imp_ids[:4] = [0, 9, 10, 2 ** 63 - 1]                      # 1 to 19 digits
    path = str(tmp_path / "prediction.txt")
    nbytes = trun.write_prediction(path, imp_ids, ptr, rank)
    text = open(path, "rb").read()
    r = rank.cpu().numpy()
    assert nbytes == len(text) and text == _py_format(imp_ids, ptr, r)
    back = _parse(text)
    assert [i for i, _ in back] == imp_ids.tolist()
    for b, (_, ranks) in enumerate(back):
        assert ranks == r[ptr[b]:ptr[b + 1]].tolist()
        assert sorted(ranks) == list(range(1, len(ranks) + 1))


@gpu
def test_format_prediction_any_int32_and_empty_impressions():
    import tinyrec.ops as ops
    rng = np.random.default_rng(9)
    sizes = [0, 1, 0, 31, 32, 33, 64, 65, 500, 0]
    ptr = np.zeros(len(sizes) + 1, dtype=np.int64)
    np.cumsum(sizes, out=ptr[1:])
    rank = rng.integers(-2 ** 31, 2 ** 31, size=int(ptr[-1])).astype(np.int32)
    rank[:3] = [0, -2 ** 31, 2 ** 31 - 1]
    rank[5:40] = rng.integers(0, 10, size=35)
    imp_ids = np.arange(len(sizes), dtype=np.int64) * 123457
    text = ops.format_prediction(torch.from_numpy(imp_ids).cuda(), torch.from_numpy(ptr).cuda(),
                                 torch.from_numpy(rank).cuda())
    assert bytes(text.cpu().numpy()) == _py_format(imp_ids, ptr, rank)
    empty = ops.format_prediction(torch.zeros(0, dtype=torch.int64, device="cuda"),
                                  torch.zeros(1, dtype=torch.int64, device="cuda"),
                                  torch.zeros(0, dtype=torch.int32, device="cuda"))
    assert empty.numel() == 0


# ------------------------------------------------------------------------------------------------ the driver
@gpu
def test_predict_test_writes_what_write_prediction_writes(tmp_path):
    import tinyrec.checkpoint as ckpt
    import tinyrec.dataloader as dl
    import tinyrec.model_bert as mb
    import tinyrec.run as trun
    import tinyrec.synth as synth
    n_news, H, L, layers = 300, 20, 12, 2
    news = synth.news_table(n_news, L=L, seed=21)
    sd = synth.kd_model_state(layers, 2, 24, noisy=True)
    args = synth.demo_args(num_student_layers=layers, num_teachers=2, user_log_length=H, batch_size=4, enable_hvd=False,
                           model_dir=str(tmp_path / "model"), load_ckpt_name=None, user_log_mask=True)
    model = mb.Model(args)
    model.load_state_dict(sd, strict=True)
    os.makedirs(args.model_dir)
    ckpt.save_checkpoint(os.path.join(args.model_dir, "epoch-3.pt"), model)
    rng = np.random.default_rng(22)
    lines = []
    for i in range(150):
        clicks = " ".join(f"N{x}" for x in rng.integers(1, n_news + 1, size=rng.integers(0, 30)))
        imps = " ".join(f"N{x}" for x in rng.integers(1, n_news + 40, size=rng.integers(2, 60)))   # some unknown
        lines.append(f"{1000 + 7 * i}\tU{i}\t11/15/2019 8:00:00 AM\t{clicks}\t{imps}\n")
    news_index = {f"N{i}": i for i in range(1, n_news + 1)}
    imp_ids, hist, mask, ptr, cand = dl.pack_test_lines(lines, news_index, H)
    out = str(tmp_path / "prediction.txt")
    trun.predict_test(args, None, news, imp_ids, hist, mask, ptr, cand, out)
    model.cuda().eval()
    table = trun.build_news_table(model.student.news_encoder, news, batch_size=args.batch_size * 16)
    _, rank = trun.predict(model.student.user_encoder, table, hist, mask, ptr, cand)
    ref = str(tmp_path / "reference.txt")
    trun.write_prediction(ref, imp_ids, ptr, rank)
    got = open(out, "rb").read()
    assert got == open(ref, "rb").read() and len(got.splitlines()) == 150
    assert got.startswith(b"1000 [")


@gpu
def test_predict_rejects_malformed_inputs_before_staging():
    import tinyrec._lib as L
    import tinyrec.run as trun

    class NoCall:
        def forward_gather(self, *a):
            raise AssertionError("staged")

    table = _table(256, n=50).cuda()
    for args in _bad_inputs():
        with pytest.raises(L.TinyRecError):
            trun.predict(NoCall(), table, *args)
    hist, mask = np.zeros((3, 5), np.int32), np.zeros((3, 5), np.float32)
    ptr, cand = np.array([0, 1, 2, 3]), np.ones(3, np.int32)
    with pytest.raises(L.TinyRecError):
        trun.predict(NoCall(), _table(96, n=50).cuda(), hist, mask, ptr, cand)     # D not instantiated
    with pytest.raises(L.TinyRecError):
        trun.predict(NoCall(), table, hist, mask, ptr, cand, batch_size=0)
    with pytest.raises(L.TinyRecError):
        trun.predict(object(), table, hist, mask, ptr, cand)                       # no forward_gather


# ------------------------------------------------------------------------------------------------ host side (no GPU)
def _bad_inputs():
    h, m = np.zeros((3, 5), np.int32), np.zeros((3, 5), np.float32)
    ptr, cand = np.array([0, 1, 2, 3]), np.ones(3, np.int32)
    big = np.array([0, 1, 2, 51203])
    return [
        (np.zeros((3, 0), np.int32), np.zeros((3, 0), np.float32), ptr, cand),     # H = 0
        (np.zeros((3, 513), np.int32), np.zeros((3, 513), np.float32), ptr, cand),  # H > 512
        (h, m[:, :4], ptr, cand),                                                   # mask shape
        (h[0], m[0], ptr, cand),                                                    # rank
        (h.astype(np.float32), m, ptr, cand),                                       # dtype
        (h, m, np.array([1, 1, 2, 3]), cand),                                       # ptr[0] != 0
        (h, m, np.array([0, 2, 1, 3]), cand),                                       # decreasing
        (h, m, np.array([0, 1, 2, 4]), cand),                                       # ptr[-1] != nnz
        (h, m, np.array([0, 1, 3]), cand),                                          # n + 1 entries
        (h, m, ptr.astype(np.float64), cand),                                       # dtype
        (h, m, ptr, cand.astype(np.float32)),
        (h, m, ptr, np.array([1, 2, 2 ** 40])),                                     # outside int32
        (h, m, big, np.ones(51203, np.int32)),                                      # C > 51 200
    ]


def test_check_predict_rejects_malformed_inputs():
    import tinyrec._lib as L
    import tinyrec.ops as ops
    h, m = np.zeros((3, 512), np.int64), np.zeros((3, 512), np.float64)
    got = ops.check_predict(64, h, m, [0, 0, 2, 51202], np.ones(51202, np.int64))
    assert [a.dtype for a in got] == [np.int32, np.float32, np.int64, np.int32]
    for args in _bad_inputs():
        with pytest.raises(L.TinyRecError):
            ops.check_predict(256, *args)
    for D in (48, 96, 1024):
        with pytest.raises(L.TinyRecError):
            ops.check_predict(D, h, m, [0, 0, 2, 3], np.ones(3, np.int32))


def test_write_prediction_rejects_mismatched_inputs(tmp_path):
    import tinyrec._lib as L
    import tinyrec.run as trun
    rank = torch.ones(5, dtype=torch.int32)
    ptr = np.array([0, 2, 5])
    path = str(tmp_path / "p.txt")
    for ids, p, r in (([1, 2, 3], ptr, rank),                 # one id too many
                      ([1], ptr, rank),
                      ([1, -2], ptr, rank),                   # negative id
                      ([1.0, 2.0], ptr, rank),                # not integers
                      ([1, 2], np.array([0, 2, 4]), rank),    # ptr[-1] != nnz
                      ([1, 2], np.array([0, 3, 2, 5]), rank),
                      ([1, 2], ptr, rank.long()),             # rank dtype
                      ([1, 2], ptr, rank.view(5, 1))):
        with pytest.raises(L.TinyRecError):
            trun.write_prediction(path, ids, p, r)
    assert not os.path.exists(path)


def test_parse_test_line_with_and_without_labels():
    import tinyrec.dataloader as dl
    news_index = {"N1": 1, "N2": 2, "N3": 3, "N4": 4}
    plain = dl.parse_test_line("17\tU1\t11/15/2019 8:00:00 AM\tN1 N2 NX\tN3 N4 N9 N1\n", news_index, 4)
    labelled = dl.parse_test_line(b"17\tU1\t11/15/2019 8:00:00 AM\tN1 N2 NX\tN3-1 N4-0 N9-0 N1-1", news_index, 4)
    assert plain == labelled == (17, [0, 1, 2, 0], [0, 1, 1, 1], [3, 4, 0, 1])
    imp_ids, hist, mask, ptr, cand = dl.pack_test_lines(
        ["5\tU\tt\t\tN1-0 N2-1\n", "\n", "6\tU\tt\tN4\tN3\n"], news_index, 2)
    assert imp_ids.tolist() == [5, 6] and hist.tolist() == [[0, 0], [0, 4]] and mask.tolist() == [[0, 0], [0, 1]]
    assert ptr.tolist() == [0, 2, 3] and cand.tolist() == [1, 2, 3]
    assert (imp_ids.dtype, hist.dtype, mask.dtype, ptr.dtype, cand.dtype) == (np.int64, np.int32, np.float32, np.int64,
                                                                               np.int32)


def test_predict_sass_has_no_spills_and_shares_the_scoring_kernel():
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
    new = [n for n in funcs if re.search(r"predict_(rank|line_bytes|write)_kernel", n)]
    assert len(new) == 3
    for n in new:
        assert not re.search(r"\b(STL|LDL)\b", funcs[n]), f"{n} uses local memory"
    # the scores come from tnr_eval_metrics' own kernels: one copy of each instantiation in the library
    assert len([n for n in funcs if "eval_score_kernel" in n]) == 5
