"""The fp32 inference mode of the user encoders (``args.precision = 'fp32'``): the 3xTF32 user-encoder forward (plain and
gather) and Q/K/V projection GEMM against float64, sharp attention logits on which the TF32 kernels miss 1e-4 and the
split kernels do not, ``ModelBert.forward`` against the reference's fixtures and the float64 oracle, and
``run.evaluate`` with an fp32 user encoder.

Bound: the 1e-4 parity level of BASELINE.json north_star, as the max over rows of the row-relative error
||y - ref|| / ||ref||, on user vectors and on each impression's row of click scores.  The kernels alone are held to about
twice their measured error.  Every measured error is recorded with conftest.report."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, report

BOUND = 1e-4
KERNEL_BOUND = 1e-5         # split user encoder alone (measured up to 4.3e-6, the fp32 weighted sum over H = 512 rows)
SHARP_BOUND = 2e-5          # split user encoder alone on logits spanning tens (measured up to 8.6e-6)
GEMM_BOUND = 5e-6           # split Q/K/V projection GEMM (measured up to 2.2e-6)
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
def test_user_encoder_precision_field():
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    from tinyrec._lib import TinyRecError
    for model in ("NAML", "NRMS"):
        ue = mb.UserEncoder(synth.demo_args(model=model))
        assert ue.precision == "bf16"                                                   # reference args
        ue32 = mb.UserEncoder(synth.demo_args(model=model, precision="fp32"))
        assert ue32.precision == "fp32"
        assert list(ue32.state_dict()) == list(ue.state_dict())                        # a plain attribute, no new keys
        for bad in ("fp16", "FP32", "tf32", None):
            with pytest.raises(TinyRecError):
                mb.UserEncoder(synth.demo_args(model=model, precision=bad))
    m = mb.ModelBert(synth.demo_args(num_student_layers=1, precision="fp32"))
    assert m.news_encoder.precision == m.user_encoder.precision == "fp32"


def _hmma_counts():
    lib = os.path.join(ROOT, "tiny-newsrec_b200", "libtinyrec.so")
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(lib) or not os.path.exists(tool):
        pytest.skip("needs the built libtinyrec.so and cuobjdump")
    out = subprocess.run([tool, "-sass", lib], capture_output=True, text=True, check=True).stdout
    counts, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = 0
        elif cur is not None and re.search(r"\bHMMA\.", line):
            counts[cur] += 1
    return counts


def test_split_kernels_issue_three_mma_per_tf32_mma():
    """Each 3xTF32 instantiation issues exactly three mma.sync for every one of its TF32 twin (no lo term dropped)."""
    c = _hmma_counts()
    pairs = [("_ZN3tnr23user_encoder_fwd_kernelILb0ELb0EEEvNS_11UeFwdParamsE",
              "_ZN3tnr23user_encoder_fwd_kernelILb0ELb1EEEvNS_11UeFwdParamsE"),
             ("_ZN3tnr23user_encoder_fwd_kernelILb1ELb0EEEvNS_11UeFwdParamsE",
              "_ZN3tnr23user_encoder_fwd_kernelILb1ELb1EEEvNS_11UeFwdParamsE"),
             ("_ZN3tnr15sgemm_nt_kernelILb0EEEvPKfS2_S2_Pfiiixxxx", "_ZN3tnr15sgemm_nt_kernelILb1EEEvPKfS2_S2_Pfiiixxxx")]
    for tf32, split in pairs:
        assert c[tf32] > 0 and c[split] == 3 * c[tf32], (tf32, c[tf32], c[split])


# ------------------------------------------------------------------------------------------------ kernels
def _ue_ref(v, mask, pad, W1, b1, w2, b2, use_mask):
    """model_bert.py:155-176 (NAML) + :15-34 in float64: (user [B, D], a [B, H])."""
    v, mask = v.double(), mask.double()
    if not use_mask:
        v = v * mask.unsqueeze(-1) + pad.double().view(1, 1, -1) * (1 - mask.unsqueeze(-1))
    alpha = torch.exp(torch.tanh(v @ W1.double().t() + b1.double()) @ w2.double() + b2.double())
    if use_mask:
        alpha = alpha * mask
    a = alpha / (alpha.sum(1, keepdim=True) + 1e-8)
    return (a.unsqueeze(-1) * v).sum(1), a


def _mask(B, H, seed):
    """Front-padded histories plus: an all-masked one (1), a full one (2), one live row at h = H - 1 (3), fractional
    masks (4, 5)."""
    g = torch.Generator().manual_seed(seed)
    mask = (torch.rand(B, H, generator=g) > 0.3).float()
    mask[1] = 0
    mask[2] = 1
    mask[3] = 0
    mask[3, H - 1] = 1
    mask[4] = 0.25
    mask[5, ::2] = 0.5
    return mask.cuda()


def _pool_params(D, Q, seed, sharp):
    """pad_doc, att_fc1 / att_fc2 for rows of scale 0.5.  ``sharp``: fc1 pre-activations of std ~2 and an fc2 that
    spreads the attention logits over tens (|logit| up to ~40), as trained weights do; otherwise the synthetic scale
    of the other user-encoder tests (logits within a few units)."""
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)  # noqa: E731
    w1s, w2s = (4.0 / D ** 0.5, 0.5) if sharp else (0.06, 0.1)
    return [t.cuda() for t in (r(D) * 0.5, r(Q, D) * w1s, r(Q) * 0.1, r(Q) * w2s, r(1))]


def _run_ue(vecs, mask, params, use_mask, B, H, fp32):
    import tinyrec.ops as ops
    D = vecs.shape[1]
    user, a = torch.empty(B, D, device="cuda"), torch.empty(B, H, device="cuda")
    ops.user_encoder_fwd(vecs, mask, *params, use_mask, user, a, None, B, H, fp32=fp32)
    return user, a


@gpu
@pytest.mark.parametrize("use_mask", [False, True])
@pytest.mark.parametrize("D", [64, 256])
@pytest.mark.parametrize("H", [1, 50, 64, 65, 200, 512])
def test_split_user_encoder_vs_float64(H, D, use_mask):
    import tinyrec.ops as ops
    B, Q, N = 7, 200, 3000
    case = f"H{H}_D{D}_mask{int(use_mask)}"
    g = torch.Generator().manual_seed(H * 10 + D)
    mask = _mask(B, H, seed=H)
    params = _pool_params(D, Q, seed=D + H, sharp=False)
    vecs = (torch.randn(B * H, D, generator=g) * 0.5).cuda()
    user, a = _run_ue(vecs, mask, params, use_mask, B, H, fp32=True)
    ru, ra = _ue_ref(vecs.view(B, H, D), mask, *params, use_mask)
    _chk(f"fp32_ue.plain.user.{case}", _rowrel(user, ru), KERNEL_BOUND)
    _chk(f"fp32_ue.plain.a.{case}", _rowrel(a, ra), KERNEL_BOUND)
    if use_mask:
        assert float(user[1].abs().max()) == 0.0 and float(a[1].abs().max()) == 0.0     # all masked: 0 / (0 + 1e-8)
    # gather form, with out-of-range ids (they read row 0, as the loader does)
    table = (torch.randn(N, D, generator=g) * 0.5).cuda()
    idx = torch.randint(0, N, (B, H), generator=g).int()
    idx[0, 0] = -1
    idx[2, H - 1] = N
    idx[6, :min(H, 3)] = N + 5
    idx = idx.cuda()
    ug, ag = torch.empty(B, D, device="cuda"), torch.empty(B, H, device="cuda")
    ops.user_encoder_fwd_gather(table, idx, mask, *params, use_mask, ug, ag, fp32=True)
    safe = torch.where((idx >= 0) & (idx < N), idx, torch.zeros_like(idx)).long()
    rgu, rga = _ue_ref(table[safe], mask, *params, use_mask)
    _chk(f"fp32_ue.gather.user.{case}", _rowrel(ug, rgu), KERNEL_BOUND)
    _chk(f"fp32_ue.gather.a.{case}", _rowrel(ag, rga), KERNEL_BOUND)
    if use_mask:
        assert float(ug[1].abs().max()) == 0.0


@gpu
@pytest.mark.parametrize("use_mask", [False, True])
@pytest.mark.parametrize("H", [50, 200])
def test_split_user_encoder_sharp_logits(H, use_mask):
    """Logits that span tens: the TF32 kernel's ~2^-11 operand rounding moves them by ~1e-3 and the user vector by more
    than 1e-4; the split kernel stays at fp32 accuracy."""
    B, D, Q = 7, 256, 200
    case = f"H{H}_mask{int(use_mask)}"
    mask = _mask(B, H, seed=H + 1)
    params = _pool_params(D, Q, seed=H, sharp=True)
    vecs = (torch.randn(B * H, D, generator=torch.Generator().manual_seed(H)) * 0.5).cuda()
    ru, _ = _ue_ref(vecs.view(B, H, D), mask, *params, use_mask)
    v = vecs.view(B, H, D).double()
    if not use_mask:
        v = v * mask.double().unsqueeze(-1) + params[0].double() * (1 - mask.double().unsqueeze(-1))
    logit = torch.tanh(v @ params[1].double().t() + params[2].double()) @ params[3].double()
    report(f"fp32_ue.sharp.logit_spread.{case}", float(logit.max() - logit.min()), None)
    tf32_user, _ = _run_ue(vecs, mask, params, use_mask, B, H, fp32=False)
    tf32_err = _rowrel(tf32_user, ru)
    report(f"fp32_ue.sharp.tf32_kernel.user.{case}", tf32_err, None)
    assert tf32_err > BOUND, tf32_err                      # the case separates the two modes
    user, _ = _run_ue(vecs, mask, params, use_mask, B, H, fp32=True)
    _chk(f"fp32_ue.sharp.split_kernel.user.{case}", _rowrel(user, ru), SHARP_BOUND)


@gpu
@pytest.mark.parametrize("R", [350, 3 * 512, 4096 * 50 // 16])
def test_split_sgemm_nt_nrms_projection(R):
    """The batched (x3) Q/K/V projection of NRMS: [R, 256] rows times [3][256, 256] weights + bias, strided as the
    flat parameter buffer lays them out."""
    import tinyrec.ops as ops
    D, Dh = 256, 256
    g = torch.Generator().manual_seed(R)
    x = torch.randn(R, D, generator=g) * 0.5
    W = torch.randn(3, Dh, D, generator=g) * (6.0 / (D + Dh)) ** 0.5
    b = torch.randn(3, Dh, generator=g) * 0.06
    out = torch.full((3, R, Dh), float("nan"), device="cuda")
    ops.sgemm_nt(x.cuda(), W.cuda(), b.cuda(), out, R, Dh, D, 3, 0, Dh * D, Dh, R * Dh, fp32=True)
    ref = torch.einsum("rd,pnd->prn", x.double(), W.double()) + b.double()[:, None, :]
    _chk(f"fp32_sgemm_nt.R{R}", _rowrel(out.view(3 * R, Dh), ref.reshape(3 * R, Dh)), GEMM_BOUND)
    tf = torch.empty(3, R, Dh, device="cuda")
    ops.sgemm_nt(x.cuda(), W.cuda(), b.cuda(), tf, R, Dh, D, 3, 0, Dh * D, Dh, R * Dh)
    report(f"fp32_sgemm_nt.tf32_kernel.R{R}", _rowrel(tf.view(3 * R, Dh), ref.reshape(3 * R, Dh)), None)


# ------------------------------------------------------------------------------------------------ modules
def _sharpen(sd, pfx, x, mask, use_mask, nrms):
    """Scale a user encoder's weights (in place) so that, on these inputs, the NRMS scores q.k / 4 and the pooling
    logits span tens: fc1 pre-activations of std 2, fc2 and W_Q / W_K chosen from the float64 forward.  x float64
    [B, H, D]; the pooling statistics are taken over all rows."""
    from oracle import model as om
    sd64 = _sd64(sd)
    if nrms:
        mp = pfx + "multi_head_self_attn."
        v = x if use_mask else x * mask.unsqueeze(-1) + sd64[pfx + "pad_doc"] * (1 - mask.unsqueeze(-1))
        q = v @ sd64[mp + "W_Q.weight"].t() + sd64[mp + "W_Q.bias"]
        k = v @ sd64[mp + "W_K.weight"].t() + sd64[mp + "W_K.bias"]
        s = (q.view(*q.shape[:2], -1, 16) * k.view(*k.shape[:2], -1, 16)).sum(-1) / 4
        f = (6.0 / float(s.std())) ** 0.5                        # q.k / 4 of std ~6: scores span tens
        for nm in ("W_Q", "W_K"):
            sd[mp + nm + ".weight"] = sd[mp + nm + ".weight"] * f
            sd[mp + nm + ".bias"] = sd[mp + nm + ".bias"] * f
        sd64 = _sd64(sd)
        x = om.multi_head_self_attn(sd64, mp, v, mask if use_mask else None)
        use_mask = True
    ap = pfx + "attn."
    pre = x @ sd64[ap + "att_fc1.weight"].t()
    sd[ap + "att_fc1.weight"] = sd[ap + "att_fc1.weight"] * (2.0 / float(pre.std()))
    w2 = sd[ap + "att_fc2.weight"]
    sd[ap + "att_fc2.weight"] = w2 * (0.6 / float(w2.std()))    # logits of std ~5 over Q = 200 tanh units
    return sd


def _model_bert(sd, layers, H, ulm, model, precision):
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    m = mb.ModelBert(synth.demo_args(num_student_layers=layers, user_log_length=H, user_log_mask=ulm, model=model,
                                     precision=precision))
    m.load_state_dict(sd, strict=True)
    return m.cuda().eval()


@gpu
@pytest.mark.parametrize("tag,ulm", [("pad", False), ("mask", True)])
def test_model_bert_fp32_user_and_score_vs_reference_golden(golden, tag, ulm):
    import tinyrec.synth as synth
    g = golden("modelbert")
    layers = int(g["layers"])
    H = g["history"].shape[1]
    m = _model_bert(synth.model_bert_state("", layers, int(g["seed"]), noisy=True), layers, H, ulm, "NAML", "fp32")
    with torch.no_grad():
        score, _, _, uv = m(torch.from_numpy(g["history"]).cuda(), torch.from_numpy(g["history_mask"]).cuda(),
                            torch.from_numpy(g["candidate"]).cuda())
    ref_u, ref_s = torch.from_numpy(g[f"user_{tag}"]).double(), torch.from_numpy(g[f"score_{tag}"]).double()
    _chk(f"fp32.golden.user_{tag}", _rowrel(uv, ref_u), BOUND)
    # A click score is a dot product, and its error scales with ||c_k|| ||u||, the size of the terms it sums.  Rows whose
    # scores cancel far below that scale (impression 1 of the pad branch: |s| ~ ||c|| ||u|| / 130, where the reference's
    # own fp32 scores are 3e-6 off float64) turn the news encoder's candidate error into a larger row-relative error:
    # recorded for every row, bounded on the rows that do not cancel; every score is bounded on the dot-product scale.
    scale = torch.from_numpy(g[f"cand_{tag}"]).double().norm(dim=-1) * ref_u.norm(dim=-1, keepdim=True)
    err = (score.double().cpu() - ref_s).abs()
    _chk(f"fp32.golden.score_{tag}.vs_term_scale", float((err / scale.clamp_min(1e-300)).max()), BOUND)
    report(f"fp32.golden.score_{tag}.row_rel_all_rows", _rowrel(score, ref_s), None)
    plain = ref_s.norm(dim=1) >= 0.1 * scale.norm(dim=1)
    assert int(plain.sum()) >= 2
    _chk(f"fp32.golden.score_{tag}.row_rel", _rowrel(score.cpu()[plain], ref_s[plain]), BOUND)
    if ulm:
        assert float(uv[1].abs().max()) == 0.0 and float(score[1].abs().max()) == 0.0    # the all-masked impression


@gpu
@pytest.mark.parametrize("ulm", [False, True])
@pytest.mark.parametrize("H", [50, 200])
@pytest.mark.parametrize("model", ["NAML", "NRMS"])
def test_model_bert_fp32_sharp_vs_float64_oracle(model, H, ulm):
    import tinyrec.synth as synth
    from oracle import model as om
    layers, B, K, L = 1, 6, 5, 16
    case = f"{model}.H{H}.ulm{int(ulm)}"
    sd = synth.model_bert_state("", layers, 11, noisy=True, model=model)
    news = synth.news_table(B * (H + K), L=L, seed=H)
    x = torch.from_numpy(news[1:].astype(np.int64))
    history, candidate = x[:B * H].view(B, H, -1), x[B * H:].view(B, K, -1)
    hmask = _mask(B, H, seed=H).cpu()
    hmask[0, :H // 3] = 0
    with torch.no_grad():
        hist64 = om.news_encoder(_sd64(sd), "news_encoder.", history.reshape(B * H, -1), layers).view(B, H, -1)
    sd = _sharpen(sd, "user_encoder.", hist64, hmask.double(), ulm, model == "NRMS")
    with torch.no_grad():
        ref = om.model_bert_forward(_sd64(sd), "", history, hmask.double(), candidate, layers, ulm)
    outs = {}
    for precision in ("fp32", "bf16"):
        m = _model_bert(sd, layers, H, ulm, model, precision)
        with torch.no_grad():
            outs[precision] = m(history.cuda(), hmask.cuda(), candidate.cuda())
    score, _, _, user = outs["fp32"]
    _chk(f"fp32.oracle64.sharp.user.{case}", _rowrel(user, ref[3]), BOUND)
    _chk(f"fp32.oracle64.sharp.score.{case}", _rowrel(score, ref[0]), BOUND)
    report(f"fp32.oracle64.sharp.bf16_mode_user.{case}", _rowrel(outs["bf16"][3], ref[3]), None)
    # the user encoder alone, on the fp32 mode's own news vectors: what the user-encoder kernels add
    m = _model_bert(sd, layers, H, ulm, model, "fp32")
    with torch.no_grad():
        hv = outs["fp32"][1]
        alone = om.user_encoder(_sd64(sd), "user_encoder.", hv.double().cpu(), hmask.double(), ulm)
        u2 = m.user_encoder(hv, hmask.cuda())
    _chk(f"fp32.oracle64.sharp.user_encoder_alone.{case}", _rowrel(u2, alone), KERNEL_BOUND)


# ------------------------------------------------------------------------------------------------ evaluate
@gpu
@pytest.mark.parametrize("ulm", [False, True])
@pytest.mark.parametrize("model", ["NAML", "NRMS"])
def test_evaluate_fp32_user_encoder_vs_float64(model, ulm):
    """``run.evaluate`` with an fp32 user encoder: its user vectors and click scores against float64, and its metrics
    against the oracle's on the float64 scores (exact, except where the float64 scores of a clicked and a non-clicked
    candidate are closer than fp32 can resolve)."""
    import tinyrec.model_bert as mb
    import tinyrec.ops as ops
    import tinyrec.run as trun
    import tinyrec.synth as synth
    from oracle import metrics as omet, model as om
    from test_drivers_gpu import _eval_problem
    H, D = 50, 256
    case = f"{model}.ulm{int(ulm)}"
    hist, hmask, ptr, cand, lab, kinds, table = _eval_problem(H=H, D=D)
    n = hist.shape[0]
    args = synth.demo_args(user_log_mask=ulm, model=model, precision="fp32")
    x64 = table.double()[torch.from_numpy(hist.astype(np.int64))]
    sd = _sharpen(synth.user_encoder_state("", D, args.user_query_vector_dim, 3, model=model), "", x64,
                  torch.from_numpy(hmask).double(), ulm, model == "NRMS")
    ue = mb.UserEncoder(args)
    ue.load_state_dict(sd, strict=True)
    ue.cuda().eval()
    tab_d = table.cuda()
    mean, total, per = trun.evaluate(ue, tab_d, hist, hmask, ptr, cand, lab, batch_size=256, return_per_impression=True)
    assert total == n
    per = per.cpu().numpy()
    with torch.no_grad():
        user = ue.forward_gather(tab_d, torch.from_numpy(hist).cuda(), torch.from_numpy(hmask).cuda())
        scores = torch.zeros(len(cand), device="cuda", dtype=torch.float32)
        per2 = torch.zeros(n, 5, device="cuda", dtype=torch.float64)
        ops.eval_metrics(tab_d, user, torch.from_numpy(ptr).cuda(), torch.from_numpy(cand).cuda(), torch.from_numpy(lab).cuda(),
                         int(np.diff(ptr).max()), per2, None, scores)
        o_user = om.user_encoder(_sd64(sd), "", x64, torch.from_numpy(hmask).double(), ulm)
    assert np.array_equal(per2.cpu().numpy()[:, :4], per[:, :4])          # the driver ran these very kernels
    _chk(f"fp32.evaluate.user.{case}", _rowrel(user, o_user), BOUND)
    ue_bf16 = mb.UserEncoder(synth.demo_args(user_log_mask=ulm, model=model))
    ue_bf16.load_state_dict(sd, strict=True)
    with torch.no_grad():
        report(f"fp32.evaluate.bf16_mode_user.{case}",
               _rowrel(ue_bf16.cuda().eval().forward_gather(tab_d, torch.from_numpy(hist).cuda(),
                                                            torch.from_numpy(hmask).cuda()), o_user), None)
    scores = scores.cpu().numpy().astype(np.float64)
    tab64, o_user = table.double().numpy(), o_user.numpy()
    worst, skipped, near = 0.0, 0, 0
    o_per = []
    for i in range(n):
        seg = slice(int(ptr[i]), int(ptr[i + 1]))
        y = lab[seg]
        o_sc = tab64[cand[seg]] @ o_user[i]
        if np.abs(o_sc).max() > 0:
            worst = max(worst, float(np.linalg.norm(scores[seg] - o_sc) / np.linalg.norm(o_sc)))
        else:
            assert not scores[seg].any()                                    # an empty history under the mask
        o_m = omet.impression_metrics(y, o_sc)
        o_per.append(o_m)
        if o_m is None:
            assert not per[i, :4].any()
            continue
        if kinds[i] == 3:                                                   # clicked and not clicked: argsort order unspecified
            skipped += 1
            continue
        gap = np.abs(o_sc[y == 1][:, None] - o_sc[y == 0][None, :]).min()
        if gap < BOUND * np.abs(o_sc).max():                                # closer than the scores' accuracy
            near += 1
            continue
        assert np.allclose(per[i, :4], o_m, rtol=0, atol=1e-12), (i, per[i], o_m)
    _chk(f"fp32.evaluate.score_row.{case}", worst, BOUND)
    report(f"fp32.evaluate.near_tie_impressions.{case}", near, None)
    assert near <= n // 20 and skipped > 0
    o_mean, _ = omet.eval_reduce(o_per, n)
    _chk(f"fp32.evaluate.mean_auc.{case}", abs(float(mean[0]) - float(o_mean[0])), 1e-4)
