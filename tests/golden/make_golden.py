#!/usr/bin/env python
"""Generate tests/golden/*.npz from the REAL reference code.

Run in the build container only (needs /root/reference):
    python tests/golden/make_golden.py

The reference modules (Tiny-NewsRec/model_bert.py, model_bert_2.py,
tnlrv3/modeling.py, metrics.py, dataloader.py) are imported through
``ref_shim`` and executed on CPU fp32 in ``eval()`` mode; weights come from
``tinyrec.synth`` (deterministic per (seed, key)) and are loaded with
``load_state_dict(strict=True)``, which also pins the state_dict key names.
Fixtures hold inputs + reference outputs (+ a weight checksum), never weights.
"""
import os
import random
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import ref_shim  # noqa: E402
import tinyrec.synth as synth  # noqa: E402

ref_modeling = ref_shim.install()
import model_bert as ref_mb  # noqa: E402
import model_bert_2 as ref_mb2  # noqa: E402
import metrics as ref_metrics  # noqa: E402

torch.set_grad_enabled(True)


def checksum(sd):
    return np.array([float(v.double().sum()) for v in sd.values()], dtype=np.float64)


def rand_news(rng, n, L, all_pad_row=None, full_row=None):
    lens = rng.integers(2, L + 1, size=n)
    if full_row is not None:
        lens[full_row] = L
    ids = rng.integers(1000, 30522, size=(n, L))
    mask = (np.arange(L)[None, :] < lens[:, None]).astype(np.int64)
    ids = ids * mask
    ids[:, 0] = 101 * mask[:, 0]
    if all_pad_row is not None:
        ids[all_pad_row] = 0
        mask[all_pad_row] = 0
    return np.concatenate([ids, mask], axis=1).astype(np.int64)


def grad_summary(name, g):
    g = g.detach()
    out = {f"gsum/{name}": np.float64(g.double().sum()), f"gabs/{name}": np.float64(g.double().abs().sum())}
    if g.numel() <= 4096:
        out[f"gfull/{name}"] = g.numpy().astype(np.float32)
    else:
        out[f"gslice/{name}"] = g[:16, :16].numpy().astype(np.float32)
    return out


def gen_relpos():
    rel = torch.arange(-600, 601)
    b = ref_modeling.relative_position_bucket(rel, num_buckets=32, max_distance=128)
    np.savez_compressed(os.path.join(HERE, "relpos.npz"), rel=rel.numpy(), bucket=b.numpy())


def gen_encoder():
    seed, layers, n, L = 7, 2, 5, 12
    args = ref_shim.make_args(num_student_layers=layers)
    ne = ref_mb.NewsEncoder(args, is_teacher=False).eval()
    sd = synth.model_bert_state("", layers, seed, noisy=True)
    sd = {k[len("news_encoder."):]: v for k, v in sd.items() if k.startswith("news_encoder.")}
    ne.load_state_dict(sd, strict=True)
    rng = np.random.default_rng(11)
    x = rand_news(rng, n, L, all_pad_row=3, full_row=0)
    xt = torch.from_numpy(x)
    with torch.no_grad():
        vec = ne(xt)
        outs = ne.bert_model(xt[:, :L], xt[:, L:])
        hidden = torch.stack(outs[3], 0)           # [layers+1, n, L, E]
    np.savez_compressed(os.path.join(HERE, "encoder.npz"), seed=seed, layers=layers, x=x,
                        news_vec=vec.numpy(), hidden=hidden.numpy().astype(np.float32),
                        wsum=checksum(sd))


def gen_modelbert():
    seed, layers, B, H, K, L = 3, 1, 3, 4, 2, 10
    rng = np.random.default_rng(5)
    hist = rand_news(rng, B * H, L).reshape(B, H, 2 * L)
    cand = rand_news(rng, B * K, L).reshape(B, K, 2 * L)
    hmask = np.array([[0, 0, 1, 1], [0, 0, 0, 0], [1, 1, 1, 1]], dtype=np.float32)
    hist[0, :2] = 0
    hist[1, :] = 0
    out = dict(seed=seed, layers=layers, history=hist, candidate=cand, history_mask=hmask)
    sd = synth.model_bert_state("", layers, seed, noisy=True)
    for ulm in (False, True):
        args = ref_shim.make_args(num_student_layers=layers, user_log_length=H, user_log_mask=ulm)
        m = ref_mb.ModelBert(args, is_teacher=False).eval()
        m.load_state_dict(sd, strict=True)
        with torch.no_grad():
            score, hv, cv, uv = m(torch.from_numpy(hist), torch.from_numpy(hmask), torch.from_numpy(cand))
        tag = "mask" if ulm else "pad"
        out.update({f"score_{tag}": score.numpy(), f"hist_{tag}": hv.numpy(), f"cand_{tag}": cv.numpy(),
                    f"user_{tag}": uv.numpy()})
    # PLM-NR / teacher form with CE loss (model_bert_2.py:192-213)
    args = ref_shim.make_args(num_hidden_layers=layers, user_log_length=H, user_log_mask=False)
    m2 = ref_mb2.ModelBert(args).eval()
    m2.load_state_dict(sd, strict=True)
    label = np.array([1, 0, 1], dtype=np.int64)
    with torch.no_grad():
        loss, score = m2(torch.from_numpy(hist), torch.from_numpy(hmask), torch.from_numpy(cand),
                         torch.from_numpy(label))
    out.update(plmnr_label=label, plmnr_loss=np.float64(loss), plmnr_score=score.numpy(), wsum=checksum(sd))
    np.savez_compressed(os.path.join(HERE, "modelbert.npz"), **out)


def gen_kd():
    seed, layers, M, B, H, K, L, D = 9, 2, 3, 3, 4, 3, 9, 256
    trainable = [1]
    rng = np.random.default_rng(21)
    hist = rand_news(rng, B * H, L).reshape(B, H, 2 * L)
    cand = rand_news(rng, B * K, L).reshape(B, K, 2 * L)
    hmask = np.array([[0, 1, 1, 1], [0, 0, 0, 1], [1, 1, 1, 1]], dtype=np.float32)
    hist[0, :1] = 0
    hist[1, :3] = 0
    label = np.array([2, 0, 1], dtype=np.int64)
    th = [rng.standard_normal((B, H, D)).astype(np.float32) * 0.3 for _ in range(M)]
    tc = [rng.standard_normal((B, K, D)).astype(np.float32) * 0.3 for _ in range(M)]
    out = dict(seed=seed, layers=layers, M=M, history=hist, candidate=cand, history_mask=hmask, label=label,
               trainable=np.array(trainable), temperature=2.0, coef=0.2,
               **{f"th{i}": th[i] for i in range(M)}, **{f"tc{i}": tc[i] for i in range(M)})
    sd = synth.kd_model_state(layers, M, seed, noisy=True)
    for ulm in (False, True):
        args = ref_shim.make_args(num_student_layers=layers, user_log_length=H, user_log_mask=ulm,
                                  num_teachers=M, temperature=2.0, coef=0.2)
        m = ref_mb.Model(args).eval()
        m.load_state_dict(sd, strict=True)
        # freeze policy of run.py:101-112
        for p in m.teachers.parameters():
            p.requires_grad = False
        for p in m.student.news_encoder.bert_model.parameters():
            p.requires_grad = False
        for i, layer in enumerate(m.student.news_encoder.bert_model.bert.encoder.layer):
            if i in trainable:
                for p in layer.parameters():
                    p.requires_grad = True
        res = m(torch.from_numpy(hist), torch.from_numpy(hmask), torch.from_numpy(cand),
                torch.from_numpy(label), [torch.from_numpy(t) for t in th], [torch.from_numpy(t) for t in tc])
        tag = "mask" if ulm else "pad"
        for nm, v in zip(("total", "distill", "emb", "target"), res[:4]):
            out[f"{nm}_{tag}"] = np.float64(v.detach())
        out[f"score_{tag}"] = res[4].detach().numpy()
        if not ulm:
            res[0].backward()
            names = []
            for nm, p in m.named_parameters():
                if p.requires_grad:
                    names.append(nm)
                    out.update(grad_summary(nm, p.grad))
            out["trainable_names"] = np.array(names)
    out["wsum"] = checksum(sd)
    np.savez_compressed(os.path.join(HERE, "kd.npz"), **out)


def gen_metrics():
    from sklearn.metrics import roc_auc_score
    rng = np.random.default_rng(99)
    ptr, scores, labels, vals = [0], [], [], []
    for i in range(60):
        C = int(rng.integers(2, 70))
        s = rng.standard_normal(C).astype(np.float32)
        if i % 3 == 0:
            s = np.round(s, 1)               # ties
        if i % 10 == 9 and C <= 16:
            s[:] = 0.5                       # all tied
        y = (rng.random(C) < 0.2).astype(np.int64)
        if i == 7:
            y[:] = 0                         # skipped impression (run.py:348)
        elif i == 8:
            y[:] = 1
        elif y.sum() == 0:
            y[0] = 1
        elif y.sum() == C:
            y[0] = 0
        if y.mean() == 0 or y.mean() == 1:
            vals.append([np.nan] * 4)
        else:
            vals.append([roc_auc_score(y, s), ref_metrics.mrr_score(y, s), ref_metrics.ndcg_score(y, s, k=5),
                         ref_metrics.ndcg_score(y, s, k=10)])
        scores.append(s)
        labels.append(y)
        ptr.append(ptr[-1] + C)
    np.savez_compressed(os.path.join(HERE, "metrics.npz"), ptr=np.array(ptr), score=np.concatenate(scores),
                        label=np.concatenate(labels), vals=np.array(vals, dtype=np.float64))


def gen_auc_ties():
    """scikit-learn's roc_auc_score (metrics.py:1) on the 200 random tie-heavy cases that
    test_oracle_auc_matches_installed_sklearn_on_random_ties draws from default_rng(0)."""
    from sklearn.metrics import roc_auc_score
    rng = np.random.default_rng(0)
    ptr, scores, labels, auc = [0], [], [], []
    for _ in range(200):
        n = int(rng.integers(2, 60))
        y = (rng.random(n) < 0.3).astype(np.int64)
        if y.min() == y.max():
            y[0], y[1] = 0, 1
        s = np.round(rng.standard_normal(n), 1).astype(np.float32)
        auc.append(roc_auc_score(y, s))
        scores.append(s)
        labels.append(y)
        ptr.append(ptr[-1] + n)
    np.savez_compressed(os.path.join(HERE, "auc_ties.npz"), ptr=np.array(ptr), score=np.concatenate(scores),
                        label=np.concatenate(labels), auc=np.array(auc, dtype=np.float64))


def gen_adam():
    g = torch.Generator().manual_seed(4)
    p = torch.randn(1000, generator=g)
    p0 = p.clone()
    p.requires_grad_(True)
    opt = torch.optim.Adam([p], lr=1e-4, amsgrad=True)          # run.py:134
    grads, ps = [], []
    for step in range(5):
        gr = torch.randn(1000, generator=g) * (10.0 if step == 1 else 0.1)   # spike so vmax matters
        p.grad = gr.clone()
        opt.step()
        grads.append(gr.numpy())
        ps.append(p.detach().clone().numpy())
    np.savez_compressed(os.path.join(HERE, "adam.npz"), p0=p0.numpy(), grads=np.stack(grads), params=np.stack(ps))


def gen_batching():
    """dataloader.py needs `streaming` -> tensorflow; a stub module is enough because
    only the numpy/python batch assembly (`_process`) is exercised."""
    tf = types.ModuleType("tensorflow")
    tf.io = types.SimpleNamespace(gfile=types.SimpleNamespace())
    sys.modules.setdefault("tensorflow", tf)
    import dataloader as ref_dl
    rng = np.random.default_rng(3)
    n_news, L, D, M, H, npratio = 40, 6, 8, 2, 5, 4
    news_index = {f"N{i}": i for i in range(1, n_news + 1)}
    news_combined = rng.integers(0, 1000, size=(n_news + 1, 2 * L)).astype(np.int32)
    news_combined[0] = 0
    teacher = [rng.standard_normal((n_news + 1, D)).astype(np.float32) for _ in range(M)]
    args = types.SimpleNamespace(npratio=npratio, user_log_length=H, batch_size=4, shuffle_buffer_size=1,
                                 num_teachers=M)
    dl = ref_dl.DataLoaderTrain(data_dir="", filename_pat="", args=args, world_size=1, worker_rank=0,
                                cuda_device_idx=0, news_index=news_index, news_combined=news_combined,
                                teacher_embs=teacher, word_dict=None, enable_gpu=False)
    lines, clicks_all, pos_all, neg_all = [], [], [], []
    for b in range(4):
        nclick = [0, 3, 5, 9][b]
        clicks = [f"N{int(i)}" for i in rng.integers(1, n_news + 1, size=nclick)]
        if b == 1:
            clicks[1] = "NX_unknown"
        pos = [f"N{int(rng.integers(1, n_news + 1))}"]
        neg = [f"N{int(i)}" for i in rng.integers(1, n_news + 1, size=npratio)]
        clicks_all.append(" ".join(clicks)); pos_all.append(pos[0]); neg_all.append(" ".join(neg))
        lines.append("\t".join(["0", "U1", "t", " ".join(clicks), " ".join(pos), " ".join(neg)]).encode())
    random.seed(123)
    uf, lm, nf, lab, thb, tcb = dl._process(lines)
    np.savez_compressed(
        os.path.join(HERE, "batching.npz"), news_combined=news_combined, t0=teacher[0], t1=teacher[1],
        clicks=np.array(clicks_all), pos=np.array(pos_all), neg=np.array(neg_all), H=H, npratio=npratio,
        user_feature=uf.numpy(), log_mask=lm.numpy(), news_feature=nf.numpy(), label=lab.numpy(),
        th0=thb[0].numpy(), th1=thb[1].numpy(), tc0=tcb[0].numpy(), tc1=tcb[1].numpy())


def gen_unilm_convert():
    """A UniLM-format state dict (fused qkv_linear, q_bias / v_bias, encoder.rel_pos_bias) through the
    reference's converter and position-table resize logic (tnlrv3/convert_state_dict.py:39-71,
    tnlrv3/modeling.py:88-118 restated inline there; here the converter is called directly)."""
    import tnlrv3.convert_state_dict as ref_conv
    g = torch.Generator().manual_seed(11)
    E, A, layers = 16, 2, 2
    sd = {"bert.embeddings.word_embeddings.weight": torch.randn(50, E, generator=g),
          "bert.embeddings.position_embeddings.weight": torch.randn(12, E, generator=g),
          "bert.encoder.rel_pos_bias.weight": torch.randn(A, 32, generator=g)}
    for l in range(layers):
        pfx = f"bert.encoder.layer.{l}.attention.self."
        sd[pfx + "qkv_linear.weight"] = torch.randn(3 * E, E, generator=g)
        sd[pfx + "q_bias"] = torch.randn(1, 1, E, generator=g)
        sd[pfx + "v_bias"] = torch.randn(1, 1, E, generator=g)
        sd[f"bert.encoder.layer.{l}.output.dense.weight"] = torch.randn(E, 4 * E, generator=g)
    out = ref_conv.state_dict_convert["tnlrv3"]({k: v.clone() for k, v in sd.items()})
    fix = {"in/" + k: v.numpy() for k, v in sd.items()}
    fix.update({"out/" + k: v.numpy() for k, v in out.items()})
    fix["out_keys"] = np.array(list(out.keys()))
    np.savez_compressed(os.path.join(HERE, "unilm_convert.npz"), **fix)


def gen_nrms():
    """KD ``Model`` with the NRMS user encoders (args.model = 'NRMS': 16-head exp-normalised self-attention
    over the history in front of the additive pooling, model_bert.py:37-100,145-148,162-164,171-173), both
    ``user_log_mask`` branches, losses + scores + gradients of every trainable tensor."""
    seed, layers, M, B, H, K, L, D = 13, 1, 2, 3, 5, 3, 8, 256
    rng = np.random.default_rng(31)
    hist = rand_news(rng, B * H, L).reshape(B, H, 2 * L)
    cand = rand_news(rng, B * K, L).reshape(B, K, 2 * L)
    hmask = np.array([[0, 0, 1, 1, 1], [0, 0, 0, 0, 1], [1, 1, 1, 1, 1]], dtype=np.float32)
    hist[0, :2] = 0
    hist[1, :4] = 0
    label = np.array([1, 2, 0], dtype=np.int64)
    th = [rng.standard_normal((B, H, D)).astype(np.float32) * 0.3 for _ in range(M)]
    tc = [rng.standard_normal((B, K, D)).astype(np.float32) * 0.3 for _ in range(M)]
    out = dict(seed=seed, layers=layers, M=M, history=hist, candidate=cand, history_mask=hmask, label=label,
               temperature=1.5, coef=0.3,
               **{f"th{i}": th[i] for i in range(M)}, **{f"tc{i}": tc[i] for i in range(M)})
    sd = synth.kd_model_state(layers, M, seed, noisy=True, model="NRMS", n_heads=16)
    for ulm in (False, True):
        args = ref_shim.make_args(num_student_layers=layers, user_log_length=H, user_log_mask=ulm, num_teachers=M,
                                  temperature=1.5, coef=0.3, model="NRMS", num_attention_heads=16)
        m = ref_mb.Model(args).eval()
        assert list(m.state_dict().keys()) == list(sd.keys())
        m.load_state_dict(sd, strict=True)
        for p in m.teachers.parameters():
            p.requires_grad = False
        for p in m.student.news_encoder.bert_model.parameters():
            p.requires_grad = False
        for p in m.student.news_encoder.bert_model.bert.encoder.layer[0].parameters():
            p.requires_grad = True
        res = m(torch.from_numpy(hist), torch.from_numpy(hmask), torch.from_numpy(cand),
                torch.from_numpy(label), [torch.from_numpy(t) for t in th], [torch.from_numpy(t) for t in tc])
        tag = "mask" if ulm else "pad"
        for nm, v in zip(("total", "distill", "emb", "target"), res[:4]):
            out[f"{nm}_{tag}"] = np.float64(v.detach())
        out[f"score_{tag}"] = res[4].detach().numpy()
        m.zero_grad()
        res[0].backward()
        names = []
        for nm, p in m.named_parameters():
            if p.requires_grad and p.grad is not None:       # pad_doc has no gradient in the user_log_mask branch
                names.append(nm)
                out.update({f"{tag}/{k}": v for k, v in grad_summary(nm, p.grad).items()})
        out[f"trainable_names_{tag}"] = np.array(names)
    out["wsum"] = checksum(sd)
    out["state_keys"] = np.array(list(sd.keys()))
    np.savez_compressed(os.path.join(HERE, "nrms.npz"), **out)


def gen_post_train():
    """``TitleBodySimModel`` of Domian-specific_Post-train.ipynb, built by EXECUTING the notebook's own cells 10-11
    (AttentionPooling / NewsEncoder / TitleBodySimModel) through the shim: 12-layer encoder as the cell hard-codes,
    1+K titles and one body per sample through the same encoder, CE over the title scores.  Pins the two-pass
    title / body path that ``tinyrec.post_train`` runs (the first-stage KD wrapper of Post-train_KD.ipynb shares it;
    its cell 14 is not runnable as published)."""
    import json
    import shutil
    import tempfile
    import torch.nn.functional as F_
    from torch import nn as nn_
    from utils import MODEL_CLASSES
    nb = json.load(open(os.path.join(ref_shim.REF_ROOT, "Domian-specific_Post-train.ipynb")))
    tmp = tempfile.mkdtemp()
    shutil.copy(os.path.join(ref_shim.REF_ROOT, "Tiny-NewsRec/tnlrv3/config/tnlrv3-base-uncased-config.json"),
                os.path.join(tmp, "unilm2-base-uncased-config.json"))
    ns = dict(nn=nn_, torch=torch, F=F_, os=os, np=np, MODEL_CLASSES=MODEL_CLASSES, path_turing=tmp)
    for c in (10, 11):
        exec("".join(nb["cells"][c]["source"]), ns)
    seed, layers, B, K1, Lt, Lb = 17, 12, 2, 3, 8, 40
    rng = np.random.default_rng(41)
    title = rand_news(rng, B * K1, Lt).reshape(B, K1, 2 * Lt)
    body = rand_news(rng, B, Lb, full_row=0)
    labels = np.array([2, 0], dtype=np.int64)
    args = types.SimpleNamespace(news_query_vector_dim=200, news_dim=256)
    m = ns["TitleBodySimModel"](args).eval()
    full = synth.model_bert_state("", layers, seed, noisy=True)
    sd = {k: v for k, v in full.items() if k.startswith("news_encoder.")}
    assert list(m.state_dict().keys()) == list(sd.keys())
    m.load_state_dict(sd, strict=True)
    for p in m.news_encoder.bert_model.parameters():
        p.requires_grad = False
    for i in (10, 11):
        for p in m.news_encoder.bert_model.bert.encoder.layer[i].parameters():
            p.requires_grad = True
    scores, loss = m(torch.from_numpy(title), torch.from_numpy(body), torch.from_numpy(labels))
    loss.backward()
    out = dict(seed=seed, layers=layers, title=title, body=body, labels=labels, scores=scores.detach().numpy(),
               loss=np.float64(loss.detach()), trainable=np.array([10, 11]))
    names = []
    for nm, p in m.named_parameters():
        if p.requires_grad and p.grad is not None:
            names.append(nm)
            out.update(grad_summary(nm, p.grad))
    out["trainable_names"] = np.array(names)
    out["wsum_head"] = checksum({k: v for k, v in sd.items() if ".attn." in k or ".dense." in k})
    np.savez_compressed(os.path.join(HERE, "post_train.npz"), **out)
    shutil.rmtree(tmp)


if __name__ == "__main__":
    gen_relpos()
    gen_encoder()
    gen_modelbert()
    gen_kd()
    gen_metrics()
    gen_auc_ties()
    gen_adam()
    gen_batching()
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))
    gen_unilm_convert()
    gen_nrms()
    gen_post_train()
