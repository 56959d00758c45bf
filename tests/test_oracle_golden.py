"""Pin the oracle (oracle/) against vectors produced by the real reference code
(tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

import oracle
from oracle import model as om, metrics as omet, batching as ob, optim as oopt
import tinyrec.synth as synth

# The fixtures were recorded with 8 torch intra-op threads.  Some pinned gradients vanish in exact arithmetic (the
# attention key bias and the additive-attention output bias: a constant added to every logit of a softmax row cancels),
# so their recorded values are fp32 rounding noise that depends on how the reductions are split over threads; with
# any other thread count the split, and the noise, differ.
FIXTURE_THREADS = 8


@pytest.fixture(autouse=True)
def _fixture_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(FIXTURE_THREADS)
    yield
    torch.set_num_threads(n)


def _wsum(sd):
    return np.array([float(v.double().sum()) for v in sd.values()], dtype=np.float64)


def _check_weights(sd, g):
    np.testing.assert_allclose(_wsum(sd), g["wsum"], rtol=1e-12, atol=1e-9,
                               err_msg="synthetic weights differ from the ones the fixture was made with")


def test_relpos_bucket(golden):
    g = golden("relpos")
    b = om.rel_pos_bucket(torch.from_numpy(g["rel"]))
    assert np.array_equal(b.numpy(), g["bucket"])


def test_relpos_table_matches_onehot_linear():
    w = torch.randn(12, 32)
    L = 30
    t = om.rel_pos_bias_table(w, L)
    pos = torch.arange(L)
    rel = pos[None, :] - pos[:, None]
    onehot = torch.nn.functional.one_hot(om.rel_pos_bucket(rel), 32).float()
    ref = torch.nn.functional.linear(onehot, w).permute(2, 0, 1)
    assert torch.equal(t, ref)


def test_encoder_hidden_and_news_vec(golden):
    g = golden("encoder")
    layers = int(g["layers"])
    sd = synth.model_bert_state("", layers, int(g["seed"]), noisy=True)
    sd = {k[len("news_encoder."):]: v for k, v in sd.items() if k.startswith("news_encoder.")}
    _check_weights(sd, g)
    x = torch.from_numpy(g["x"])
    L = x.shape[1] // 2
    with torch.no_grad():
        hs = om.bert_last_hidden(sd, "bert_model.", x[:, :L], x[:, L:], layers, all_hidden=True)
        vec = om.news_encoder(sd, "", x, layers)
    np.testing.assert_allclose(torch.stack(hs, 0).numpy(), g["hidden"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(vec.numpy(), g["news_vec"], rtol=1e-4, atol=2e-5)
    assert np.isfinite(vec.numpy()).all()          # all-pad row stays finite


@pytest.mark.parametrize("tag,ulm", [("pad", False), ("mask", True)])
def test_model_bert_forward(golden, tag, ulm):
    g = golden("modelbert")
    layers = int(g["layers"])
    sd = synth.model_bert_state("", layers, int(g["seed"]), noisy=True)
    _check_weights(sd, g)
    with torch.no_grad():
        score, hv, cv, uv = om.model_bert_forward(
            sd, "", torch.from_numpy(g["history"]), torch.from_numpy(g["history_mask"]),
            torch.from_numpy(g["candidate"]), layers, ulm)
    for got, key in ((score, "score"), (hv, "hist"), (cv, "cand"), (uv, "user")):
        np.testing.assert_allclose(got.numpy(), g[f"{key}_{tag}"], rtol=1e-4, atol=2e-5)
    if ulm:   # fully masked history -> exactly zero user vector (0 / (0 + 1e-8))
        assert np.all(uv.numpy()[1] == 0.0)


def test_plmnr_loss(golden):
    g = golden("modelbert")
    layers = int(g["layers"])
    sd = synth.model_bert_state("", layers, int(g["seed"]), noisy=True)
    with torch.no_grad():
        loss, score = om.plmnr_forward(sd, torch.from_numpy(g["history"]), torch.from_numpy(g["history_mask"]),
                                       torch.from_numpy(g["candidate"]), torch.from_numpy(g["plmnr_label"]),
                                       layers, False)
    np.testing.assert_allclose(float(loss), float(g["plmnr_loss"]), rtol=1e-5)
    np.testing.assert_allclose(score.numpy(), g["plmnr_score"], rtol=1e-4, atol=2e-5)


def _kd_inputs(g):
    M = int(g["M"])
    th = [torch.from_numpy(g[f"th{i}"]) for i in range(M)]
    tc = [torch.from_numpy(g[f"tc{i}"]) for i in range(M)]
    return (torch.from_numpy(g["history"]), torch.from_numpy(g["history_mask"]), torch.from_numpy(g["candidate"]),
            torch.from_numpy(g["label"]), th, tc)


@pytest.mark.parametrize("tag,ulm", [("pad", False), ("mask", True)])
def test_kd_forward(golden, tag, ulm):
    g = golden("kd")
    layers, M = int(g["layers"]), int(g["M"])
    sd = synth.kd_model_state(layers, M, int(g["seed"]), noisy=True)
    _check_weights(sd, g)
    with torch.no_grad():
        res = om.kd_model_forward(sd, *_kd_inputs(g), layers, ulm, float(g["temperature"]), float(g["coef"]))
    for v, nm in zip(res[:4], ("total", "distill", "emb", "target")):
        np.testing.assert_allclose(float(v), float(g[f"{nm}_{tag}"]), rtol=2e-5)
    np.testing.assert_allclose(res[4].numpy(), g[f"score_{tag}"], rtol=1e-4, atol=2e-5)


def test_kd_gradients_and_freeze_policy(golden):
    g = golden("kd")
    layers, M = int(g["layers"]), int(g["M"])
    sd = synth.kd_model_state(layers, M, int(g["seed"]), noisy=True)
    keys = om.trainable_keys(sd, [int(i) for i in g["trainable"]])
    assert keys == [str(s) for s in g["trainable_names"]]
    for k in keys:
        sd[k].requires_grad_(True)
    total = om.kd_model_forward(sd, *_kd_inputs(g), layers, False, float(g["temperature"]), float(g["coef"]))[0]
    total.backward()
    for k in keys:
        gr = sd[k].grad
        np.testing.assert_allclose(float(gr.double().sum()), float(g[f"gsum/{k}"]), rtol=2e-3, atol=1e-6)
        np.testing.assert_allclose(float(gr.double().abs().sum()), float(g[f"gabs/{k}"]), rtol=1e-4)
        if f"gfull/{k}" in g.files:
            np.testing.assert_allclose(gr.numpy(), g[f"gfull/{k}"], rtol=1e-3, atol=1e-7)
        else:
            np.testing.assert_allclose(gr[:16, :16].numpy(), g[f"gslice/{k}"], rtol=1e-3, atol=1e-7)


def test_metrics(golden):
    g = golden("metrics")
    ptr = g["ptr"]
    n_skip = 0
    for i in range(len(ptr) - 1):
        s, y = g["score"][ptr[i]:ptr[i + 1]], g["label"][ptr[i]:ptr[i + 1]]
        m = omet.impression_metrics(y, s)
        if np.isnan(g["vals"][i, 0]):
            assert m is None
            n_skip += 1
        else:
            np.testing.assert_allclose(np.array(m), g["vals"][i], rtol=1e-12, atol=1e-12)
    assert n_skip == 2


def test_eval_reduce_divides_by_all_impressions():
    mean, sums = omet.eval_reduce([(1.0, 0.5, 0.5, 0.5), None, (0.0, 0.5, 0.25, 0.25)], 3)
    np.testing.assert_allclose(sums, [1.0, 1.0, 0.75, 0.75])
    np.testing.assert_allclose(mean, sums / 3.0)


def test_adam_amsgrad(golden):
    g = golden("adam")
    p = torch.from_numpy(g["p0"].copy())
    m, v, vmax = torch.zeros_like(p), torch.zeros_like(p), torch.zeros_like(p)
    for step in range(g["grads"].shape[0]):
        oopt.adam_amsgrad_step(p, torch.from_numpy(g["grads"][step]), m, v, vmax, step + 1, lr=1e-4)
        np.testing.assert_allclose(p.numpy(), g["params"][step], rtol=1e-6, atol=1e-7)


def test_batching_bit_exact(golden):
    import random
    g = golden("batching")
    H, npratio = int(g["H"]), int(g["npratio"])
    n_news = g["news_combined"].shape[0] - 1
    news_index = {f"N{i}": i for i in range(1, n_news + 1)}
    random.seed(123)
    hist_idx, masks, cand_idx, labels = [], [], [], []
    for clicks, pos, neg in zip(g["clicks"], g["pos"], g["neg"]):
        idx, mask = ob.pad_history(ob.to_index(str(clicks).split(), news_index), H)
        label = random.randint(0, npratio)                      # dataloader.py:135
        cand = ob.insert_positive(ob.to_index([str(pos)], news_index),
                                  ob.to_index(str(neg).split(), news_index), label)
        hist_idx.append(idx); masks.append(mask); cand_idx.append(cand); labels.append(label)
    hist, cand, th, tc = ob.train_batch(np.array(hist_idx), np.array(cand_idx), g["news_combined"],
                                        [g["t0"], g["t1"]])
    assert np.array_equal(hist, g["user_feature"])
    assert np.array_equal(cand, g["news_feature"])
    assert np.array_equal(np.array(masks, dtype=np.float32), g["log_mask"])
    assert np.array_equal(np.array(labels), g["label"])
    for i in range(2):
        assert np.array_equal(th[i], g[f"th{i}"])
        assert np.array_equal(tc[i], g[f"tc{i}"])


def test_shard_round_robin():
    assert ob.shard_round_robin(7, 1, 3) == [1, 4]


# ------------------------------------------------------------------ NRMS user encoder (SURVEY 8f rank 2)
@pytest.mark.parametrize("tag,ulm", [("pad", False), ("mask", True)])
def test_nrms_kd_forward_and_gradients(golden, tag, ulm):
    """Oracle vs the reference ``Model`` with args.model = 'NRMS' (fixture: make_golden.py:gen_nrms)."""
    g = golden("nrms")
    layers, M = int(g["layers"]), int(g["M"])
    sd = synth.kd_model_state(layers, M, int(g["seed"]), noisy=True, model="NRMS", n_heads=16)
    assert list(sd.keys()) == [str(k) for k in g["state_keys"]]                 # reference state_dict order
    _check_weights(sd, g)
    keys = [str(s) for s in g[f"trainable_names_{tag}"]]
    for k in keys:
        sd[k].requires_grad_(True)
    res = om.kd_model_forward(sd, *_kd_inputs(g), layers, ulm, float(g["temperature"]), float(g["coef"]))
    for v, nm in zip(res[:4], ("total", "distill", "emb", "target")):
        np.testing.assert_allclose(float(v), float(g[f"{nm}_{tag}"]), rtol=2e-5)
    np.testing.assert_allclose(res[4].detach().numpy(), g[f"score_{tag}"], rtol=1e-4, atol=2e-5)
    res[0].backward()
    for k in keys:
        gr = sd[k].grad
        np.testing.assert_allclose(float(gr.double().abs().sum()), float(g[f"{tag}/gabs/{k}"]), rtol=2e-4, atol=1e-9)
        if f"{tag}/gfull/{k}" in g.files:
            np.testing.assert_allclose(gr.numpy(), g[f"{tag}/gfull/{k}"], rtol=2e-3, atol=2e-7)


# ------------------------------------------------------------------ post-training title / body model (SURVEY 8f rank 3)
def test_domain_post_train_forward_and_gradients(golden):
    """Oracle vs ``TitleBodySimModel`` of Domian-specific_Post-train.ipynb, executed from the notebook's own cells
    (fixture: make_golden.py:gen_post_train): 12-layer encoder, titles and body through the same encoder, CE."""
    g = golden("post_train")
    layers = int(g["layers"])
    full = synth.model_bert_state("", layers, int(g["seed"]), noisy=True)
    sd = {k: v for k, v in full.items() if k.startswith("news_encoder.")}
    keys = [str(s) for s in g["trainable_names"]]
    for k in keys:
        sd[k].requires_grad_(True)
    scores, loss = om.domain_post_train_forward(sd, torch.from_numpy(g["title"]), torch.from_numpy(g["body"]),
                                                torch.from_numpy(g["labels"]), layers)
    np.testing.assert_allclose(scores.detach().numpy(), g["scores"], rtol=2e-5, atol=2e-4)
    np.testing.assert_allclose(float(loss.detach()), float(g["loss"]), rtol=1e-4, atol=1e-5)
    loss.backward()
    for k in keys:
        gr = sd[k].grad
        np.testing.assert_allclose(float(gr.double().abs().sum()), float(g[f"gabs/{k}"]), rtol=5e-4, atol=1e-9)
        if f"gfull/{k}" in g.files:
            np.testing.assert_allclose(gr.numpy(), g[f"gfull/{k}"], rtol=5e-3, atol=1e-6)


def test_oracle_auc_matches_installed_sklearn_on_random_ties(golden):
    """The tie-aware Mann-Whitney restatement of ``roc_auc_score`` (metrics.py:1 -- third-party, unpinned) against
    scikit-learn on random scores with many ties: the values it returned when the fixture was made
    (make_golden.py:gen_auc_ties), and the installed scikit-learn where there is one; then the doc-sim loop against a
    vectorised formula."""
    import importlib.util
    import random
    g = golden("auc_ties")
    sk = None
    if importlib.util.find_spec("sklearn") is not None:
        import sklearn.metrics as sk
    rng = np.random.default_rng(0)
    for i in range(200):
        n = int(rng.integers(2, 60))
        y = (rng.random(n) < 0.3).astype(np.int64)
        if y.min() == y.max():
            y[0], y[1] = 0, 1
        s = np.round(rng.standard_normal(n), 1).astype(np.float32)       # rounding makes ties common
        lo, hi = g["ptr"][i], g["ptr"][i + 1]
        assert np.array_equal(y, g["label"][lo:hi]) and np.array_equal(s, g["score"][lo:hi])
        np.testing.assert_allclose(omet.auc(y, s), g["auc"][i], atol=1e-12)
        if sk is not None:
            np.testing.assert_allclose(omet.auc(y, s), sk.roc_auc_score(y, s), atol=1e-12)
    table = rng.standard_normal((30, 16)).astype(np.float32)
    got = omet.doc_sim(table, 400, random.Random(5))
    r = random.Random(5)
    tot = 0.0
    for _ in range(400):
        i, j = r.randrange(1, 30), r.randrange(1, 30)
        if i != j:
            tot += float(table[i] @ table[j]) / (float(np.linalg.norm(table[i])) * float(np.linalg.norm(table[j])))
    assert abs(got - tot / 400) < 1e-6
