#!/usr/bin/env python
"""Cost of full-encoder fine-tuning on the kd4 workload (bench.py: B 32, H 50, K 5, L 30, M 4, 4-layer student).

1. The graphed train step (tinyrec.run.GraphedTrainStep over the device loader's index batches) for three
   requires_grad policies, alternated round by round in one process:
     ref    -- the reference's policy (run.py:101-112): layers {2, 3} trainable;
     all    -- everything in the student encoder trainable;
     bottom -- the embedding block and rel_pos_bias trainable, every layer frozen.
2. Device-event times of the embedding backward (tnr_embed_ln_bwd: word, position, token-type tables and the
   LayerNorm) and of the attention backward with the rel-pos bias gradient (tnr_attn_relpos_bwd_drel) against the one
   without it (tnr_attn_relpos_bwd), at L = 30 and L = 100 on the kd4 news rows (1 760 rows per step).  For the
   embedding backward also GB/s over its algorithmic bytes: dy read (T E 2), word-row re-read (T E 2) and the
   read-modify-write of the touched fp32 gradient rows (2 U E 4, U = distinct non-zero ids), and that rate as a
   fraction of 7.7 TB/s.
The card's name and power limit are read in the same run (nvidia-smi --query-gpu, read-only).

    python tools/full_finetune_bench.py --rounds 3 --steps 20 --out profiles/full_finetune_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK = 7.7e12


def _device_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as exc:  # noqa: BLE001  (reported, not hidden)
        info["power_limit"] = f"unavailable: {type(exc).__name__}"
    return info


def _set_policy(model, policy):
    bm = model.student.news_encoder.bert_model
    for p in bm.parameters():
        p.requires_grad = policy == "all"
    if policy == "ref":
        for i in (2, 3):
            for p in bm.bert.encoder.layer[i].parameters():
                p.requires_grad = True
    if policy == "bottom":
        for p in bm.bert.embeddings.parameters():
            p.requires_grad = True
        bm.bert.rel_pos_bias.weight.requires_grad = True


def _events(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def step_times(rounds, steps):
    import bench
    import tinyrec.optim as topt
    import tinyrec.run as trun
    dev = torch.device("cuda", 0)
    batcher, dev_batches, _ = bench.make_inputs(0, dev)
    runs = {}
    for policy in ("ref", "all", "bottom"):
        model, _ = bench.make_model(4, [2, 3], dev)
        _set_policy(model, policy)
        opt = topt.Adam(model, lr=1e-5)
        g = trun.GraphedTrainStep(model, opt, dev_batches[0], warmup=3, batcher=batcher)
        runs[policy] = (model, g)
    ms = {p: [] for p in runs}
    for _ in range(rounds):
        for p, (_, g) in runs.items():
            it = iter(range(10 ** 9))
            _events(lambda: g(*dev_batches[next(it) % len(dev_batches)]), 3)          # re-warm after the other policies
            ms[p].append(_events(lambda: g(*dev_batches[next(it) % len(dev_batches)]), steps))
    out = {}
    for p, v in ms.items():
        st = runs[p][0].train_state()
        out[p] = {"ms_per_step": v, "median_ms": float(np.median(v)), "trainable_floats": int(st.flat.numel)}
    return out, batcher, dev_batches


def kernel_times(batcher, dev_batches, steps):
    import bench
    import tinyrec.ops as ops
    import tinyrec.synth as synth
    from tinyrec.engine import rel_pos_bucket_table
    dev = torch.device("cuda", 0)
    E, A, vocab = 768, 12, 30522
    g = torch.Generator(device=dev).manual_seed(7)
    word = (torch.randn(vocab, E, generator=g, device=dev) * 0.05).to(torch.bfloat16)
    pos = torch.randn(512, E, generator=g, device=dev) * 0.05
    typ = torch.randn(2, E, generator=g, device=dev) * 0.05
    gamma = 1 + 0.1 * torch.randn(E, generator=g, device=dev)
    seed = torch.tensor([11], device=dev, dtype=torch.int64)
    out = {}
    for L in (30, 100):
        if L == bench.L:
            hist_idx, _, cand_idx, _ = dev_batches[0]
            history, candidate, _, _ = batcher.assemble(hist_idx, cand_idx)
            x = torch.cat([history.reshape(-1, 2 * L), candidate.reshape(-1, 2 * L)], 0).contiguous()
        else:
            x = torch.from_numpy(synth.news_table(bench.B * (bench.H + bench.K) - 1, L=L, seed=3).astype(np.int64)).to(dev)
        n = x.shape[0]
        T = n * L
        ids = x[:, :L]
        U = int(torch.unique(ids[ids != 0]).numel())
        dy = (torch.randn(T, E, generator=g, device=dev) * 0.01).to(torch.bfloat16)
        dword = torch.zeros(vocab, E, device=dev)
        dpos = torch.zeros(512, E, device=dev)
        dtyp = torch.zeros(2, E, device=dev)
        dg, db = torch.zeros(E, device=dev), torch.zeros(E, device=dev)
        drop = ops.make_drop(seed, 0, 0.1)
        emb = lambda: ops.embed_ln_bwd(x, L, word, pos, typ[0], gamma, 1e-12, dy, dword=dword, dpos=dpos,  # noqa: E731
                                       dtype0=dtyp[0], dgamma=dg, dbeta=db, drop=drop)
        emb_word_only = lambda: ops.embed_ln_bwd(x, L, word, pos, typ[0], gamma, 1e-12, dy, dword=dword, drop=drop)  # noqa: E731
        for f in (emb, emb_word_only):
            _events(f, 3)
        t_emb = _events(emb, steps)
        t_word = _events(emb_word_only, steps)
        algo_bytes = T * E * 2 + T * E * 2 + 2 * U * E * 4
        qkv = (torch.randn(T, 3 * E, generator=g, device=dev) * 0.5).to(torch.bfloat16)
        dctx = torch.randn(T, E, generator=g, device=dev).to(torch.bfloat16)
        dqkv = torch.empty_like(qkv)
        tab = rel_pos_bucket_table(L)
        bucket = torch.cat([tab[1:, 0].flip(0), tab[0, :]]).to(device=dev, dtype=torch.int32)
        relpos = torch.randn(A, 2 * L - 1, generator=g, device=dev)
        drel = torch.zeros(A, 32, device=dev)
        dbias = torch.zeros(3 * E, device=dev)
        adrop = ops.make_drop(seed, 13, 0.1)
        plain = lambda: ops.attn_bwd(qkv, x, L, relpos, dctx, dqkv, A, drop=adrop, dbias=dbias)  # noqa: E731
        withrel = lambda: ops.attn_bwd_drel(qkv, x, L, relpos, dctx, dqkv, A, bucket, drel, drop=adrop, dbias=dbias)  # noqa: E731
        for f in (plain, withrel):
            _events(f, 3)
        tp, tr = [], []
        for _ in range(3):                                        # alternated
            tp.append(_events(plain, steps))
            tr.append(_events(withrel, steps))
        out[f"L{L}"] = {
            "news_rows": n, "tokens": T, "distinct_nonpad_ids": U, "pad_fraction": float((ids == 0).float().mean()),
            "embed_bwd_ms": t_emb, "embed_bwd_word_only_ms": t_word,
            "embed_bwd_algorithmic_bytes": algo_bytes,
            "embed_bwd_GBps": algo_bytes / (t_emb * 1e-3) / 1e9,
            "embed_bwd_fraction_of_7.7TBps": algo_bytes / (t_emb * 1e-3) / HBM_PEAK,
            "attn_bwd_ms": float(np.median(tp)), "attn_bwd_drel_ms": float(np.median(tr)),
            "attn_bwd_ms_rounds": tp, "attn_bwd_drel_ms_rounds": tr,
        }
        print(json.dumps({f"L{L}": out[f"L{L}"]}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("full_finetune_bench: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    result = {"device": _device_info(), "workload": "kd4: B 32, H 50, K 5, L 30, M 4, 4-layer student, graphed step"}
    steps, batcher, dev_batches = step_times(a.rounds, a.steps)
    print(json.dumps({"step": steps}), flush=True)
    result["step"] = steps
    result["kernels"] = kernel_times(batcher, dev_batches, a.steps * 5)
    txt = json.dumps(result, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
