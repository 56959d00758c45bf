#!/usr/bin/env python
"""Long user histories (user_log_length = H): the graphed KD train step at the kd4 configuration (4 layers, layers
{2, 3} trainable, B = 32, K = 5, L = 30, M = 4) at H = 50, 100, 200, and eval scoring (gather + user encoder + ranking
metrics over 4 096-impression batches from a precomputed 161 014-row news table) at H = 50, 100, 200, 512 for NAML
and NRMS.  Everything is device-timed with CUDA events.  The user-encoder share of each is the user-encoder launches
alone on the same inputs (train: the student + 4 teacher forward in one launch and the student backward; eval:
UserEncoder.forward_gather), also timed with CUDA events, over the time of the whole step.  The device name and power
limit are read in the same run.

    python tools/long_history_bench.py --out profiles/long_history_bench.json
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

N_NEWS, D, B, K, L, M, LAYERS, TRAINABLE = 161013, 256, 32, 5, 30, 4, 4, [2, 3]
N_BATCHES, EVAL_IMPS = 8, 4096


def _device_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as exc:  # noqa: BLE001  (reported, not hidden)
        info["power_limit"] = f"unavailable: {type(exc).__name__}"
    return info


def _timed(fn, n):
    """ms per call of fn over n calls, CUDA events around the whole window."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def bench_train(H, steps, warmup):
    import tinyrec.dataloader as dl
    import tinyrec.model_bert as mb
    import tinyrec.ops as ops
    import tinyrec.optim as topt
    import tinyrec.run as trun
    import tinyrec.synth as synth
    device = torch.device("cuda", 0)
    args = synth.demo_args(num_student_layers=LAYERS, num_teachers=M, bert_trainable_layer=TRAINABLE, user_log_length=H)
    torch.manual_seed(0)
    model = mb.Model(args)
    model.load_state_dict(synth.kd_model_state(LAYERS, M, 0), strict=True)
    model.to(device)
    for p in model.teachers.parameters():
        p.requires_grad = False
    bm = model.student.news_encoder.bert_model
    for p in bm.parameters():
        p.requires_grad = False
    for i, layer in enumerate(bm.bert.encoder.layer):
        if i in TRAINABLE:
            for p in layer.parameters():
                p.requires_grad = True
    opt = topt.Adam(model, lr=1e-4)
    news = synth.news_table(N_NEWS, L=L, seed=1234)
    g = torch.Generator(device=device).manual_seed(4321)
    tables = dl.DeviceTables(news, [], device)
    tables.teachers = [(torch.randn(N_NEWS + 1, D, generator=g, device=device) * 0.1) for _ in range(M)]
    hist_idx, hmask, cand_idx, label = synth.train_impressions(B * N_BATCHES, N_NEWS, H, K, seed=1234)
    batcher = dl.TrainBatcher(tables, B, H, K)
    batches = [tuple(torch.from_numpy(np.ascontiguousarray(a[i * B:(i + 1) * B])).to(device)
                     for a in (hist_idx, hmask, cand_idx, label)) for i in range(N_BATCHES)]
    gstep = trun.GraphedTrainStep(model, opt, batches[0], warmup=max(warmup, 3), batcher=batcher)
    for i in range(warmup):
        gstep(*batches[i % N_BATCHES])
    step_ms = _timed(lambda i: gstep(*batches[i % N_BATCHES]), steps)
    # the user-encoder launches of one step on the same shapes: student + M teacher encoders forward, student backward
    ue = model.student.user_encoder.attn
    Q = ue.att_fc1.weight.shape[0]
    vecs = [torch.randn(B * H, D, device=device) * 0.1 for _ in range(M + 1)]
    mask = batches[0][1].float().contiguous()
    pad = model.student.user_encoder.pad_doc.detach().view(-1)
    W1, b1 = ue.att_fc1.weight.detach(), ue.att_fc1.bias.detach()
    w2, b2 = ue.att_fc2.weight.detach().view(-1), ue.att_fc2.bias.detach()
    encs = [dict(vecs=v, pad_doc=pad, W1=W1, b1=b1, w2=w2, b2=b2, user=torch.empty(B, D, device=device),
                 a=torch.empty(B, H, device=device), e=torch.empty(B, H, Q, device=device) if i == 0 else None)
            for i, v in enumerate(vecs)]
    d_user, d_vecs = torch.randn(B, D, device=device), torch.zeros(B * H, D, device=device)
    grads = [torch.zeros(D, device=device), torch.zeros(Q, D, device=device), torch.zeros(Q, device=device),
             torch.zeros(Q, device=device), torch.zeros(1, device=device)]
    scratch = torch.empty(B * H * (Q + D), device=device)

    def ue_calls(_):
        ops.user_encoder_fwd_multi(encs, mask, False, B, H)
        ops.user_encoder_bwd(vecs[0], mask, pad, W1, w2, False, encs[0]["a"], encs[0]["e"], d_user, d_vecs, *grads,
                             scratch, B, H)
    for i in range(warmup):
        ue_calls(i)
    ue_ms = _timed(ue_calls, steps)
    return dict(H=H, step_ms=round(step_ms, 4), user_encoder_ms=round(ue_ms, 4), user_encoder_share=round(ue_ms / step_ms, 4))


def bench_eval(model_name, H, steps, warmup):
    import tinyrec.model_bert as mb
    import tinyrec.ops as ops
    import tinyrec.synth as synth
    device = torch.device("cuda", 0)
    args = synth.demo_args(model=model_name, user_log_length=H)
    ue = mb.UserEncoder(args)
    ue.load_state_dict(synth.user_encoder_state("", D, args.user_query_vector_dim, 0, model=model_name), strict=True)
    ue.to(device).eval()
    g = torch.Generator(device=device).manual_seed(4321)
    table = torch.randn(N_NEWS + 1, D, generator=g, device=device) * 0.1
    hist, hmask, ptr, cand, lab = synth.eval_impressions(EVAL_IMPS * N_BATCHES, N_NEWS, H, seed=1234)
    batches = []
    for b in range(N_BATCHES):
        s0, s1 = b * EVAL_IMPS, (b + 1) * EVAL_IMPS
        p0, p1 = int(ptr[s0]), int(ptr[s1])
        batches.append(tuple(torch.from_numpy(np.ascontiguousarray(t)).to(device) for t in
                             (hist[s0:s1], hmask[s0:s1], ptr[s0:s1 + 1] - p0, cand[p0:p1], lab[p0:p1]))
                       + (int(np.diff(ptr[s0:s1 + 1]).max()),))
    per = torch.zeros(EVAL_IMPS, 5, device=device, dtype=torch.float64)
    sums = torch.zeros(5, device=device, dtype=torch.float64)

    @torch.no_grad()
    def score(i):
        hi_t, hm_t, ptr_t, cand_t, lab_t, max_c = batches[i % N_BATCHES]
        user = ue.forward_gather(table, hi_t, hm_t)
        ops.eval_metrics(table, user, ptr_t, cand_t, lab_t, max_c, per, sums)

    @torch.no_grad()
    def user_only(i):
        hi_t, hm_t = batches[i % N_BATCHES][:2]
        ue.forward_gather(table, hi_t, hm_t)
    for i in range(warmup):
        score(i)
        user_only(i)
    ms = _timed(score, steps)
    ue_ms = _timed(user_only, steps)
    return dict(model=model_name, H=H, batch_ms=round(ms, 4), impressions_per_s=round(EVAL_IMPS / ms * 1e3, 1),
                user_encoder_ms=round(ue_ms, 4), user_encoder_share=round(ue_ms / ms, 4))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--train-h", type=int, nargs="*", default=[50, 100, 200])
    ap.add_argument("--eval-h", type=int, nargs="*", default=[50, 100, 200, 512])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("long_history_bench: no CUDA device (there is no CPU measurement)")
    import __graft_entry__
    __graft_entry__.build()
    res = dict(device=_device_info(), steps=a.steps, warmup=a.warmup,
               train=dict(config=f"kd4: {LAYERS} layers, trainable {TRAINABLE}, B={B}, K={K}, L={L}, M={M}, graphed step",
                          rows=[]),
               eval=dict(config=f"{EVAL_IMPS}-impression batches, {N_NEWS + 1}-row fp32 news table, D={D}", rows=[]))
    for H in a.train_h:
        res["train"]["rows"].append(bench_train(H, a.steps, a.warmup))
        print(json.dumps(res["train"]["rows"][-1]), flush=True)
        torch.cuda.empty_cache()
    for model_name in ("NAML", "NRMS"):
        for H in a.eval_h:
            res["eval"]["rows"].append(bench_eval(model_name, H, a.steps, a.warmup))
            print(json.dumps(res["eval"]["rows"][-1]), flush=True)
            torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
