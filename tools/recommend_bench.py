#!/usr/bin/env python
"""Top-k recommendation over the whole news table (tinyrec.ops.recommend_topk / tinyrec.run.recommend) on the
161 014-row fp32 table of ``bench.py --workload eval`` (randn * 0.1, D = 256), users from ``synth.eval_impressions`` at
H = 50 (NAML user encoder, random init), batches of 4 096 users, k = 10 and 64.

Per batch: users/s of the two recommendation stages (CUDA events around both), stage 1 (TF32 tcgen05 candidate
selection) and stage 2 (exact merge) device times, stage 1's executed TF32 rate over 2 B (N+1) D against the 1 125
TFLOP/s dense TF32 data-sheet figure, and the mean / largest stage-1 candidate count per user.  Baseline, alternated with
the new path in the same process: torch.matmul with TF32 allowed, then torch.topk (no history exclusion, and not the
eval scores: a baseline only).  Then ``run.recommend`` end to end (user encoding, staging, both stages) over 376 471
users.  The device name and power limit are read in the same run.

    python tools/recommend_bench.py            # writes profiles/recommend_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_NEWS, D, H, USERS, N_BATCHES, ALL_USERS = 161013, 256, 50, 4096, 4, 376471
TF32_PEAK = 1125e12


def _device_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as exc:  # noqa: BLE001  (reported, not hidden)
        info["power_limit"] = f"unavailable: {type(exc).__name__}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "recommend_bench.json"))
    ap.add_argument("--skip-whole-set", action="store_true")
    a = ap.parse_args()
    import tinyrec.model_bert as mb
    import tinyrec.ops as ops
    import tinyrec.run as trun
    import tinyrec.synth as synth
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    table = torch.randn(N_NEWS + 1, D, generator=torch.Generator(device=dev).manual_seed(4321), device=dev) * 0.1
    args = synth.demo_args(user_log_length=H)
    ue = mb.UserEncoder(args)
    ue.load_state_dict(synth.user_encoder_state("", D, 200, 0), strict=True)
    ue.to(dev).eval()
    hist, mask, _, _, _ = synth.eval_impressions(ALL_USERS, N_NEWS, H, seed=11)
    batches = []
    with torch.no_grad():
        for i in range(N_BATCHES):
            hi_t = torch.from_numpy(hist[i * USERS:(i + 1) * USERS]).to(dev)
            hm_t = torch.from_numpy(mask[i * USERS:(i + 1) * USERS]).to(dev)
            batches.append((ue.forward_gather(table, hi_t, hm_t), hi_t, hm_t))
    flops = 2.0 * USERS * (N_NEWS + 1) * D
    result = {"device": _device_info(), "table_rows": N_NEWS + 1, "news_dim": D, "history": H, "users_per_batch": USERS,
              "rotating_batches": N_BATCHES, "rounds": a.rounds,
              "timing": "CUDA events; the new path and the torch baseline alternate batch by batch; the 165 MB table "
                        "exceeds L2, so every batch reads it from HBM at least once",
              "flop_per_batch": flops, "tf32_datasheet_tflops": TF32_PEAK / 1e12, "k": {}}
    torch.backends.cuda.matmul.allow_tf32 = True
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    for k in (10, 64):
        for user, hi_t, hm_t in batches:            # warm-up of every shape
            ops.recommend_topk(table, user, hi_t, hm_t, k)
            torch.topk(torch.matmul(user, table.t()), k, dim=1)
        torch.cuda.synchronize()
        s1, s2, tot, base, cand_mean, cand_max, fb = [], [], [], [], [], [], 0
        for _ in range(a.rounds):
            for user, hi_t, hm_t in batches:
                e = [ev(), ev(), ev()]
                _, _, info = ops.recommend_topk(table, user, hi_t, hm_t, k, events=e)
                b0, b1 = ev(), ev()
                b0.record()
                torch.topk(torch.matmul(user, table.t()), k, dim=1)
                b1.record()
                torch.cuda.synchronize()
                s1.append(e[0].elapsed_time(e[1]))
                s2.append(e[1].elapsed_time(e[2]))
                tot.append(e[0].elapsed_time(e[2]))
                base.append(b0.elapsed_time(b1))
                inf = info.cpu().numpy()
                c = inf[1:][inf[1:] >= 0]
                cand_mean.append(float(c.mean()))
                cand_max.append(int(c.max()))
                fb += int(inf[0])
        med = lambda x: float(np.median(x))  # noqa: E731
        w = {"stage1_ms": med(s1), "stage2_ms": med(s2), "recommend_ms": med(tot),
             "users_per_s": USERS / (med(tot) / 1e3),
             "stage1_tflops": flops / (med(s1) / 1e3) / 1e12,
             "stage1_share_of_tf32_datasheet": flops / (med(s1) / 1e3) / TF32_PEAK,
             "candidates_per_user_mean": float(np.mean(cand_mean)), "candidates_per_user_max": int(max(cand_max)),
             "exact_pass_users": fb,
             "baseline_matmul_topk_ms": med(base), "baseline_users_per_s": USERS / (med(base) / 1e3),
             "speedup_vs_baseline": med(base) / med(tot),
             "spread_recommend_ms": [float(min(tot)), float(max(tot))], "spread_baseline_ms": [float(min(base)), float(max(base))]}
        result["k"][str(k)] = w
        print(json.dumps({f"k{k}": w}), flush=True)
    if not a.skip_whole_set:
        for k in (10, 64):
            trun.recommend(ue, table, hist[:USERS], mask[:USERS], k)     # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            trun.recommend(ue, table, hist, mask, k)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            result[f"whole_set_k{k}"] = {"users": ALL_USERS, "seconds": dt, "users_per_s": ALL_USERS / dt,
                                         "what": "run.recommend end to end: host staging, user encoding, both stages"}
            print(json.dumps({f"whole_set_k{k}": result[f"whole_set_k{k}"]}), flush=True)
    txt = json.dumps(result, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
