#!/usr/bin/env python
"""Filtered top-k recommendation (tinyrec.ops.recommend_pool / recommend_topk with a candidate pool, per-user
exclusions and per-user categories) on the 161 014-row fp32 table of ``bench.py --workload eval`` (randn * 0.1,
D = 256), NAML user encoder (random init), batches of 4 096 users, k = 10 and 64.  CUDA events per stage; the cases
alternate batch by batch within a round.

Rows (each: stage 1 / stage 2 / total device ms, users/s, stage-1 candidates per user, exact-pass users):
- unfiltered: the call without filters, users from ``synth.eval_impressions`` at H = 50;
- pool_rand10 / pool_window1: a random 10 % pool and a contiguous 1 % window.  The pool build
  (tnr_recommend_pool + the row gather, once per call) is timed separately, and torch.matmul (TF32 allowed) +
  torch.topk over ``user @ pool_table.T`` is the baseline (no history exclusion, not the eval scores: a baseline only);
- categories_1of18: 18 categories, each user allowed one;
- exclude_E512: 512 random exclusions per user;
- long_history_H512: H = 512 with every slot live, no other filter (``--long-only`` runs only this row, and
  ``--package-root`` imports the package from another checkout, so the same row can be timed on an older tree).
The device name and power limit are read in the same run.

    python tools/recommend_filter_bench.py            # writes profiles/recommend_filter_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

N_NEWS, D, H, USERS, N_BATCHES = 161013, 256, 50, 4096, 4


def _device_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as exc:  # noqa: BLE001  (reported, not hidden)
        info["power_limit"] = f"unavailable: {type(exc).__name__}"
    return info


def _encoder(H_, dev):
    import tinyrec.model_bert as mb
    import tinyrec.synth as synth
    args = synth.demo_args(user_log_length=H_)
    ue = mb.UserEncoder(args)
    ue.load_state_dict(synth.user_encoder_state("", D, 200, 0), strict=True)
    return ue.to(dev).eval()


def _batches(ue, table, hist, mask, dev):
    out = []
    with torch.no_grad():
        for i in range(N_BATCHES):
            hi_t = torch.from_numpy(np.ascontiguousarray(hist[i * USERS:(i + 1) * USERS])).to(dev)
            hm_t = torch.from_numpy(np.ascontiguousarray(mask[i * USERS:(i + 1) * USERS])).to(dev)
            out.append((ue.forward_gather(table, hi_t, hm_t), hi_t, hm_t))
    return out


def _time_cases(ops, table, batches, cases, k, rounds):
    """cases: name -> (kwargs per batch index, baseline table or None).  Median device ms over rounds x batches."""
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    for name, (kw, base_t) in cases.items():                   # warm-up of every shape
        for i, (user, hi_t, hm_t) in enumerate(batches):
            ops.recommend_topk(table, user, hi_t, hm_t, k, **kw(i))
            if base_t is not None:
                torch.topk(torch.matmul(user, base_t.t()), min(k, base_t.shape[0]), dim=1)
    torch.cuda.synchronize()
    rec = {name: dict(s1=[], s2=[], tot=[], base=[], cmean=[], cmax=[], fb=0) for name in cases}
    for _ in range(rounds):
        for i, (user, hi_t, hm_t) in enumerate(batches):
            for name, (kw, base_t) in cases.items():
                r = rec[name]
                e = [ev(), ev(), ev()]
                _, _, info = ops.recommend_topk(table, user, hi_t, hm_t, k, events=e, **kw(i))
                b0, b1 = ev(), ev()
                if base_t is not None:
                    b0.record()
                    torch.topk(torch.matmul(user, base_t.t()), min(k, base_t.shape[0]), dim=1)
                    b1.record()
                torch.cuda.synchronize()
                r["s1"].append(e[0].elapsed_time(e[1]))
                r["s2"].append(e[1].elapsed_time(e[2]))
                r["tot"].append(e[0].elapsed_time(e[2]))
                if base_t is not None:
                    r["base"].append(b0.elapsed_time(b1))
                inf = info.cpu().numpy()
                c = inf[1:][inf[1:] >= 0]
                r["cmean"].append(float(c.mean()) if len(c) else 0.0)
                r["cmax"].append(int(c.max()) if len(c) else 0)
                r["fb"] += int(inf[0])
    med = lambda x: float(np.median(x))  # noqa: E731
    out = {}
    for name, r in rec.items():
        w = {"stage1_ms": med(r["s1"]), "stage2_ms": med(r["s2"]), "recommend_ms": med(r["tot"]),
             "users_per_s": USERS / (med(r["tot"]) / 1e3), "spread_recommend_ms": [min(r["tot"]), max(r["tot"])],
             "candidates_per_user_mean": float(np.mean(r["cmean"])), "candidates_per_user_max": int(max(r["cmax"])),
             "exact_pass_users": r["fb"]}
        if r["base"]:
            w["baseline_matmul_topk_ms"] = med(r["base"])
            w["speedup_vs_baseline"] = med(r["base"]) / med(r["tot"])
        out[name] = w
    return out


def _time_pool(ops, table, cand, rounds):
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    ops.recommend_pool(table, cand)
    ts = []
    for _ in range(rounds * N_BATCHES):
        e0, e1 = ev(), ev()
        e0.record()
        pool = ops.recommend_pool(table, cand)                 # includes the one host sync (the pool size)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return pool, {"pool_build_ms": float(np.median(ts)), "pool_rows": int(pool.size),
                  "spread_pool_build_ms": [min(ts), max(ts)]}


def _long_history(ops, table, dev, rounds):
    Hl = 512
    rng = np.random.default_rng(12)
    n = USERS * N_BATCHES
    hist = rng.integers(1, N_NEWS + 1, size=(n, Hl)).astype(np.int32)
    mask = np.ones((n, Hl), dtype=np.float32)
    batches = _batches(_encoder(Hl, dev), table, hist, mask, dev)
    return {f"k{k}": _time_cases(ops, table, batches, {"long_history_H512": (lambda i: {}, None)}, k,
                                 rounds)["long_history_H512"] for k in (10, 64)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "recommend_filter_bench.json"))
    ap.add_argument("--long-only", action="store_true", help="time only the H = 512 full-history row")
    ap.add_argument("--package-root", default=ROOT, help="checkout whose tinyrec package is imported")
    a = ap.parse_args()
    sys.path.insert(0, os.path.abspath(a.package_root))
    import tinyrec.ops as ops
    import tinyrec.synth as synth
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    table = torch.randn(N_NEWS + 1, D, generator=torch.Generator(device=dev).manual_seed(4321), device=dev) * 0.1
    result = {"device": _device_info(), "package_root": os.path.relpath(os.path.abspath(a.package_root), ROOT),
              "table_rows": N_NEWS + 1, "news_dim": D, "users_per_batch": USERS, "rotating_batches": N_BATCHES,
              "rounds": a.rounds,
              "timing": "CUDA events, median over rounds x batches; cases alternate batch by batch; the 165 MB table "
                        "exceeds L2, so every unfiltered batch reads it from HBM at least once"}
    torch.backends.cuda.matmul.allow_tf32 = True
    if not a.long_only:
        hist, mask, _, _, _ = synth.eval_impressions(USERS * N_BATCHES, N_NEWS, H, seed=11)
        batches = _batches(_encoder(H, dev), table, hist, mask, dev)
        rng = np.random.default_rng(5)
        rand10 = rng.random(N_NEWS + 1) < 0.1
        window = np.zeros(N_NEWS + 1, dtype=bool)
        w0 = N_NEWS // 3
        window[w0:w0 + (N_NEWS + 1) // 100] = True
        pool10, build10 = _time_pool(ops, table, rand10, a.rounds)
        pool1, build1 = _time_pool(ops, table, window, a.rounds)
        cat = torch.from_numpy(rng.integers(0, 18, size=N_NEWS + 1))
        cat_pool = ops.recommend_pool(table, None, cat)
        one = rng.integers(0, 18, size=USERS * N_BATCHES)
        masks = torch.from_numpy((np.uint64(1) << one.astype(np.uint64)).view(np.int64)).to(dev)
        excl = torch.from_numpy(rng.integers(1, N_NEWS + 1, size=(USERS * N_BATCHES, 512)).astype(np.int32)).to(dev)
        sl = lambda t, i: t[i * USERS:(i + 1) * USERS].contiguous()  # noqa: E731
        cases = {"unfiltered": (lambda i: {}, table),
                 "pool_rand10": (lambda i: {"pool": pool10}, pool10.table),
                 "pool_window1": (lambda i: {"pool": pool1}, pool1.table),
                 "categories_1of18": (lambda i: {"pool": cat_pool, "user_categories": sl(masks, i)}, None),
                 "exclude_E512": (lambda i: {"exclude": sl(excl, i)}, None)}
        for k in (10, 64):
            rows = _time_cases(ops, table, batches, cases, k, a.rounds)
            rows["pool_rand10"].update(build10)
            rows["pool_window1"].update(build1)
            result[f"k{k}"] = rows
            print(json.dumps({f"k{k}": rows}), flush=True)
    result["long_history_H512"] = _long_history(ops, table, dev, a.rounds)
    print(json.dumps({"long_history_H512": result["long_history_H512"]}), flush=True)
    txt = json.dumps(result, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
