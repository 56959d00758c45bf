#!/usr/bin/env python
"""bf16 vs fp32 (args.precision) news-table build: the 12-layer teacher table over the whole 161 014-row news set
through tinyrec.run.build_news_table, at L = 30 and L = 180, the two precisions alternated in one process and timed
with CUDA events.  Reports news/s, the fp32 / bf16 time ratio, and the GEMM rate (executed work: the fp32 path runs
every GEMM with K' = 3K; 'useful' divides that by 3), with the device name and power limit read in the same run.

    python tools/table_fp32_bench.py --rounds 3 --out profiles/table_fp32_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {30: dict(mean_len=14.0, std_len=4.0, min_len=4), 180: dict(mean_len=140.0, std_len=40.0, min_len=10)}
N_NEWS, LAYERS, BATCH = 161013, 12, 4096


def _device_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as exc:  # noqa: BLE001  (reported, not hidden)
        info["power_limit"] = f"unavailable: {type(exc).__name__}"
    return info


def _timed_table(trun, enc, news):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    tab = trun.build_news_table(enc, news, batch_size=BATCH, sharded=False)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3, tab


def _gemm_rate(ops, enc, x):
    """GEMM FLOP (as executed) and GEMM device time of one batch, from CUDA events around every GEMM launch."""
    ops.stats.gemm_events = []
    with torch.no_grad():
        enc(x)
    torch.cuda.synchronize()
    ev, ops.stats.gemm_events = ops.stats.gemm_events, None
    flop = sum(f for f, _, _ in ev)
    ms = sum(s.elapsed_time(e) for _, s, e in ev)
    return flop, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import tinyrec.model_bert_2 as mb2
    import tinyrec.ops as ops
    import tinyrec.run as trun
    import tinyrec.synth as synth
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    sd = synth.model_bert_state("", LAYERS, 0)
    encs = {}
    for prec in ("bf16", "fp32"):
        m = mb2.ModelBert(synth.demo_args(num_hidden_layers=LAYERS, precision=prec))
        m.load_state_dict(sd, strict=True)
        encs[prec] = m.to(dev).eval().news_encoder
    result = {"device": _device_info(), "rows": N_NEWS + 1, "layers": LAYERS, "batch_rows": BATCH, "rounds": a.rounds,
              "timing": "CUDA events around tinyrec.run.build_news_table (host int32 rows in, fp32 table out)",
              "weights": "random init (synth.model_bert_state seed 0)", "workloads": {}}
    for L, wl in WORKLOADS.items():
        news = synth.news_table(N_NEWS, L=L, seed=1234, **wl)
        times = {"bf16": [], "fp32": []}
        for prec in ("bf16", "fp32"):                     # warm-up: workspaces, weight images, module load
            _timed_table(trun, encs[prec], news[:2 * BATCH])
        tabs = {}
        for _ in range(a.rounds):
            for prec in ("bf16", "fp32"):
                s, tabs[prec] = _timed_table(trun, encs[prec], news)
                times[prec].append(s)
        diff = (tabs["fp32"].double() - tabs["bf16"].double()).norm(dim=1) / tabs["fp32"].double().norm(dim=1)
        x = torch.from_numpy(news[1:BATCH + 1]).to(dev).to(torch.int64)
        w = {"bf16_vs_fp32_max_row_rel": float(diff.max())}
        for prec in ("bf16", "fp32"):
            best = min(times[prec])
            flop, gms = _gemm_rate(ops, encs[prec], x)
            w[prec] = {"seconds": times[prec], "news_per_sec_best": (N_NEWS + 1) / best,
                       "gemm_tflops_executed": flop / (gms * 1e-3) / 1e12, "gemm_ms_per_batch": gms,
                       "gemm_tflop_executed_per_batch": flop / 1e12}
            if prec == "fp32":
                w[prec]["gemm_tflops_useful"] = w[prec]["gemm_tflops_executed"] / 3
        w["fp32_over_bf16_time"] = min(times["fp32"]) / min(times["bf16"])
        result["workloads"][f"L{L}"] = w
        del tabs
        torch.cuda.empty_cache()
    txt = json.dumps(result, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
