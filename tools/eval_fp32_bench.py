#!/usr/bin/env python
"""bf16- vs fp32-mode (args.precision) user encoders in eval scoring: batches of 4 096 impressions scored from a
161 014-row fp32 news table (UserEncoder.forward_gather + tnr_eval_metrics, as tinyrec.run.evaluate runs them), for
NAML and NRMS at H = 50 and 200, the two modes alternated in one process.  Reports impressions/s (CUDA events around
whole batches), the device time of every user-encoder op per batch (CUDA events around each op, in a separate pass),
the bf16 / fp32 user-vector difference, and the device name and power limit read in the same run.

In bf16 mode the NAML pooling is the tcgen05 TF32 scoring GEMM (tnr_user_encoder_score); in fp32 mode it is the 3xTF32
per-impression kernel (tnr_user_encoder_fwd_gather_f32, or tnr_user_encoder_fwd_f32 behind the NRMS attention).

    python tools/eval_fp32_bench.py --rounds 3 --steps 16 --out profiles/eval_fp32_bench.json
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

N_NEWS, D, IMPS, N_BATCHES = 161013, 256, 4096, 4
USER_OPS = ("user_encoder_score", "user_encoder_fwd_gather", "user_encoder_fwd", "gather_rows_f32", "nrms_blend_fwd",
            "sgemm_nt", "nrms_attn_fwd")


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
    ap.add_argument("--steps", type=int, default=16, help="batches per timed window")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import tinyrec.model_bert as mb
    import tinyrec.ops as ops
    import tinyrec.synth as synth
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(4321)
    table = torch.randn(N_NEWS + 1, D, generator=g, device=dev) * 0.1
    result = {"device": _device_info(), "table_rows": N_NEWS + 1, "news_dim": D, "impressions_per_batch": IMPS,
              "rotating_batches": N_BATCHES, "rounds": a.rounds, "batches_per_window": a.steps,
              "timing": "CUDA events around forward_gather + eval_metrics per window; per-op events in a separate pass",
              "weights": "random init (synth.user_encoder_state seed 0)", "workloads": {}}
    for model in ("NAML", "NRMS"):
        sd = synth.user_encoder_state("", D, 200, 0, model=model)
        for H in (50, 200):
            hist, hmask, ptr, cand, lab = synth.eval_impressions(IMPS * N_BATCHES, N_NEWS, H, seed=1234)
            batches = []
            for b in range(N_BATCHES):
                s0, s1 = b * IMPS, (b + 1) * IMPS
                p0, p1 = int(ptr[s0]), int(ptr[s1])
                batches.append((torch.from_numpy(hist[s0:s1]).to(dev), torch.from_numpy(hmask[s0:s1]).to(dev),
                                torch.from_numpy(ptr[s0:s1 + 1] - p0).to(dev), torch.from_numpy(cand[p0:p1]).to(dev),
                                torch.from_numpy(lab[p0:p1]).to(dev), int(np.diff(ptr[s0:s1 + 1]).max())))
            per = torch.zeros(IMPS, 5, device=dev, dtype=torch.float64)
            sums = torch.zeros(5, device=dev, dtype=torch.float64)
            ues = {}
            for prec in ("bf16", "fp32"):
                ue = mb.UserEncoder(synth.demo_args(model=model, user_log_length=H, precision=prec))
                ue.load_state_dict(sd, strict=True)
                ues[prec] = ue.to(dev).eval()

            @torch.no_grad()
            def score(ue, bt):
                hi_t, hm_t, ptr_t, cand_t, lab_t, max_c = bt
                user = ue.forward_gather(table, hi_t, hm_t)
                ops.eval_metrics(table, user, ptr_t, cand_t, lab_t, max_c, per, sums)
                return user

            def window(ue):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for i in range(a.steps):
                    score(ue, batches[i % N_BATCHES])
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / 1e3

            for prec in ("bf16", "fp32"):                      # warm-up: module load, workspaces, packed weights
                for i in range(N_BATCHES):
                    score(ues[prec], batches[i])
            times = {"bf16": [], "fp32": []}
            for _ in range(a.rounds):
                for prec in ("bf16", "fp32"):
                    times[prec].append(window(ues[prec]))
            w = {}
            users = {}
            for prec in ("bf16", "fp32"):
                ops.stats.op_events = []
                for i in range(N_BATCHES):
                    users[prec] = score(ues[prec], batches[i])
                torch.cuda.synchronize()
                ev, ops.stats.op_events = ops.stats.op_events, None
                per_op = {}
                for name, _, s_, e_ in ev:
                    if name in USER_OPS:
                        per_op[name] = per_op.get(name, 0.0) + s_.elapsed_time(e_) / N_BATCHES
                best = min(times[prec])
                w[prec] = {"seconds_per_window": times[prec], "impressions_per_sec_best": IMPS * a.steps / best,
                           "ms_per_batch_best": best * 1e3 / a.steps, "user_encoder_ms_per_batch": per_op,
                           "user_encoder_ms_per_batch_total": sum(per_op.values())}
            u32, u16 = users["fp32"].double(), users["bf16"].double()
            w["bf16_vs_fp32_user_max_row_rel"] = float(((u16 - u32).norm(dim=1) /
                                                        u32.norm(dim=1).clamp_min(1e-300)).max())
            w["fp32_over_bf16_time"] = min(times["fp32"]) / min(times["bf16"])
            result["workloads"][f"{model}_H{H}"] = w
            print(json.dumps({f"{model}_H{H}": w}), flush=True)
            del batches, ues, users
            torch.cuda.empty_cache()
    txt = json.dumps(result, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
