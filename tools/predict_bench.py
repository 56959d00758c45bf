#!/usr/bin/env python
"""Prediction files (tinyrec.run.predict + write_prediction) on the 161 014-row fp32 table of ``bench.py --workload
eval`` (randn * 0.1, D = 256), NAML user encoder (random init), H = 50, default batch size (16 384 impressions).

Two impression sets from ``synth.eval_impressions`` (C ~ clip(round(LogNormal(3.2, 0.8)), 2, 300)):
- dev: 376 471 impressions, the size of the MIND-large dev split;
- test: 2 370 727 impressions, the size of the MIND-large test split.
Per set:
- end to end (host clock around work that ends in a device synchronise): ``predict``, ``write_prediction`` and both
  together, alternated round by round with ``evaluate`` on the same impressions (with the synthetic labels);
- the steps of ``write_prediction``: the device formatting (CUDA events), the D2H copy of the text into pinned memory
  (CUDA events; bytes and GB/s) and the file write (host clock, into a temporary directory);
- device time per batch split into user encoder, scoring, ranking and formatting, from one ``torch.profiler`` pass
  of its own (kernel time summed by kernel name, divided by the number of batches; formatting runs once per file);
- the plain-Python formatter (``f"{id} [{','.join(map(str, ranks))}]\\n"`` over the host ranks), host clock.
The device name and power limit are read in the same run.

    python tools/predict_bench.py [--out profiles/predict_bench.json] [--rounds 5]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_NEWS, D, H = 161013, 256, 50
SETS = {"dev": 376471, "test": 2370727}


def _device_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as exc:  # noqa: BLE001  (reported, not hidden)
        info["power_limit"] = f"unavailable: {type(exc).__name__}"
    return info


def _py_format(imp_ids, ptr, rank):
    r, p = rank.tolist(), ptr.tolist()
    return "".join(f"{i} [{','.join(map(str, r[p[b]:p[b + 1]]))}]\n" for b, i in enumerate(imp_ids.tolist())).encode()


def _timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t) * 1e3


def _stats(xs):
    xs = sorted(xs)
    return {"median": round(xs[len(xs) // 2], 3), "min": round(xs[0], 3), "max": round(xs[-1], 3), "n": len(xs)}


def _profile_split(trun, ops, ue, table, hist, mask, ptr, cand, imp_ids, n_batches):
    """device ms per batch by kernel group from one profiled predict + format"""
    from torch.profiler import ProfilerActivity, profile
    dev = table.device
    ids_t, ptr_t = torch.from_numpy(imp_ids).to(dev), torch.from_numpy(ptr).to(dev)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _, rank = trun.predict(ue, table, hist, mask, ptr, cand)
        ops.format_prediction(ids_t, ptr_t, rank)
        torch.cuda.synchronize()
    groups = {"user_encoder": 0.0, "scoring": 0.0, "ranking": 0.0, "formatting": 0.0, "copies_and_fills": 0.0}
    kernels = {}
    for e in prof.key_averages():
        us = getattr(e, "self_device_time_total", None)
        if us is None:
            us = getattr(e, "self_cuda_time_total", 0.0)
        if not us:
            continue
        name = e.key
        kernels[name[:120]] = round(us / 1e3, 4)
        if "eval_score_kernel" in name:
            g = "scoring"
        elif "predict_rank_kernel" in name:
            g = "ranking"
        elif "predict_line_bytes" in name or "predict_write" in name or "DeviceScan" in name or "Scan" in name:
            g = "formatting"
        elif "Memcpy" in name or "Memset" in name or "fill" in name.lower():
            g = "copies_and_fills"
        else:
            g = "user_encoder"
        groups[g] += us / 1e3
    per_batch = {g: round(v / n_batches, 4) for g, v in groups.items() if g != "formatting"}
    return {"device_ms_per_batch": per_batch, "formatting_device_ms_per_file": round(groups["formatting"], 4),
            "formatting_device_ms_per_batch_equivalent": round(groups["formatting"] / n_batches, 4),
            "device_ms_total": {g: round(v, 4) for g, v in groups.items()}, "kernels_ms_total": kernels}


def run_set(name, n, rounds, trun, ops, synth, ue, table, tmp):
    hist, mask, ptr, cand, lab = synth.eval_impressions(n, N_NEWS, H, seed=7)
    imp_ids = np.arange(1, n + 1, dtype=np.int64)
    nnz = int(ptr[-1])
    n_batches = (n + 16383) // 16384
    path = os.path.join(tmp, f"prediction_{name}.txt")
    dev = table.device
    # warm-up of every shape
    trun.evaluate(ue, table, hist, mask, ptr, cand, lab)
    _, rank = trun.predict(ue, table, hist, mask, ptr, cand)
    nbytes = trun.write_prediction(path, imp_ids, ptr, rank)
    torch.cuda.synchronize()
    t = dict(evaluate=[], predict=[], write_prediction=[], predict_plus_write=[], format_device=[], d2h=[],
             file_write=[])
    ids_t, ptr_t = torch.from_numpy(imp_ids).to(dev), torch.from_numpy(ptr).to(dev)
    pinned = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    for _ in range(rounds):
        _, ms = _timed(lambda: trun.evaluate(ue, table, hist, mask, ptr, cand, lab))
        t["evaluate"].append(ms)
        (_, rank), ms_p = _timed(lambda: trun.predict(ue, table, hist, mask, ptr, cand))
        _, ms_w = _timed(lambda: trun.write_prediction(path, imp_ids, ptr, rank))
        t["predict"].append(ms_p)
        t["write_prediction"].append(ms_w)
        t["predict_plus_write"].append(ms_p + ms_w)
        # the steps of write_prediction, one by one
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        text = ops.format_prediction(ids_t, ptr_t, rank)
        e[1].record()
        pinned[:text.numel()].copy_(text, non_blocking=True)
        e[2].record()
        torch.cuda.synchronize()
        t["format_device"].append(e[0].elapsed_time(e[1]))
        t["d2h"].append(e[1].elapsed_time(e[2]))
        t0 = time.perf_counter()
        with open(path, "wb") as f:
            f.write(memoryview(pinned[:text.numel()].numpy()))
        t["file_write"].append((time.perf_counter() - t0) * 1e3)
    rank_h = rank.cpu().numpy()
    t0 = time.perf_counter()
    ref = _py_format(imp_ids, ptr, rank_h)
    py_ms = (time.perf_counter() - t0) * 1e3
    same = ref == open(path, "rb").read()
    out = {"impressions": n, "candidates": nnz, "batches": n_batches, "file_bytes": nbytes,
           "file_equals_python_formatter": same, "python_formatter_ms": round(py_ms, 1),
           "ms": {k: _stats(v) for k, v in t.items()},
           "d2h_GBps_median": round(nbytes / (_stats(t["d2h"])["median"] * 1e-3) / 1e9, 2)}
    out["profile"] = _profile_split(trun, ops, ue, table, hist, mask, ptr, cand, imp_ids, n_batches)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "predict_bench.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--sets", default="dev,test")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("predict_bench: needs a CUDA device")
    import tinyrec.model_bert as mb
    import tinyrec.ops as ops
    import tinyrec.run as trun
    import tinyrec.synth as synth
    dev = torch.device("cuda", 0)
    res = {"device": _device_info(), "table_rows": N_NEWS + 1, "D": D, "H": H, "batch_size": 16384,
           "user_encoder": "NAML, random init, bf16 mode", "rounds": a.rounds,
           "timing": "host clock around synchronised calls (end to end); CUDA events for formatting and the D2H copy; "
                     "per-kernel split from a separate torch.profiler pass"}
    table = (torch.randn(N_NEWS + 1, D, generator=torch.Generator().manual_seed(1)) * 0.1).to(dev)
    args = synth.demo_args(user_log_length=H)
    ue = mb.UserEncoder(args)
    ue.load_state_dict(synth.user_encoder_state("", D, args.user_query_vector_dim, 0), strict=True)
    ue = ue.to(dev).eval()
    with tempfile.TemporaryDirectory() as tmp:
        for name in a.sets.split(","):
            res[name] = run_set(name, SETS[name], a.rounds, trun, ops, synth, ue, table, tmp)
            print(name, json.dumps({k: v for k, v in res[name].items() if k != "profile"}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
