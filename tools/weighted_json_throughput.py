"""Likelihood-weighted device JSON entry (kc_consolidate_json_packed_weighted, self-defined: DESIGN.md §5) next to the unweighted
one (kc_consolidate_json_packed) on the SAME texts, plus the CUDA-event times of its two new kernels.  One JSON line.

Workloads: S32 candidate texts at n = 16 (the bench schema), and a config-4-shaped batch (n = 32, 256K records, 8..64 token
logprobs per candidate; short records of 4 vote fields and one number).  Per workload and entry: wall-clock records/s around the
C-ABI call (best of --reps after one warm-up call), the H2D bytes the call reports (texts + offsets, and with weighting the token
logprobs + their offsets), and the per-stage device times.  Kernels: kc_candidate_weights_f32 and kc_weighted_vote_groups_i8 on
the config-4 shape, mean of --iters launches between CUDA events, algorithmic bytes over time against the HBM peak
(MEASURED_PEAKS.json hbm_gbs when present).  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from k_llms_b200 import _native as K  # noqa: E402

FALLBACK_HBM_GBS = 6650.0


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except (OSError, KeyError, ValueError):
        return FALLBACK_HBM_GBS, "fallback (no MEASURED_PEAKS.json)"


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as exc:  # noqa: BLE001
        return {"name": None, "error": repr(exc)}


def logprobs_for(rng, n_seq, lo=8, hi=64):
    lens = rng.integers(lo, hi + 1, n_seq)
    lp_off = np.zeros(n_seq + 1, dtype=np.int64)
    np.cumsum(lens, out=lp_off[1:])
    lp = K.pinned_empty((int(lp_off[-1]),), np.float32)
    lp[:] = -rng.exponential(0.5, int(lp_off[-1])).astype(np.float32)
    return lp, lp_off


def config4_texts(R, n, rng):
    pool = [json.dumps({"city": ["Paris", "paris", "Lyon", "Nice"][i % 4], "ok": bool(i & 4), "tier": ["gold", "Silver"][(i >> 3) & 1],
                        "code": ["a1", "b2", "A1"][i % 3], "n": i % 5}) for i in range(64)]
    L = max(len(t) for t in pool)
    pool_bytes = np.frombuffer("".join(t.ljust(L) for t in pool).encode(), dtype=np.uint8).reshape(64, L)
    blob = K.pinned_empty((R * n * L,), np.uint8)
    blob[:] = pool_bytes[rng.integers(0, 64, R * n)].reshape(-1)
    return blob, np.arange(R * n + 1, dtype=np.int64) * L


def run_entry(blob, off, n, logprobs, reps):
    K.consolidate_json_packed(blob, off, n, logprobs=logprobs).close()  # warm-up: grows the pooled buffers
    best, stats = None, None
    for _ in range(reps):
        t0 = time.perf_counter()
        res = K.consolidate_json_packed(blob, off, n, logprobs=logprobs)
        dt = time.perf_counter() - t0
        ok = int((res.status == 0).sum())
        if best is None or dt < best:
            best, stats = dt, res.stats.as_dict()
        res.close()
    R = (len(off) - 1) // n
    h2d = stats["input_bytes"] + (R * n + 1) * 8 * (2 if logprobs is not None else 1)
    return {"records_per_s": R / best, "wall_ms": best * 1e3, "on_device": ok, "h2d_bytes": int(h2d),
            "input_bytes": int(stats["input_bytes"]), "h2d_ms": stats["h2d_ms"], "plan_ms": stats["plan_ms"],
            "kernel_ms": stats["kernel_ms"], "emit_ms": stats["emit_ms"], "d2h_ms": stats["d2h_ms"], "chunks": stats["chunks"]}


def kernel_times(R, n, fields, iters, peak):
    import torch
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(7)
    seq = -torch.rand(R, n, device=dev, generator=g) * 20.0
    cells = torch.randint(-1, 4, (R * fields, n), device=dev, generator=g, dtype=torch.int32).to(torch.int8)
    rec = torch.arange(R, device=dev, dtype=torch.int32).repeat_interleave(fields)
    w = K.candidate_weights(seq)
    K.weighted_vote_groups(cells, rec, w)
    torch.cuda.synchronize()
    out = {}
    for name, fn, nbytes in (
            ("kc_candidate_weights_f32", lambda: K.candidate_weights(seq), R * n * 4 * 2),
            ("kc_weighted_vote_groups_i8", lambda: K.weighted_vote_groups(cells, rec, w),
             R * fields * (n + 4 + 4 + 8) + R * n * 4)):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        gbs = nbytes / (ms * 1e-3) / 1e9
        out[name] = {"ms": ms, "algorithmic_bytes": nbytes, "gb_per_s": gbs, "of_hbm_peak": gbs / peak}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--s32-records", type=int, default=256 * 1024)
    ap.add_argument("--c4-records", type=int, default=256 * 1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("weighted_json_throughput.py measures on the GPU: no CUDA device")
    peak, peak_src = hbm_peak()
    rng = np.random.default_rng(20261017)
    res = {"tool": "weighted_json_throughput", "card": card(), "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "workloads": {}}
    n = 16
    blob, off = K.s32_texts_packed(args.s32_records, n, 20260921)
    lp = logprobs_for(rng, args.s32_records * n)
    res["workloads"]["s32_n16"] = {"records": args.s32_records, "n": n, "tokens_per_candidate": "8..64",
                                   "unweighted": run_entry(blob, off, n, None, args.reps),
                                   "weighted": run_entry(blob, off, n, lp, args.reps)}
    del blob, off, lp
    n = 32
    blob, off = config4_texts(args.c4_records, n, rng)
    lp = logprobs_for(rng, args.c4_records * n)
    res["workloads"]["config4_n32"] = {"records": args.c4_records, "n": n, "tokens_per_candidate": "8..64",
                                       "unweighted": run_entry(blob, off, n, None, args.reps),
                                       "weighted": run_entry(blob, off, n, lp, args.reps)}
    res["kernels"] = kernel_times(args.c4_records, 32, 4, args.iters, peak)
    res["kernels"]["shape"] = f"{args.c4_records} records x 4 vote groups x n = 32 (int8 cells)"
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
