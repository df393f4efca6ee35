#!/usr/bin/env python
"""bench.py — consensus records/s on schema S32 (BASELINE.json `metric`), device-resident and end-to-end.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--n 16] [--records 1000000] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: K1 (vote, 24 fields) + K2 (numeric, 8 fields) over
`records` records per GPU with n candidates (BASELINE configs[1]: 1M x 32 fields, n=16); at N > 1 every rank owns
its own 1M-record shard (weak scaling, configs[4]) and a step ends with every rank holding every rank's packed output
columns: by default the reassembly is fused into the kernels (P2P stores into the peers' copies of a symmetric-memory
buffer; --route multimem: NVSwitch multicast stores), --reassembly nccl runs a pipelined NCCL all-gather instead.
One JSON line on stdout (rank 0).

value      whole-job records/s, inputs resident in HBM, CUDA events, max over ranks, barrier + synchronize on both sides.
e2e        the reference's unit of work through the C ABI with HOST buffers: n candidate JSON TEXTS per record in (pinned host
           memory) -> consensus JSON + likelihoods JSON texts out (host memory), kc_consolidate_json_packed (H1g: the JSON
           work runs on the device), WALL CLOCK around the call, max over ranks; `stages` splits the device time into
           H2D / plan (scan, type, encode) / kernels (K1 + K2) / emit / D2H.
e2e_columnar  last round's leg: kc_consensus_host_i8 on pre-encoded pinned int8 / f64 columns (no JSON), CUDA events.
roofline   dominant kernel: algorithmic bytes (SURVEY.md §8d) / its mean launch time, over MEASURED_PEAKS.json hbm_gbs.
cpu_baseline  the CPU arm on a bounded sample (rank 0, N=1): the SAME boundary as e2e — json.loads of the n candidate texts,
           alignment pre-pass, consensus, json.dumps — with the oracle port of the reference's Python path (the reference is
           pure Python and cannot travel to the GPU box; measured in the build container the port is ~1.3x FASTER than the
           unmodified reference, so the ratio is conservative), on every core the process may use (affinity and cgroup
           quota); `consensus_only` repeats last round's parse-free variant (Python dicts in, no JSON) for continuity.
--impl reference  times that CPU path alone.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "consensus records/sec at n=16 (1M x 32-field); achieved HBM GB/s vs peak"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md, used only when MEASURED_PEAKS.json is absent


def ncu_traffic(kind: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of this
    workload (profiles/r1_ncu_traffic.json) — not measured live (a number taken under a profiler is not a bench value)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r1_ncu_traffic.json")) as f:
            return float(json.load(f)["kernels"][kind]["traffic_bytes"])
    except Exception:
        return None


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------- CPU arm (oracle port)

def usable_cores() -> int:
    """Cores this process may really use: the affinity mask, capped by the cgroup CPU quota (os.cpu_count() ignores both)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:  # cgroup v2: "<quota|max> <period>"
            q, per = f.read().split()
            if q != "max":
                quota = float(q) / float(per)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                per = float(f.read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(quota + 0.5)))
    return n


def _s32_candidate_dicts(count, n, seed):
    import numpy as np  # noqa: F401
    from k_llms_b200 import synth
    codes, none_code, vals = synth.s32_numpy(count, n, seed)
    vocab = ["alpha", "Bravo", "charlie", "DELTA", "echo", "foxtrot", "golf", "Hotel"]
    variants = [lambda w: w, lambda w: w.upper(), lambda w: w.lower() + "!", lambda w: " " + w]
    records = []
    for r in range(count):
        cands = []
        for c in range(n):
            d = {}
            for f in range(16):
                k = int(codes[r, f, c])
                d[f"f{f:02d}"] = None if k < 0 else variants[(r + c + f) % 4](vocab[k])
            for f in range(16, 24):
                k = int(codes[r, f, c])
                d[f"f{f:02d}"] = None if k < 0 else bool(k)
            for f in range(8):
                v = vals[r, f, c]
                d[f"f{24 + f:02d}"] = None if v != v else (int(v) if f < 6 else float(v))
            cands.append(d)
        records.append(cands)
    return records


def _cpu_worker(args):
    """Build `count` S32 records (untimed), then time the per-record loop.  mode "json": the reference's unit of work —
    n candidate TEXTS in, json.loads each (consolidation.py:25-38), alignment pre-pass + consensus (client order,
    consolidation.py:333-349), json.dumps of the consensus and of the likelihoods.  mode "dicts": consensus only, Python
    candidate dicts in (no parsing, no alignment, no output text)."""
    seed, count, n, mode = args
    import json as _json
    from oracle import consensus_py as O
    records = _s32_candidate_dicts(count, n, seed)
    embed = lambda texts: [[0.0] for _ in texts]  # noqa: E731
    if mode == "json":
        texts = [[_json.dumps(d) for d in cands] for cands in records]
        del records
        t0 = time.perf_counter()
        for cand_texts in texts:
            value, conf = O.client_order([_json.loads(t) for t in cand_texts], embed=embed)
            _json.dumps(value), _json.dumps(conf)
        return count, time.perf_counter() - t0
    t0 = time.perf_counter()
    for cands in records:
        O.consensus(cands, embed=embed)
    return count, time.perf_counter() - t0


def cpu_baseline(n: int, per_worker: int, cores: int, mode: str = "json"):
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        t0 = time.perf_counter()
        res = pool.map(_cpu_worker, [(20260921 + 2 + 1000 * i, per_worker, n, mode) for i in range(cores)])
        wall = time.perf_counter() - t0
    total = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    what = ("n candidate JSON texts per record -> json.loads -> alignment pre-pass + consensus (oracle/consensus_py.client_order) -> "
            "json.dumps of consensus and likelihoods" if mode == "json" else
            "Python candidate dicts -> oracle/consensus_py.consensus (no parsing, no alignment, no output text)")
    return {"value": total / busy, "unit": "records/s", "cores": cores, "kind": "port", "boundary": mode,
            "sample": f"{total} records ({per_worker}/worker) of the S32 n={n} workload; {what}; multiprocessing.Pool({cores}) "
                      f"= usable cores (affinity + cgroup quota; os.cpu_count() says {os.cpu_count()}); slowest worker {busy:.1f}s, "
                      f"wall incl. record construction {wall:.1f}s",
            "per_core": total / busy / cores,
            "note": "port of the reference's Python path; in the build container the unmodified reference ran 1.3x SLOWER than this port "
                    "(892 vs 1181 records/s/core on S32, same outputs)",
            "cpu_model": _cpu_model()}


def _cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = usable_cores()
    per_worker = max(100, int(args.cpu_records_per_core))
    vals = []
    base = None
    for _ in range(max(1, min(args.steps, 3))):  # each step = one bounded sample; keep the whole arm within minutes
        base = cpu_baseline(args.n, per_worker, cores, "json")
        vals.append(base["value"])
    value = statistics.median(vals)
    base["value"] = value
    base["consensus_only"] = cpu_baseline(args.n, per_worker, cores, "dicts")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "records/s", "n_gpus": args.gpus,
            "steps": len(vals), "warmup": 0, "ms_per_step": 1e3 * (per_worker * cores) / value, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "python objects (float64 / str)", "data": "synthetic",
            "config": {"workload": f"S32 schema (16 str-enum + 8 bool + 6 int + 2 float fields), n={args.n}, "
                                   f"{per_worker * cores} records per step (bounded sample of the 1M-record batch), JSON texts in -> "
                                   "consensus + likelihoods JSON texts out (the boundary of the GPU arm's e2e)"},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference is pure Python and absent on the GPU box; this arm runs the oracle port of its per-record path"}
    emit(line)


# ----------------------------------------------------------------------------- clocks sampler

class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.samples = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.samples.append((time.time(), parts))

    def stop(self):
        if self.proc:
            self.proc.terminate()

    def summary(self, t0: float, t1: float):
        win = [p for t, p in self.samples if t0 <= t <= t1]
        scope = "timed region"
        if len(win) < 3:
            win, scope = [p for _, p in self.samples], "whole run (timed region shorter than the sampling period)"
        if not win:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "window": "nvidia-smi unavailable"}
        sm = [float(p[0]) for p in win if p[0].replace(".", "").isdigit()]
        reasons = set()
        for p in win:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(win[0][1]) if win[0][1].isdigit() else None,
                "reasons": sorted(reasons), "samples": len(win), "window": scope}


# ----------------------------------------------------------------------------- GPU arm

def bind_to_gpu_numa_node(gpu_index: int):
    """Run this process on the CPUs of the NUMA node the GPU hangs off, so that the page-locked host buffers it allocates
    (first touch) are local to the GPU's PCIe root: with 8 ranks streaming ~50 GB/s each, remote-node memory would put half
    of the traffic on the socket interconnect.  Returns the node or None (single node / information unavailable)."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(gpu_index).pci_bus_id
        dom = torch.cuda.get_device_properties(gpu_index).pci_domain_id
        dev_id = torch.cuda.get_device_properties(gpu_index).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev_id:02x}.0/numa_node"
        node = int(open(path).read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


DUMP_RECORDS = 1 << 16  # 512 B per record as float64: 32 MiB in all


def dump_outputs(out_dir, n_records, win, vmeta, value, nmeta):
    """Write this rank's results of the last timed step as float64 .npy files: the winning code and result word of every
    vote field, the value and result word of every numeric field, for a fixed sample of records (all of them up to
    DUMP_RECORDS; beyond, a seeded sample in record order, listed in records.npy).  float64 holds every int32 code and
    uint32 word exactly, so two builds can be compared bit for bit."""
    import numpy as np
    import torch
    idx = np.arange(n_records)
    if n_records > DUMP_RECORDS:
        idx = np.sort(np.random.default_rng(0).choice(n_records, DUMP_RECORDS, replace=False))
    rows = torch.from_numpy(idx).to(win.device)
    pick = lambda t: t.view(n_records, -1)[rows].cpu().numpy()  # noqa: E731
    arrays = {"records": idx.astype(np.float64),
              "vote_win_code": pick(win).astype(np.float64),
              "vote_meta": pick(vmeta).view(np.uint32).astype(np.float64),
              "numeric_value": pick(value),
              "numeric_meta": pick(nmeta).view(np.uint32).astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_gpu_arm(args):
    import numpy as np
    import torch
    from k_llms_b200 import _native as K
    from k_llms_b200 import synth
    from k_llms_b200.distributed import (FusedShardedConsensus, OutputLayout, PipelinedShardedConsensus, ShardedConsensus,
                                         wire_pack_num, wire_pack_votes)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None  # pinned host buffers land on the GPU's own memory node
    dist = None
    if world > 1:
        import torch.distributed as dist
        if not dist.is_initialized():  # --sweep runs several n in one process group
            dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    N, n = args.records, args.n
    codes, none_code, vals = synth.s32_torch(N, n, 20260921 + 2 + rank, dev)  # §8d: seed 20260921 + cfg, per-rank shard
    c2, v2 = codes.view(N * 24, n), vals.view(N * 8, n)
    # N > 1, fused P2P route: the gathered vote results travel packed (one word instead of two; full results stay local)
    packed = world > 1 and args.results == "packed" and args.reassembly in ("auto", "fused") and args.route in ("peers", "push")
    layout = OutputLayout(N, 24, 8, packed_votes=packed)
    # N > 1: reassembly is fused into the kernels (multimem.st through NVSwitch) when the multicast mapping exists,
    # else the pipelined NCCL all-gather (--reassembly nccl forces it).
    fused = None
    pipelined = None
    if args.push_mode == "auto":
        # measured on this pool (profiles/r2_push_sweep_n{2,8}.txt): at 2 GPUs the step is compute-bound and K1 storing its words
        # remotely itself while copy engines ship K2's results wins (0.58 ms); from 4 GPUs on the step is NVLink-ingress-bound
        # and the push kernel's 16-byte stores use the link best (1.67 ms at 8 GPUs vs 2.19 ms for round 1's fused scalar stores)
        args.push_mode = "hybrid" if world <= 2 else "wire"
        if args.push_chunks <= 0:
            args.push_chunks = 1 if world <= 2 else 4
    if args.push_chunks <= 0:
        args.push_chunks = 4
    if world > 1 and args.reassembly in ("auto", "fused") and args.route == "push":
        # default: full results stay local (fast kernels); a push kernel on a side stream packs chunk c into the wire format
        # (128 B/record) and stores it into every peer's copy with 16-byte vectors while chunk c + 1 is computed
        try:
            pipelined = PipelinedShardedConsensus(N, 24, 8, dev, chunks=args.push_chunks, wide=n > 31, push_ctas=args.push_ctas,
                                                  mode=args.push_mode)
            if not pipelined.available():
                pipelined = None
        except Exception as exc:
            print(f"pipelined push unavailable: {exc}", file=sys.stderr)
            pipelined = None
    if world > 1 and pipelined is None and args.reassembly in ("auto", "fused"):
        if args.route == "push":
            args.route = "peers"
        try:
            fused = FusedShardedConsensus(layout, dev, route=args.route)
            if not fused.available():
                fused = None
        except Exception as exc:  # symmetric memory unavailable on this stack
            print(f"fused reassembly unavailable: {exc}", file=sys.stderr)
            fused = None
        if fused is None and args.reassembly == "fused":
            raise RuntimeError("--reassembly fused requested but no multicast mapping is available")
    if fused is None and layout.packed_votes:  # the NCCL path gathers the full two-word vote results
        packed = False
        layout = OutputLayout(N, 24, 8)
    chunks = args.chunks if (world > 1 and fused is None) else 1  # NCCL path: pipeline depth of compute vs all-gather
    if pipelined is not None:
        chunks = args.push_chunks
    while N % chunks:
        chunks -= 1
    sharded = pipelined if pipelined is not None else (ShardedConsensus(layout, dev, chunks=chunks) if fused is None else None)
    R = N // chunks
    lib = K.load()
    K.check(lib.kc_set_device(local_rank))
    sp = int(torch.cuda.current_stream().cuda_stream)
    kernel_events = []  # (start, mid, end) per chunk launch, only while timing

    def compute(c, views):
        win, vmeta, value, nmeta = views
        cc, vv = c2[c * R * 24:(c + 1) * R * 24], v2[c * R * 8:(c + 1) * R * 8]
        if kernel_events is not None and timing[0]:
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record()
        if pipelined is not None:
            pipelined.vote(c, cc.data_ptr(), R * 24, n, none_code.data_ptr(), 24, sp)
        else:
            K.check(lib.kc_vote_i32(cc.data_ptr(), R * 24, n, none_code.data_ptr(), 24, win.data_ptr(), vmeta.data_ptr(), sp))
        if timing[0]:
            e[1].record()
        if pipelined is not None:
            pipelined.numeric(c, vv.data_ptr(), R * 8, n, 0.03, 1e-6, sp)
        else:
            K.check(lib.kc_numeric_f64(vv.data_ptr(), R * 8, n, 0.03, 1e-6, value.data_ptr(), nmeta.data_ptr(), sp))
        if timing[0]:
            e[2].record()
            kernel_events.append(e)

    def fused_launch(f):
        if timing[0]:
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record()
        f.vote(c2.data_ptr(), N * 24, n, none_code.data_ptr(), 24, sp)
        if timing[0]:
            e[1].record()
        f.numeric(v2.data_ptr(), N * 8, n, 0.03, 1e-6, sp)
        if timing[0]:
            e[2].record()
            kernel_events.append(e)

    def compute_numeric(c, views):  # mode hybrid: K2 of the chunk on its own (its values / words then travel by copy engine ...)
        vv = v2[c * R * 8:(c + 1) * R * 8]
        if timing[0]:
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            e[2].record()
            split_events.append(e)
        pipelined.numeric(c, vv.data_ptr(), R * 8, n, 0.03, 1e-6, sp)
        if timing[0]:
            e[3].record()

    def compute_vote(c, views):  # ... while K1 stores its wire words into the peers' copies itself
        cc = c2[c * R * 24:(c + 1) * R * 24]
        if timing[0]:
            e = split_events[-1]
            e[0].record()
        pipelined.vote(c, cc.data_ptr(), R * 24, n, none_code.data_ptr(), 24, sp)
        if timing[0]:
            e[1].record()

    split_events = []  # (vote start, vote end, numeric start, numeric end) per chunk, hybrid mode

    def one_step():
        if fused is not None:
            fused.step(fused_launch)
        elif pipelined is not None and args.push_mode == "hybrid":
            pipelined.step(compute, compute_numeric=compute_numeric, compute_vote=compute_vote)
        else:
            sharded.step(compute)

    timing = [False]
    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        one_step()
    barrier()

    # --- timed: exactly K steps; per-kernel events on the launching stream ride along
    K_steps = args.steps
    timing[0] = True
    t_wall0 = time.time()
    barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(K_steps):
        one_step()
    stop.record()
    barrier()
    t_wall1 = time.time()
    timing[0] = False
    ms_total = max_over_ranks(start.elapsed_time(stop))
    ms_step = ms_total / K_steps
    vote_ms = sum(e[0].elapsed_time(e[1]) for e in kernel_events) / K_steps   # per step (all chunks)
    num_ms = sum(e[1].elapsed_time(e[2]) for e in kernel_events) / K_steps
    if split_events:
        vote_ms = sum(e[0].elapsed_time(e[1]) for e in split_events) / K_steps
        num_ms = sum(e[2].elapsed_time(e[3]) for e in split_events) / K_steps
    compute_ms = max_over_ranks(vote_ms + num_ms)
    value_rps = world * N / (ms_step / 1e3)
    gather_ms = 0.0
    if dist is not None and fused is None:  # the all-gather alone (no compute to hide behind), for the record
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(5):
            sharded.step(lambda c, v: None)
        g1.record()
        barrier()
        gather_ms = max_over_ranks(g0.elapsed_time(g1) / 5)
    kernels_in_step_ms = compute_ms  # K1 + K2 event times INSIDE the step (they share the GPU with the transfer at N > 1)
    if pipelined is not None:
        # compute_only proper: the same launches with the reassembly switched off (no pushes, no barrier), device events, max over ranks
        timing[0] = False
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = max(5, min(K_steps, 50))
        c0.record()
        for _ in range(reps):
            if args.push_mode == "hybrid":
                pipelined.step(compute, gather=False, compute_numeric=compute_numeric, compute_vote=compute_vote)
            else:
                pipelined.step(compute, gather=False)
        c1.record()
        barrier()
        compute_ms = max_over_ranks(c0.elapsed_time(c1) / reps)
    reassembly_check = None
    if pipelined is not None:
        # outside the timed region: EVERY rank's slot on THIS GPU must hold exactly the wire words of that rank's results —
        # the expected words travel through an NCCL all-gather (an independent route) and are compared bit for bit
        if pipelined.overflowed():
            raise RuntimeError("a result does not fit the narrow wire words: rerun with n > 31 semantics (wide)")
        L = pipelined.layout
        mine = torch.zeros(L.nbytes, dtype=torch.uint8, device=dev)
        ev, evalue, en = L.views(mine)
        wt = torch.int32 if L.wide else torch.int16
        ev.copy_(torch.from_numpy(wire_pack_votes(pipelined.win.cpu().numpy(), pipelined.vmeta.cpu().numpy().view(np.uint32), L.wide).view(np.int32 if L.wide else np.int16)).to(dev))
        evalue.copy_(pipelined.value)
        en.copy_(torch.from_numpy(wire_pack_num(pipelined.nmeta.cpu().numpy().view(np.uint32), L.wide).view(np.int32 if L.wide else np.int16)).to(dev))
        expect = torch.empty((world, L.nbytes), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(expect.view(-1), mine)
        torch.cuda.synchronize()
        bad = [r for r in range(world) if not torch.equal(expect[r], pipelined.gathered[r])]
        assert not bad, f"rank {rank}: gathered slots {bad} differ from the NCCL-gathered wire words"
        reassembly_check = f"every slot of the gathered buffer equals the NCCL all-gather of the ranks' packed results, bit for bit ({world} x {L.nbytes} B per rank)"
    if fused is not None:
        win, vmeta, value, nmeta = fused.rank_views(rank)
        if layout.packed_votes:
            if fused.packed_overflowed():
                raise RuntimeError("a winning code >= 2^18 cannot travel packed: rerun with --results full")
            # the gathered words must be the packing of the full local results
            lw, lm = fused.local_win, fused.local_vmeta
            expect = (lw & 0x3FFFF) | (((lm >> 6) & 0x7F) << 18) | (((lm >> 20) & 0x7F) << 25)
            assert torch.equal(win, expect), "packed gathered vote words differ from the local full results"
            win, vmeta = lw, lm
    else:
        win, vmeta, value, nmeta = [torch.cat([sharded.my_views(c)[k] for c in range(chunks)]) for k in range(4)]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, N, win, vmeta, value, nmeta)

    # --- end to end, the reference's unit of work: candidate JSON texts (pinned host memory) -> consensus / likelihoods texts
    e2e = None
    e2e_sample = []
    if not args.no_e2e:
        # N > 1: a quarter-million records per rank (2.1 GB of texts each) keeps 8 ranks' page-locked buffers and generation time modest
        Rj = int(args.e2e_records) if world == 1 else min(int(args.e2e_records), 262144)
        jblob, joff = K.s32_texts_packed(Rj, n, 20260921 + 2 + 7919 * rank)  # untimed: the batch a client would hand over
        res = None
        for _ in range(2):  # warm-up: staging pools, device buffers, the pinned output blob
            res = K.consolidate_json_packed(jblob, joff, n, device=local_rank)
            res.close()
        e2e_steps = max(1, min(K_steps, args.e2e_steps))
        barrier()
        walls, stats = [], None
        for _ in range(e2e_steps):
            t0 = time.perf_counter()
            res = K.consolidate_json_packed(jblob, joff, n, device=local_rank)
            walls.append((time.perf_counter() - t0) * 1e3)
            stats = res.stats.as_dict()
            if _ + 1 < e2e_steps:
                res.close()
        barrier()
        e2e_ms = max_over_ranks(statistics.mean(walls))
        assert stats["n_device"] == Rj, f"only {stats['n_device']} of {Rj} S32 records stayed on the device path"
        # keep a sample of (candidate texts, outputs): the cpu_baseline leg (rank 0, N = 1) checks it against the oracle's client order
        e2e_sample = []
        if rank == 0:
            text = jblob[: int(joff[-1])].tobytes()
            for r in range(0, Rj, max(1, Rj // 64)):
                e2e_sample.append(([text[joff[r * n + c]:joff[r * n + c + 1]].decode() for c in range(n)], res.content(r), res.likelihoods(r)))
            del text
        res.close()
        e2e = {"value": world * Rj / (e2e_ms / 1e3), "unit": "records/s", "h2d_bytes_per_step": int(stats["input_bytes"] + joff.nbytes),
               "d2h_bytes_per_step": int(stats["output_bytes"] + 17 * Rj), "ms_per_step": e2e_ms, "steps": e2e_steps,
               "records_per_step_per_gpu": Rj, "json_GBps": world * stats["input_bytes"] / (e2e_ms / 1e3) / 1e9,
               "timing": "wall clock (time.perf_counter) around the C-ABI call, host buffers in and out",
               "path": "kc_consolidate_json_packed (C ABI): n candidate JSON texts per record in pinned host memory -> H2D -> scan / key "
                       "sort / typing / sanitised-equality codes / exact decimal->f64 on the device -> K1 + K2 -> float repr + emit on the "
                       "device -> D2H: consensus JSON + likelihoods JSON texts in host memory",
               "stages": {"note": "device time per stage summed over the chunks (CUDA events per chunk; chunks overlap on "
                                  f"{stats['streams']} streams, so the sum exceeds the wall time)",
                          "h2d_ms": stats["h2d_ms"], "plan_ms": stats["plan_ms"], "kernel_ms": stats["kernel_ms"],
                          "emit_ms": stats["emit_ms"], "d2h_ms": stats["d2h_ms"], "chunks": stats["chunks"]},
               "pcie_floor_ms": stats["input_bytes"] / 55e9 * 1e3}
        del jblob, joff

    # --- last round's leg for continuity: pre-encoded columns through the host-buffer entry (no JSON)
    e2e_columnar = None
    if not args.no_e2e and args.e2e_columnar:
        # compact host cells: votes only need equality inside a group, so int8 codes are lossless (kc_consensus_host_i8)
        h_codes = K.pinned_empty((N, 24, n), np.int8 if args.e2e_cells == "i8" else np.int32)
        h_vals = K.pinned_empty((N, 8, n), np.float64)
        h_codes[...] = codes.cpu().numpy().astype(h_codes.dtype)
        h_vals[...] = vals.cpu().numpy()
        h_none = none_code.cpu().numpy()
        out = {"win_code": K.pinned_empty((N, 24), np.int32), "vote_meta": K.pinned_empty((N, 24), np.uint32),
               "value": K.pinned_empty((N, 8), np.float64), "num_meta": K.pinned_empty((N, 8), np.uint32)}
        col_steps = max(1, min(K_steps, args.e2e_steps))
        for _ in range(2):
            K.consensus_host(h_codes, h_none, h_vals, device=local_rank, out=out)
        barrier()
        ms = []
        for _ in range(col_steps):
            r = K.consensus_host(h_codes, h_none, h_vals, device=local_rank, out=out)
            ms.append(r["device_ms"])
        barrier()
        col_ms = max_over_ranks(statistics.mean(ms))
        # the host-buffer path must agree with the device-resident one
        assert np.array_equal(out["win_code"].reshape(-1), win.cpu().numpy()), "e2e result differs from device-resident result"
        assert np.array_equal(out["value"].reshape(-1).view(np.uint64), value.cpu().numpy().view(np.uint64))
        e2e_columnar = {"value": world * N / (col_ms / 1e3), "unit": "records/s", "h2d_bytes_per_step": int(h_codes.nbytes + h_vals.nbytes),
                        "d2h_bytes_per_step": int(sum(a.nbytes for a in out.values())), "ms_per_step": col_ms, "steps": col_steps,
                        "path": f"kc_consensus_host{'_i8' if args.e2e_cells == 'i8' else ''} (C ABI): PRE-ENCODED pinned host columns "
                                f"({h_codes.dtype} vote cells, f64 numeric cells; no JSON) -> chunked H2D -> K1/K2 -> D2H on 3 streams, per rank"}

    clocks = None
    if sampler is not None:
        sampler.stop()
        clocks = sampler.summary(t_wall0, t_wall1)

    if rank == 0:
        peak, peak_src = hbm_peak()
        bytes_vote, bytes_num = N * 24 * (4 * n + 8), N * 8 * (8 * n + 12)
        # per-launch figures: a step is `chunks` launches of each kernel
        kernels = {"vote": {"ms": vote_ms / chunks, "bytes": bytes_vote // chunks},
                   "numeric": {"ms": num_ms / chunks, "bytes": bytes_num // chunks}}
        dom = max(kernels, key=lambda k: kernels[k]["ms"])
        ach = kernels[dom]["bytes"] / (kernels[dom]["ms"] / 1e3) / 1e9
        roofline = {"bound": "hbm", "kernel": {"vote": f"kc::vote_*_kernel<{n}>", "numeric": f"kc::numeric_*_kernel<{n}>"}[dom],
                    "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": ncu_traffic(dom) if (world == 1 and n == 16 and N == 1_000_000 and chunks == 1) else None,
                    "traffic_source": "profiles/r1_ncu_traffic.json (ncu --set full of this workload; bytes per launch)",
                    "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": kernels[dom]["bytes"],
                    "all_kernels": {k: {"ms_per_launch": v["ms"], "achieved_GBps": v["bytes"] / (v["ms"] / 1e3) / 1e9,
                                        "frac": v["bytes"] / (v["ms"] / 1e3) / 1e9 / peak} for k, v in kernels.items()},
                    "step_frac": (bytes_vote + bytes_num) / ((vote_ms + num_ms) / 1e3) / 1e9 / peak}
        base = None
        if world == 1 and not args.no_cpu:
            cores = usable_cores()
            if e2e is not None:  # the checker's second job in this leg: the e2e texts must be the reference's (outside every timed region)
                import json as _json
                from oracle import consensus_py as O
                embed = lambda t: [[0.0] for _ in t]  # noqa: E731
                for cand_texts, content, lik in e2e_sample:
                    cv, cc = O.client_order([_json.loads(t) for t in cand_texts], embed=embed)
                    assert (content, lik) == (_json.dumps(cv), _json.dumps(cc)), "an e2e record differs from the oracle's client order"
                e2e["checked_against_oracle"] = len(e2e_sample)
            base = cpu_baseline(n, int(args.cpu_records_per_core), cores, "json")
            base["consensus_only"] = cpu_baseline(n, int(args.cpu_records_per_core), cores, "dicts")
        line = {"metric": METRIC, "value": value_rps, "unit": "records/s", "n_gpus": world, "steps": K_steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i32 codes / f64 values",
                "data": "synthetic",
                "config": {"workload": f"S32: {N} records/GPU x 32 fields (16 str-enum + 8 bool as int32 codes, 6 int + 2 float as f64), "
                                       f"n={n}, p_agree=0.8, p_none=0.05; {world} GPU(s), {world * N} records total",
                           "l2": f"inputs are {(bytes_vote + bytes_num) / 1e9:.2f} GB per step per GPU, > 126 MB L2: no flush needed",
                           "step": "K1 vote + K2 numeric" + ("" if world == 1 else
                                   (f" in {chunks} chunks; chunk c's results are packed to the wire format (128 B/record) and stored into every "
                                    "peer's copy by a push kernel (16-byte P2P stores over NVLink) on a side stream while chunk c+1 is "
                                    "computed + one cross-GPU barrier") if pipelined is not None else
                                   ((" with every result also stored into the peers' copies (P2P over NVLink"
                                     + (", vote results as one packed word: 192 B/record" if layout.packed_votes else ", 288 B/record")
                                     + ") + one cross-GPU barrier" if fused.route == "peers" else
                                     " with results multimem.st-replicated to every GPU through NVSwitch + one cross-GPU barrier")
                                    if fused is not None else " + pipelined NCCL all-gather of the output columns")),
                           "parallelism": (f"records sharded {world}-way; reassembly "
                                           + ("by a pipelined push kernel (P2P stores, wire format)" if pipelined is not None else
                                              (f"fused into the kernels ({'P2P stores to the peers' if fused.route == 'peers' else 'NVSwitch multicast stores'})")
                                              if fused is not None else "NCCL all-gather"))
                                          if world > 1 else "single GPU"},
                "e2e": e2e, "e2e_columnar": e2e_columnar, "gpu_launches": 2 * chunks * K_steps, "clocks": clocks, "roofline": roofline, "cpu_baseline": base,
                "compute_only": {"value": world * N / (compute_ms / 1e3), "ms_per_step": compute_ms,
                                 "note": "the step's kernel launches with the reassembly switched off" if pipelined is not None else "K1 + K2 event times inside the step",
                                 "kernels_inside_step_ms": kernels_in_step_ms,
                                 "all_gather_alone_ms": gather_ms, "gathered_bytes_per_rank": int((pipelined.layout.nbytes if pipelined is not None else layout.nbytes) * world),
                                 "pipeline_chunks": chunks, "numa_node": numa, "reassembly_check": reassembly_check,
                                 "bound": ("NVLink ingress of the reassembly: every GPU receives (N-1) x its share" if world > 1 else "HBM"),
                                 "reassembly": ("none" if world == 1 else f"push-{args.push_mode}-wire" + ("32" if pipelined.layout.wide else "16") if pipelined is not None else (f"fused-{fused.route}" + ("-packed" if layout.packed_votes else ""))
                                                if fused is not None else "nccl"),
                                 "nvlink_floor_ms": (world - 1) * (pipelined.layout.nbytes if pipelined is not None else layout.nbytes) / 770e9 * 1e3 if world > 1 else 0.0}}
        emit(line)
    if dist is not None and not getattr(args, "keep_group", False):
        dist.destroy_process_group()


_REAL_STDOUT = None


def _capture_stdout():
    """NCCL and friends print to fd 1 (e.g. "NCCL version ..."); the contract is ONE JSON line on stdout.  Point fd 1
    at stderr for the whole run and keep the real stdout for the final line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=16)
    ap.add_argument("--records", type=int, default=1_000_000, help="records per GPU")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--e2e-records", type=int, default=1_000_000, help="records per GPU of the JSON-texts e2e leg (8.2 KB of JSON each at n=16)")
    ap.add_argument("--e2e-columnar", type=int, default=1, help="also run last round's pre-encoded-columns leg (0 to skip)")
    ap.add_argument("--e2e-cells", default="i8", choices=["i8", "i32"], help="host encoding of vote cells for the e2e leg")
    ap.add_argument("--chunks", type=int, default=8, help="N>1, NCCL reassembly: pipeline chunks of compute vs all-gather")
    ap.add_argument("--reassembly", default="auto", choices=["auto", "fused", "nccl"])
    ap.add_argument("--results", default="packed", choices=["packed", "full"],
                    help="N>1 with the fused P2P route: gathered vote results as one packed word (code:18|support:7|present:7, "
                         "192 B/record over NVLink) or as the full two words (288 B/record)")
    ap.add_argument("--route", default="push", choices=["push", "peers", "multimem"],
                    help="reassembly without NCCL: push = results stay local, a push kernel packs and stores them into every peer's "
                         "copy on a side stream (default); peers / multimem = stores fused into K1 / K2 (P2P / NVSwitch multicast)")
    ap.add_argument("--push-chunks", type=int, default=0, help="route push: chunks of the shard (compute chunk c+1 overlaps the push of chunk c)")
    ap.add_argument("--push-ctas", type=int, default=0, help="route push: CTAs of the push kernel (0 = 2 per SM)")
    ap.add_argument("--push-mode", default="auto", choices=["auto", "hybrid", "wire", "pack", "dma"],
                    help="route push: hybrid = K1 stores its wire words into the peers' copies itself, K2's values / words travel by copy engine; "
                         "wire = K1 writes the wire words locally, a push kernel replicates; pack = the push kernel packs the full results; "
                         "dma = copy engines replicate the whole slot")
    ap.add_argument("--cpu-records-per-core", type=int, default=1000)
    ap.add_argument("--sweep", default="", help="comma-separated candidate counts, e.g. 2,4,8,16,32,64: one JSON line per n (configs[4])")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the last step's results (a seeded sample of records) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.sweep or args.impl == "reference"):
        ap.error("--dump-outputs takes the results of one GPU run: not with --sweep or --impl reference")
    args.sweep_push_mode, args.sweep_push_chunks = args.push_mode, args.push_chunks
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus != world and world == 1 and args.gpus > 1 and args.impl == "b200":
        # convenience: spawn torchrun ourselves when asked for N GPUs outside a launcher
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", "29577", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    _capture_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.sweep:
        # BASELINE configs[4]: one line per n (device-resident step incl. the multi-GPU reassembly; no e2e / CPU legs)
        args.no_e2e, args.no_cpu = True, True
        ns = [int(x) for x in args.sweep.split(",")]
        for i, nn in enumerate(ns):
            args.n = nn
            args.push_mode, args.push_chunks = args.sweep_push_mode, args.sweep_push_chunks
            args.keep_group = i + 1 < len(ns)
            run_gpu_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
