#!/usr/bin/env python
"""bench.py — candidate x trace reward evals/sec (BASELINE.json metric) on N B200s.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...        # the reference arm: CPU oracle, all host threads
    python bench.py ... --dump-outputs DIR      # also write what the last timed step returned, DIR/<name>.npy

A "step" is one pass of the hot path over the resident workload — ONE kernel launch per rank:
K1 reward9 (Form D, 36 B/eval) with the K2 detect6 corpus scan on its spare warp; the last CTA
joins the shards' int64 partial vectors over NVLink peer memory (N > 1) and runs K3 (segmented
sum + radix top-K); the result block lands in the caller's page-locked buffer.

Workload: BASELINE configs[2] = 256 candidates x 10 M records (92.16 GB) + the 10 M-record corpus.
N > 1, default `--scaling strong`: the SAME 256 x 10 M is sharded over the record axis (T_global
fixed, T_per_gpu = T_global / N; SURVEY 8d config 3 "T-sharded for 2/4/8") — `value` is that;
the weak-scaling number (256 x 10 M per GPU) is measured in the same run and reported beside it
under "weak_scaling".  Every measured number carries a parity block checked against the CPU oracle
outside the timed region; a mismatch makes the run exit non-zero.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "candidate_x_trace_reward_evals_per_sec"
UNIT = "evals/s"
SEED = 0x5EED0003


def read_traffic(C, T):
    """DRAM bytes of one fused K1 launch from the committed ncu capture (profiles/traffic.json) and the capture's name;
    (None, None) when the benchmarked launch is not the profiled one (other shape, or a changed kernel)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)["k_reward9"]
        if (t["C"], t["T"]) == (C, T):
            return t["dram_bytes_read"] + t["dram_bytes_write"], t.get("source", "profiles/traffic.json")
    except Exception:
        pass
    return None, None


def read_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, line in self.rows:
            if ts < t0 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(out_dir: str, res) -> None:
    """What a caller of the timed step receives (its ScoreResult: scores, counts, top-K, corpus report; not the timings) as
    float64 arrays in out_dir/<name>.npy.  The workload comes from SEED, so two builds run with the same arguments can be
    compared output for output.  Integers are exact in float64 here: counts are at most the record count, indices below it."""
    os.makedirs(out_dir, exist_ok=True)
    rep = res.report
    arrays = {
        "scores": res.scores, "counts": res.counts, "topk": res.topk,
        "report_totals": [rep.total, rep.good, rep.bad, rep.none, rep.goodRate, rep.withReward, rep.rewardSum, rep.avgReward,
                          rep.toolCalls, rep.toolSucc, rep.toolFail, rep.toolSuccessRate],
        "report_by_mode": [[*rep.byMode[m], rep.byModeGoodRate[m]] for m in range(len(rep.byMode))],
        "report_dims": [[d.sum, d.count, d.avg, d.low_flag, d.low_severity, d.sugg_flag, d.sugg_priority] for d in rep.dim],
        "report_patterns": [[p.count, p.flag, p.severity, *p.examples] for p in rep.pat],
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def bind_to_gpu_numa_node(local: int) -> str:
    """Pin this rank to the CPUs of its GPU's NUMA node before it allocates pinned host buffers
    (first touch places them next to the GPU's PCIe root: matters for the 8-rank e2e leg)."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = torch.cuda.get_device_properties(local).pci_domain_id
        dev = torch.cuda.get_device_properties(local).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return "numa: single node"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"numa node {node} ({len(cpus)} cpus)"
    except Exception as ex:
        return f"numa binding skipped: {ex}"
    return "numa binding skipped"


def host_cpu_budget() -> dict:
    """What the box really gives this process: affinity mask and the cgroup CPU quota (a quota below the mask
    bounds every multi-threaded CPU number of this run: the measurement pod grants 16 CPUs of its 128)."""
    out = {"affinity_cpus": len(os.sched_getaffinity(0))}
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        out["cgroup_cpu_max"] = "unlimited" if q == "max" else round(int(q) / int(p), 2)
    except Exception:
        out["cgroup_cpu_max"] = "unknown"
    return out


def usable_threads(affinity=None) -> int:
    """Host threads worth starting: the affinity mask capped by the cgroup CPU quota (more threads than quota only
    buys throttling: 128 threads under a 16-CPU quota ran 2x slower than 16)."""
    n = len(affinity if affinity is not None else os.sched_getaffinity(0))
    q = host_cpu_budget()["cgroup_cpu_max"]
    if isinstance(q, float) and q >= 1:
        n = min(n, int(q + 0.5))
    return max(1, n)


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_sample_shape(C: int):
    """Bounded sample of configs[2] at its true candidate : record ratio: C x Ts Form D + a Ts-record corpus, sized to
    a quarter of the free host memory (256 x 1 M = 9.2 GB when it fits)."""
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 16 << 30
    Ts = int(min(1_000_000, (avail // 4) // (C * 36 + 32)))
    return C, max(Ts // 1000 * 1000, 10_000)


class CpuArm:
    """The reference's CPU implementation of the step = the oracle port (the reference is TypeScript; no JS runtime
    exists here or on the GPU box): orc_score_dims_mt + orc_topk + orc_report_build_mt on all host threads."""

    def __init__(self, C: int):
        import oracle
        oracle.build()
        self.orc = oracle
        self.threads = usable_threads()
        self.C, self.T = cpu_sample_shape(C)
        t0 = time.perf_counter()
        self.dims = oracle.gen_dims(SEED, 0, self.C, 0, self.T, 300, self.threads)
        self.recs = oracle.gen_records(SEED, oracle.STREAM_CORPUS, 0, 1, 0, self.T, 300, self.threads).reshape(-1)
        self.gen_s = time.perf_counter() - t0

    def step(self):
        s, n = self.orc.score_dims(self.dims, nthreads=self.threads)
        self.orc.topk(s, self.C // 4)
        self.orc.report(self.recs, nthreads=self.threads)

    def time_steps(self, steps: int, warmup: int):
        for _ in range(warmup):
            self.step()
        ts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            self.step()
            ts.append(time.perf_counter() - t0)
        return ts

    def single_thread_rate(self, seconds: float = 3.0) -> float:
        """The parity oracle itself: one thread, exact reference order (SURVEY 8d "CPU baseline" (i))."""
        sub = self.dims[:2]
        t0, n = time.perf_counter(), 0
        while time.perf_counter() - t0 < seconds:
            self.orc.score_dims(sub, nthreads=0)
            n += 1
        return 2 * self.T * n / (time.perf_counter() - t0)

    def describe(self, ts) -> dict:
        med = float(np.median(ts))
        return {"value": self.C * self.T / med, "unit": UNIT, "cores": self.threads, "kind": "port",
                "sample": f"{self.C} candidates x {self.T} records Form D ({self.C * self.T * 36 / 1e9:.2f} GB) + {self.T}-record corpus per step "
                          f"(configs[2] generator, seed {SEED:#x}, true candidate:record ratio), {len(ts)} timed steps after warm-up; "
                          f"oracle/apo_oracle.c on a persistent pinned thread pool (orc_score_dims_mt + orc_topk + orc_report_build_mt); "
                          f"the reference TypeScript cannot run here (no JS runtime)",
                "ms_per_step_median": med * 1e3, "ms_per_step_min": min(ts) * 1e3, "ms_per_step_max": max(ts) * 1e3,
                "spread": (max(ts) - min(ts)) / med, "host_GBps": (self.C * self.T * 36 + self.T * 32) / med / 1e9,
                "host": host_cpu_budget()}


def cpu_baseline(C: int, target_s: float = 12.0) -> dict:
    arm = CpuArm(C)
    one = arm.time_steps(1, 1)[0]
    steps = max(5, min(200, int(target_s / max(one, 1e-3))))
    d = arm.describe(arm.time_steps(steps, 1))
    d["single_thread_value"] = arm.single_thread_rate()
    d["speedup_vs_single_thread"] = d["value"] / d["single_thread_value"]
    return d


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path, all host threads, on a bounded sample of
    the GPU arm's config (same metric / unit).  Rank 0 alone runs and prints."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    arm = CpuArm(args.candidates)
    ts = arm.time_steps(args.steps, args.warmup)
    d = arm.describe(ts)
    dt = float(np.mean(ts))
    v = arm.C * arm.T / dt
    d["value"] = v
    # the same step when the caller holds trace records (the reference's own representation) instead of dims:
    # TCS:668-763 per evaluation + the mean — the CPU side of the e2e_records16 leg of the GPU arm (32-candidate slice)
    Cr = min(32, arm.C)
    roll = arm.orc.gen_records(SEED, arm.orc.STREAM_ROLLOUT, 0, Cr, 0, arm.T, 300, arm.threads)
    arm.orc.score_records(roll, nthreads=arm.threads)
    t0 = time.perf_counter()
    nrec = max(2, args.steps // 2)
    for _ in range(nrec):
        arm.orc.score_records(roll, nthreads=arm.threads)
    v_rec = Cr * arm.T / ((time.perf_counter() - t0) / nrec)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": args.scaling if args.gpus > 1 else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"configs[2] {args.candidates}-beam x 10M-span finalReward + detect6 + top-K "
                               f"(bounded CPU sample: {arm.C} x {arm.T} + {arm.T}-record corpus per step)", "C": arm.C, "T": arm.T},
        "cpu_baseline": d,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "from_records": {"value": v_rec, "unit": UNIT, "note": f"{Cr} x {arm.T} per-(candidate, record) trace records: dims derived per evaluation on the CPU"},
    }))


# ------------------------------------------------------------------------------------------------ GPU arm
class Harness:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.all_cpus = os.sched_getaffinity(0)
        self.numa_note = bind_to_gpu_numa_node(self.local) if self.world > 1 else "single rank: no binding"
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.pkg = importlib.import_module("senweaver-ide_b200")
        self.stream = torch.cuda.current_stream()

    def engine(self):
        eng = self.pkg.Engine(self.local)
        if self.world > 1:
            box = [self.pkg.Engine.comm_unique_id() if self.rank == 0 else None]
            self.dist.broadcast_object_list(box, src=0)
            eng.comm_init(self.world, self.rank, box[0])
        return eng

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps: int, warmup: int, sampler=None):
        """W warm-up calls, then exactly `steps` calls between barrier + synchronize, CUDA events on the launching
        stream, max over ranks.  Returns (ms per step, list of per-step results)."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        if sampler is not None:
            sampler.start()
            time.sleep(0.3)
        self.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        res = []
        w0 = time.perf_counter()
        ev0.record(self.stream)
        for _ in range(steps):
            res.append(fn())
        ev1.record(self.stream)
        self.barrier()
        w1 = time.perf_counter()
        ms = self.max_over_ranks(ev0.elapsed_time(ev1) / steps)
        return ms, res, (w0, w1)


def check_parity(H: Harness, eng, C: int, K: int, shards, last, layout_name: str, budget_s: float) -> dict:
    """Oracle parity of the measured configuration, outside the timed region (SURVEY 8c/8d):
      * full record axis: exact integer sums of the oracle (orc_score_generated_fx, the generator restated in C) for the
        candidates on both sides of the top-K boundary, the best one and a spread of others — as many as `budget_s` allows,
        all C when it fits; compared with the joined int64 partials with NO tolerance;
      * spot windows on every rank's shard (3 windows x 3 candidates per shard), exact;
      * scores == correctly rounded quotient of the exact sums, top-K == (score desc, index asc) order of them;
      * the whole corpus report (tallies, byMode, pattern counts / flags / severities / first-3 examples, per-dimension
        counts exactly; averages within 1e-5 relative) against orc_report_generated over all T_global records."""
    pkg, rank, world = H.pkg, H.rank, H.world
    sh = pkg.sharding
    out = {"layout": layout_name}
    tA = time.perf_counter()
    Tg = shards[-1][1]                                                     # shards: [first, last) of every rank, rank order
    Tmin = min(b - a for a, b in shards)
    sums, counts = eng.debug_partials(C)                                  # joined integers of the last timed step
    # windows: every rank scores the same relative window of its own shard; the join adds them up
    tail = max(0, (Tmin - 1000) // 8 * 8)
    rel = [(0, min(2048, Tmin)), ((Tmin // 2) // 8 * 8, min(2048, Tmin - (Tmin // 2) // 8 * 8)), (tail, Tmin - tail)]
    wcands = sorted({0, C // 2, C - 1})
    win_parts = []
    for first, count in rel:
        eng.score(C, 1, first=first, count=count)
        win_parts.append(eng.debug_partials(C))
    ok = True
    if rank == 0:
        import oracle
        oracle.build()
        nthreads = usable_threads(H.all_cpus)
        os.sched_setaffinity(0, H.all_cpus)
        exp_scores = sh.scores_from_partials(sums, counts)
        out["scores_from_exact_sums"] = bool(np.array_equal(exp_scores, last.scores))
        order = sh.topk_indices(exp_scores, C)
        out["topk_consistent"] = bool(np.array_equal(order[:K], last.topk))
        # candidates to verify on the full record axis, most important first
        prio = [int(order[0]), int(order[K - 1])] + ([int(order[K])] if K < C else []) + [int(order[-1])]
        prio += [int(x) for x in order[max(0, K - 3):K + 3]]
        prio += [int(x) for x in np.linspace(0, C - 1, 8).astype(int)]
        prio += [int(x) for x in order]
        seen, cl = set(), []
        for c in prio:
            if c not in seen:
                seen.add(c); cl.append(c)
        checked, exact, tB = 0, True, time.perf_counter()
        batch = 4
        while checked < len(cl):
            part = cl[checked:checked + batch]
            es, en = oracle.score_generated_fx(SEED, part, 0, Tg, 300, nthreads=nthreads)
            for c, s_, n_ in zip(part, es, en):
                if sums[c] != s_ or counts[c] != n_:
                    exact = False
            checked += len(part)
            el = time.perf_counter() - tB
            if checked >= 8 and el * len(cl) / checked > 1.5 * budget_s and el * (checked + batch) / checked > budget_s:
                break                                             # all C do not fit the budget (the boundary candidates came first)
            batch = min(64, batch * 2)
        out["full_axis_candidates_checked"] = checked
        out["full_axis_candidates_of"] = C
        out["full_axis_seconds"] = round(time.perf_counter() - tB, 2)
        out["partials_exact"] = exact
        # top-K vs the CPU reference: exact when every candidate was recomputed, else boundary-verified
        out["topk_match"] = bool(exact and out["topk_consistent"] and out["scores_from_exact_sums"])
        out["topk_check"] = "all candidates recomputed by the oracle" if checked == C else \
            "top-K boundary candidates (K-th, K+1-th and neighbours), best and worst recomputed by the oracle; order of the rest follows from the exact GPU sums"
        wins_ok, nwin = True, 0
        for (first, count), (ws, wn) in zip(rel, win_parts):
            for c in wcands:
                es = en = 0
                for r in range(world):
                    a, b = oracle.score_generated_fx(SEED, [c], shards[r][0] + first, count, 300, nthreads=1)
                    es += a[0]; en += b[0]
                nwin += world
                if ws[c] != es or wn[c] != en:
                    wins_ok = False
        out["windows"] = nwin
        out["windows_exact"] = wins_ok
        tC = time.perf_counter()
        ref = oracle.report_generated(SEED, 0, Tg, 0, 300, nthreads=nthreads)
        rep = last.report
        rep_ok = (rep.total, rep.good, rep.bad, rep.none, rep.withReward, rep.toolCalls, rep.toolSucc, rep.toolFail) == \
                 (ref.total, ref.good, ref.bad, ref.none, ref.withReward, ref.toolCalls, ref.toolSucc, ref.toolFail)
        for m in range(5):
            rep_ok &= list(rep.byMode[m]) == list(ref.byMode[m])
        for p in range(6):
            rep_ok &= (rep.pat[p].count, rep.pat[p].flag, rep.pat[p].severity, list(rep.pat[p].examples)) == \
                      (ref.pat[p].count, ref.pat[p].flag, ref.pat[p].severity, list(ref.pat[p].examples))
        rel_ok = abs(rep.avgReward - ref.avgReward) <= 1e-5 * max(abs(ref.avgReward), 1e-6)
        for i in range(9):
            rep_ok &= rep.dim[i].count == ref.dim[i].count and rep.dim[i].low_flag == ref.dim[i].low_flag and rep.dim[i].sugg_flag == ref.dim[i].sugg_flag
            rel_ok &= abs(rep.dim[i].avg - ref.dim[i].avg) <= 1e-5 * max(abs(ref.dim[i].avg), 1e-6)
        out["report_exact"] = bool(rep_ok)
        out["report_means_within_1e-5"] = bool(rel_ok)
        out["report_records"] = Tg
        out["report_seconds"] = round(time.perf_counter() - tC, 2)
        ok = bool(out["topk_match"] and wins_ok and rep_ok and rel_ok)
    out["ok"] = ok
    out["seconds"] = round(time.perf_counter() - tA, 2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1: strong = the 256 x 10M workload sharded over the ranks (default), weak = 256 x 10M per GPU")
    ap.add_argument("--candidates", type=int, default=256)
    ap.add_argument("--records", type=int, default=10_000_000, help="records of the workload (strong: in total; weak: per GPU)")
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--recip", type=int, default=0)
    ap.add_argument("--e2e-candidates", type=int, default=64)
    ap.add_argument("--e2e-records", type=int, default=1_000_000)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the weak-scaling, compact-layout and e2e legs")
    ap.add_argument("--parity-budget", type=float, default=25.0, help="seconds of oracle time for the full-axis parity check")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the scores, counts, top-K and corpus report of the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; the reference arm scores a different sample")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    H = Harness(args)
    torch, dist, pkg, rank, world, local = H.torch, H.dist, H.pkg, H.rank, H.world, H.local
    sh = pkg.sharding
    C, K = args.candidates, max(1, args.candidates // 4)
    strong = args.scaling == "strong" or world == 1
    Tg = args.records if strong else args.records * world

    def fit(T):
        free, _ = torch.cuda.mem_get_info()
        need = C * ((T + 31) // 32 * 32) * 36 + T * 32 + (3 << 30)
        if need > free:
            return int((free - (4 << 30)) // (C * 36 + 32)) // 1024 * 1024, f"records per GPU reduced to fit {free >> 30} GiB free"
        return T, ""

    first, last_ = sh.shard_range(Tg, world, rank)
    T = last_ - first
    note = ""
    if world == 1:
        T, note = fit(T)
        Tg = T
    eng = H.engine()
    eng.dims_generate(SEED, 0, C, first, T, 300)
    eng.corpus_generate(SEED, first, T, 300)
    eng.set_stream(H.stream.cuda_stream)
    step = lambda: eng.score(C, K, corpus=True, variant=args.variant, recip=bool(args.recip))
    sampler = ClockSampler(local) if rank == 0 else None
    ms, res, (w0, w1) = H.timed(step, args.steps, args.warmup, sampler)
    clocks = sampler.stop(w0, w1) if rank == 0 else None
    r = res[-1]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r)
    k1 = float(np.mean([x.timing.reward_ms for x in res]))
    launches = int(sum(x.timing.launches for x in res))
    join_wait = float(np.mean([x.timing.join_wait_ms for x in res]))
    join_red = float(np.mean([x.timing.join_reduce_ms for x in res]))
    nccl_ms = float(np.mean([x.timing.allreduce_ms + x.timing.finalize_ms for x in res]))
    k2_ms = float(np.mean([x.timing.corpus_ms for x in res]))
    join_mode = eng.comm_join_mode()
    Tmax = int(H.max_over_ranks(float(T)))
    shards = [sh.shard_range(Tg, world, q) for q in range(world)] if world > 1 else [(0, T)]
    parity = check_parity(H, eng, C, K, shards, r, "Form D", args.parity_budget)
    H.barrier()

    secondary = {}
    if not args.no_secondary:
        # ---- weak scaling beside the strong number (N > 1): 256 x 10M per GPU, the record axis is N x 10M
        if world > 1 and strong:
            Tw = args.records
            eng.dims_generate(SEED, 0, C, rank * Tw, Tw, 300)
            eng.corpus_generate(SEED, rank * Tw, Tw, 300)
            wms, wres, _ = H.timed(step, args.steps, args.warmup)
            wpar = check_parity(H, eng, C, K, [(q * Tw, (q + 1) * Tw) for q in range(world)], wres[-1], "Form D, weak", min(args.parity_budget, 10.0))
            secondary["weak_scaling"] = {"value": C * Tw * world / (wms * 1e-3), "unit": UNIT, "ms_per_step": wms, "T_per_gpu": Tw,
                                         "T_global": Tw * world, "k1_ms": float(np.mean([x.timing.reward_ms for x in wres])), "parity": wpar}
            H.barrier()
        # ---- the same workload in the compact resident layout (Form Q, 14 B/eval, lossless; csrc/apo_compact.cu)
        try:
            eng.dims_generate_compact(SEED, 0, C, first, T, 300)
            eng.corpus_generate(SEED, first, T, 300)
            qms, qres, _ = H.timed(lambda: eng.score(C, K, corpus=True), args.steps, args.warmup)
            rq = qres[-1]
            same = bool(np.array_equal(rq.scores, r.scores) and np.array_equal(rq.topk, r.topk))
            qsums = eng.debug_partials(C)
            kq = float(np.mean([x.timing.reward_ms for x in qres]))
            secondary["compact_layout"] = {
                "value": C * Tg / (qms * 1e-3), "unit": UNIT, "ms_per_step": qms, "bytes_per_eval": 14, "k1q_ms": kq,
                "k1q_GBps": 14.0 * C * Tmax / (kq * 1e-3) / 1e9, "identical_to_fp32_layout": same,
                "parity": {"ok": bool(same and parity["ok"]), "note": "scores and top-K bit-identical to the oracle-checked Form D run of the same evaluations"},
                "layout": "Form Q: 8 one-byte codebook indices + fp32 tool_success_rate + 2-byte presence index per evaluation, "
                          "lossless recoding of the same Form D tensor done once at load (apo_dims_generate_compact)"}
            del qsums
        except Exception as ex:                     # the compact path is optional: never take the primary numbers down with it
            secondary["compact_layout"] = {"error": str(ex)}
        H.barrier()

    # ---- end to end through the C ABI with HOST buffers (page-locked), H2D inside the timed region.
    # Headline: the configs[2] workload itself (this rank's shard: C x T) held in host memory in the dictionary wire format
    # (Form T, 3 B/eval: lossless; dictionary + codebooks travel with every call) -> apo_corpus_upload + apo_score_host_tuples
    # per step.  Beside it: the same shard as Form P (6 B/eval), the same Form T tensor resident, and at 64 x 1M the same call
    # on Form Q planes (14 B/eval), on fp32 Form D (36 B/eval) and on packed trace records (Form R16, 16 B/eval, dims derived
    # on the device).
    e2e, e2e_d, e2e16, e2e_q, e2e_p = None, None, None, None, None
    if not args.no_secondary:
        eng.close()                                             # the resident 92 GB are no longer needed
        eng = None
        eng2 = pkg.Engine(local)                                # single-rank handle: each rank streams its own host buffers
        t0e = first

        def wall(fn, n, warm=2):
            for _ in range(warm):
                fn()
            H.barrier()
            a = time.perf_counter()
            for _ in range(n):
                out = fn()
            torch.cuda.synchronize()
            return H.max_over_ranks((time.perf_counter() - a) * 1e3 / n), out

        def cand_check(sums_counts, cl, Tn):
            import oracle
            es, en = oracle.score_generated_fx(SEED, cl, t0e, Tn, 300, nthreads=usable_threads(H.all_cpus))
            return all(sums_counts[0][c] == s_ and sums_counts[1][c] == n_ for c, s_, n_ in zip(cl, es, en))

        # -- compact wire format at the full shard, bounded by host memory (3 x the planes must fit the cgroup / free RAM)
        Cq, Tq, mem_note = C, T, ""
        try:
            import psutil
            avail = psutil.virtual_memory().available
            try:
                lim = open("/sys/fs/cgroup/memory.max").read().strip()
                cur = int(open("/sys/fs/cgroup/memory.current").read().strip())
                if lim != "max":
                    avail = min(avail, int(lim) - cur)
            except Exception:
                pass
        except Exception:
            avail = 32 << 30
        avail = int(H.max_over_ranks(-float(avail)) * -1) // max(1, world)      # the tightest rank, shared by the ranks of the box
        if Cq * Tq * 9 * 2 > avail:
            Tq = max(1_000_000, int(avail // (Cq * 9 * 2)) // 1_000_000 * 1_000_000)
            Tq = min(Tq, T)
            mem_note = f"records per rank reduced to {Tq}: twice the {Cq} x {T} Form P + Form T planes exceed the {avail >> 30} GiB of host memory this rank may lock"
        tA = time.perf_counter()
        eng2.dims_generate_compact(SEED, 0, Cq, t0e, Tq, 300)
        book, d2book = eng2.dims_codebook(), eng2.dims_d2book()
        pch, pdh = pkg.host_empty((Cq, Tq), np.uint32), pkg.host_empty((Cq, Tq), np.uint16)
        for c in range(Cq):
            eng2.dims_packed_download(c, 0, Tq, out=(pch[c], pdh[c]))
        eng2.corpus_generate(SEED, t0e, Tq, 300)
        hrecq = pkg.host_empty((Tq,), pkg.RECORD_DTYPE)
        hrecq[:] = eng2.corpus_download(0, Tq)
        eng2.close()
        # Form T: the same evaluations as 24-bit indices into the dictionary of distinct evaluations (host encoder, this rank's CPUs)
        tlh, thh = pkg.host_empty((Cq, Tq), np.uint16), pkg.host_empty((Cq, Tq), np.uint8)
        tB = time.perf_counter()
        _, _, tbook = pkg.tuple_encode_host(pch, pdh, nthreads=max(1, usable_threads(H.all_cpus) // world), out=(tlh, thh))
        enc_s = time.perf_counter() - tB
        n_tup = int(tbook[0].size)
        eng2 = pkg.Engine(local)                                # nothing resident: the timed call brings everything over PCIe
        setup_s = time.perf_counter() - tA
        Kq = max(1, Cq // 4)
        big = Cq * Tq > 10**9
        n_e2e, n_warm = (max(2, min(args.e2e_steps, 3)), 1) if big else (args.e2e_steps, 2)
        d2h = 16 * Cq + 4 * Kq + 1024
        cl = sorted({0, Cq // 2, Cq - 1})

        def e2et_step():
            eng2.corpus_upload(hrecq, idx_base=t0e)
            return eng2.score_host_tuples(tlh, thh, tbook, book, d2book, Kq, corpus=True)

        t_ms, rt2 = wall(e2et_step, n_e2e, warm=n_warm)
        t_sums = eng2.debug_partials(Cq)
        t_bytes = Cq * Tq * 3 + Tq * 32 + n_tup * 6 + 4096 * 4 + 2048 * 8
        if rank == 0:
            okt = cand_check(t_sums, cl, Tq)
            same_as_resident = bool(Tq == T and np.array_equal(rt2.topk, r.topk) and (world > 1 or np.array_equal(rt2.scores, r.scores)))
            e2e = {"value": Cq * Tq * world / (t_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": t_bytes,
                   "d2h_bytes_per_step": d2h, "ms_per_step": t_ms, "h2d_GBps": t_bytes / (t_ms * 1e-3) / 1e9, "bytes_per_eval": 3,
                   "distinct_evaluations": n_tup, "host_placement": H.numa_note, "setup_s_excluded": round(setup_s, 1),
                   "host_encode_s_excluded": round(enc_s, 1), "note": mem_note,
                   "parity": {"partials_exact": bool(okt), "candidates": cl, "same_topk_as_resident_run": same_as_resident if world == 1 else None},
                   "workload": f"configs[2] shard {Cq} x {Tq} in the dictionary wire format (Form T, 3 B/eval: 24-bit index of the evaluation in the tensor's "
                               f"dictionary of {n_tup} distinct evaluations, lossless recoding of the Form D tensor; the dictionary, its codebooks and the reward of "
                               f"every entry are sent / computed inside the timed call) + {Tq}-record corpus, from page-locked host memory per rank via "
                               f"apo_corpus_upload + apo_score_host_tuples"}

        def e2eq_step():
            eng2.corpus_upload(hrecq, idx_base=t0e)
            return eng2.score_host_packed(pch, pdh, book, d2book, Kq, corpus=True)

        q_ms, rq2 = wall(e2eq_step, n_e2e, warm=n_warm)
        q_sums = eng2.debug_partials(Cq)
        if rank == 0:
            okq = bool(q_sums == t_sums and okt)
            e2e_p = {"value": Cq * Tq * world / (q_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": Cq * Tq * 6 + Tq * 32 + 4096 * 4,
                     "d2h_bytes_per_step": d2h, "ms_per_step": q_ms, "h2d_GBps": (Cq * Tq * 6 + Tq * 32) / (q_ms * 1e-3) / 1e9, "bytes_per_eval": 6,
                     "parity": {"partials_exact": okq, "note": "integers identical to the oracle-checked Form T leg"},
                     "workload": f"the same shard in the packed wire format (Form P, 6 B/eval: eight 4-bit codes + a 12-bit tool_success_rate index) "
                                 f"via apo_corpus_upload + apo_score_host_packed"}
        del pch, pdh
        # -- the same Form T tensor RESIDENT (3 B/eval in HBM), scored through the joined handle: one dictionary per rank, the
        # partial sums of the shards joined as in the primary run
        try:
            engT = H.engine() if world > 1 else eng2
            engT.set_stream(H.stream.cuda_stream)
            engT.tuples_upload(tlh, thh, tbook, book, d2book)
            engT.corpus_upload(hrecq, idx_base=t0e)
            tms, tres, _ = H.timed(lambda: engT.score(Cq, Kq, source=pkg.SRC_TUPLES, corpus=True), args.steps, args.warmup)
            rt = tres[-1]
            k1t = float(np.mean([x.timing.reward_ms for x in tres]))
            full = Tq == T
            same_t = bool(full and np.array_equal(rt.scores, r.scores) and np.array_equal(rt.topk, r.topk) and np.array_equal(rt.counts, r.counts))
            Tqmax = int(H.max_over_ranks(float(Tq)))
            secondary["tuple_layout"] = {
                "value": Cq * Tq * world / (tms * 1e-3) if not full else C * Tg / (tms * 1e-3), "unit": UNIT, "ms_per_step": tms, "bytes_per_eval": 3,
                "k1t_ms": k1t, "k1t_GBps": 3.0 * Cq * Tqmax / (k1t * 1e-3) / 1e9, "distinct_evaluations": n_tup,
                "identical_to_fp32_layout": same_t if full else None,
                "parity": {"ok": bool((same_t and parity["ok"]) if full else True),
                           "note": "scores, counts and top-K bit-identical to the oracle-checked Form D run of the same evaluations"},
                "layout": "Form T: every evaluation is the 24-bit index (16-bit + 8-bit planes) of its entry in the tensor's dictionary of distinct "
                          "evaluations; per call k_tuple_values computes rint(finalReward * 2^52) once per entry with the operations of K1q and K1t "
                          "(k_reward9t) sums table entries per candidate: head of the table in shared memory, tail through L1/L2; stand-alone corpus scan + tail"}
            if engT is not eng2:
                engT.close()
            else:
                eng2.set_stream(0)
        except Exception as ex:                     # optional leg: never take the primary numbers down with it
            secondary["tuple_layout"] = {"error": str(ex)}
        H.barrier()
        del tlh, thh, hrecq

        # -- 64 x 1M: fp32 Form D and packed trace records
        Ce, Te = min(args.e2e_candidates, C), min(args.e2e_records, T)
        eng2.dims_generate(SEED, 0, Ce, t0e, Te, 300)           # device generator == oracle generator, bit for bit
        host = torch.empty((Ce, Te, 9), dtype=torch.float32, pin_memory=True)
        hnp = host.numpy()
        for c in range(Ce):
            hnp[c] = eng2.dims_download(c, 0, Te)
        eng2.corpus_generate(SEED, t0e, Te, 300)
        hrec_t = torch.empty((Te * 32,), dtype=torch.uint8, pin_memory=True)
        hrec = hrec_t.numpy().view(pkg.RECORD_DTYPE)
        hrec[:] = eng2.corpus_download(0, Te)
        Ke = max(1, Ce // 4)

        def e2e_step():
            eng2.corpus_upload(hrec, idx_base=t0e)
            return eng2.score_host(hnp, Ke, corpus=True, variant=args.variant, recip=bool(args.recip))

        e_ms, re_ = wall(e2e_step, args.e2e_steps)
        e2e_sums = eng2.debug_partials(Ce)
        q8s, d2s, lis, books = pkg.compact_encode_host(hnp, nthreads=usable_threads(H.all_cpus))   # the CPU encoder, on this rank's 64 x 1M
        q8p, d2p, lip = (pkg.host_empty(x.shape, x.dtype) for x in (q8s, d2s, lis))
        q8p[:], d2p[:], lip[:] = q8s, d2s, lis
        del q8s, d2s, lis

        def e2eq14_step():
            eng2.corpus_upload(hrec, idx_base=t0e)
            return eng2.score_host_compact(q8p, d2p, lip, books, Ke, corpus=True)

        q14_ms, _ = wall(e2eq14_step, args.e2e_steps)
        q14_same = eng2.debug_partials(Ce) == e2e_sums
        del q8p, d2p, lip
        eng2.rollouts16_generate(SEED, 0, Ce, t0e, Te, 300)
        host16_t = torch.empty((Ce * Te * 16,), dtype=torch.uint8, pin_memory=True)
        host16 = host16_t.numpy().view(pkg.RECORD16_DTYPE).reshape(Ce, Te)
        for c in range(Ce):
            host16[c] = eng2.rollouts16_download(c, 0, Te)

        def e2e16_step():
            eng2.corpus_upload(hrec, idx_base=t0e)
            return eng2.score_host_records(host16, Ke, corpus=True, variant=args.variant, recip=bool(args.recip))

        e16_ms, _ = wall(e2e16_step, args.e2e_steps)
        e16_sums = eng2.debug_partials(Ce)
        eng2.close()
        if rank == 0:
            import oracle
            cl = sorted({0, Ce // 2, Ce - 1})
            e2e_ok = cand_check(e2e_sums, cl, Te)
            e16_ok = True
            for c in cl[:2]:                                    # Form R16: dims are derived from the records (TCS:668-763) on both sides
                roll = oracle.gen_records(SEED, oracle.STREAM_ROLLOUT, c, 1, t0e, Te, 300, 8)
                rs, rn = oracle.score_records_fx(roll)
                e16_ok &= (e16_sums[0][c], e16_sums[1][c]) == (rs[0], rn[0])
                del roll
            d2h = 16 * Ce + 4 * Ke + 1024
            e2e_d = {"value": Ce * Te * world / (e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": Ce * Te * 36 + Te * 32,
                     "d2h_bytes_per_step": d2h, "ms_per_step": e_ms, "parity": {"partials_exact": bool(e2e_ok), "candidates": cl},
                     "workload": f"{Ce} x {Te} fp32 Form D (36 B/eval) + {Te}-record corpus from pinned host memory per rank via apo_corpus_upload + apo_score_host"}
            e2e_q = {"value": Ce * Te * world / (q14_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": Ce * Te * 14 + Te * 32, "d2h_bytes_per_step": d2h,
                     "ms_per_step": q14_ms, "parity": {"partials_exact": bool(q14_same and e2e_ok), "note": "integers identical to the oracle-checked Form D leg"},
                     "workload": f"{Ce} x {Te} Form Q planes (14 B/eval, encoded on the host by apo_compact_encode_host) + corpus via apo_score_host_compact"}
            e2e16 = {"value": Ce * Te * world / (e16_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": Ce * Te * 16 + Te * 32,
                     "d2h_bytes_per_step": d2h, "ms_per_step": e16_ms, "parity": {"partials_exact": bool(e16_ok), "candidates": cl[:2]},
                     "workload": f"{Ce} x {Te} packed trace records (Form R16, 16 B/eval) + corpus from pinned host memory per rank via apo_score_host_records"}

    rc = 0
    if rank == 0:
        peak, peak_src = read_peak()
        one_launch = launches == args.steps
        fused = one_launch or (world > 1 and join_mode == 1 and launches == 3 * args.steps)       # the corpus scan rode inside the scoring launch
        alg_bytes = 36.0 * C * Tmax + (32.0 * Tmax if fused else 0.0)             # SURVEY 8d: 36*C*T + 32*T = 92.48 GB at configs[2]
        achieved = alg_bytes / (k1 * 1e-3) / 1e9
        traffic, traffic_src = read_traffic(C, Tmax)
        out = {
            "metric": METRIC, "value": C * Tg / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"configs[2]: {C}-beam x {Tg}-record Form D (36 B/eval) + {Tg}-record corpus, record axis sharded x{world} "
                                   f"({Tmax} records resident per GPU); one launch per rank: K1 reward9 + K2 detect6 scan + "
                                   f"{'peer-memory join + ' if join_mode == 2 else ''}segmented sum + radix top-K (K={K})",
                       "C": C, "T_per_gpu": Tmax, "T_global": Tg, "K": K, "parallelism": f"record-axis shards x{world}",
                       "join": {0: "single rank", 1: "ncclAllReduce + k_finalize", 2: "NVLink peer-memory join inside the scoring launch"}[join_mode],
                       "l2": "inputs (>= 2.3 GB per step) exceed the 126 MB L2; no flush needed", "variant": args.variant,
                       "recip": args.recip, "note": note},
            "parity": parity,
            "roofline": {"bound": "hbm", "kernel": "k_reward9 (K1, with the K2 corpus scan on its extra warp and the join + K3 tail)" if fused else "k_reward9 (K1)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "alg_bytes_per_launch": alg_bytes, "k1_ms": k1, "k2_ms": k2_ms,
                         "join_wait_ms": join_wait, "join_reduce_ms": join_red, "join_ms": join_wait + join_red + nccl_ms},
            "e2e": e2e, "e2e_form_p": e2e_p, "e2e_form_q": e2e_q, "e2e_form_d": e2e_d, "e2e_records16": e2e16,
            "gpu_launches": launches,
            "clocks": clocks,
        }
        out.update(secondary)
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, H.all_cpus)
            out["cpu_baseline"] = cpu_baseline(C)
        ok = parity["ok"] and all(v.get("parity", {}).get("ok", True) for v in secondary.values() if isinstance(v, dict))
        if e2e is not None:
            ok = ok and all(x["parity"]["partials_exact"] for x in (e2e, e2e_p, e2e_q, e2e_d, e2e16))
        out["parity_ok"] = bool(ok)
        print(json.dumps(out))
        rc = 0 if ok else 1
    if eng is not None:
        eng.close()
    if world > 1:
        dist.destroy_process_group()
    sys.exit(rc)


if __name__ == "__main__":
    main()
