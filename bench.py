#!/usr/bin/env python
"""bench.py -- Gauss-Newton solves/sec of the april_graph_cholesky{,_inc} path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload all|manhattan_batch|m3500_batch|m3500_replay|manhattan_replay]
                    [--poses P] [--replay-from S] [--shard auto|on|off] [--dump-outputs DIR]

One "step" is one pass of the hot path over one batch of synthetic/fixture input:
  *_batch   one april_graph_cholesky() call on the full graph (relinearise -> assemble ->
            factor -> 2 triangular solves -> state update), node states reset to the VERTEX2
            initial estimate before every call so each call does identical work;
  *_replay  one april_graph_cholesky_inc() call of the demo-protocol pose-by-pose replay
            (includes any batch escalation it triggers).

The metric (BASELINE.json) names four workloads.  The default run (--workload all) measures all of
them in ONE JSON line: the headline keys describe `manhattan_batch` (100 k poses / 400 k factors, the
largest single-GPU configuration; K timed steps exactly), and `workloads` carries one record each for
`m3500_batch`, `m3500_replay` and `manhattan_replay` (window from pose --replay-from), every one with
its own value / e2e / roofline / cpu_baseline, timed for >= 1 s.  --workload X measures X alone.

JSON line (rank 0):
  value        solves/s with every input already resident in HBM: the GPU pipeline
               (reset + k_linearize + k_factor + k_backsolve) timed per step with CUDA events on
               the library's stream, L2 flushed between steps (outside the timed events)
  e2e.value    solves/s through the public C API (april_graph_cholesky on HOST structs): host
               pose gather, H2D, kernels, D2H of the solution, host state update all inside;
               e2e_uncached = the same with ordering + symbolic analysis redone on every call (what the
               reference does), through aprilsam_b200_invalidate_plan()
  roofline     dominant kernel k_factor; roofline_kernels = k_linearize, k_factor, k_backsolve, each with
               algorithmic bytes per launch (SURVEY.md section 8d), the live CUDA-event time of the kernel
               inside the e2e calls, and the fraction of MEASURED_PEAKS.json hbm_gbs (k_factor also against
               the FP64 peak measured live by asam_measure_fp64_peak)
  cpu_baseline the reference's own CPU implementation (oracle/_ref) on this box, 1 thread
Multi-GPU (one process per GPU, torchrun).  manhattan_batch shards ONE solve over the GPUs
(elimination-tree shards per rank, NCCL broadcast of the shard roots' update matrices and of the solution
segments, the top of the tree replicated -- DESIGN.md section 6): every rank calls april_graph_cholesky
on its copy of the graph, value = solves / max rank time, scaling "strong", and the line carries
`parity.sharded_vs_single_gpu_max_rel`.  M3500 and every incremental workload do not shard (SURVEY.md
section 8e "replicas only"): each rank runs its own replica, value = total solves / max rank time.

--dump-outputs DIR (rank 0) writes, after the timed steps, what the last timed step of every workload
handed its caller, as float64 DIR/<workload>_<array>.npy:
  *_batch   states   node states after the last timed april_graph_cholesky call (N x 3, node order)
            step     Gauss-Newton step of the last device-resident pipeline step (N x 3, elimination order)
  *_replay  states   node states after the last timed april_graph_cholesky_inc call
The inputs are seeded, so two builds run with the same arguments can be compared array for array.  Above
64 MiB in all, every array keeps the same fixed, seeded fraction of its rows.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from aprilsam_b200 import capi, datasets  # noqa: E402
from aprilsam_b200 import harness as H  # noqa: E402

METRIC = "Gauss-Newton solves/sec (batch + incremental) on M3500 & 100k-pose graph"
ALL = ["manhattan_batch", "m3500_batch", "m3500_replay", "manhattan_replay"]
MIN_TIMED_S = 1.0  # sub-workloads: timed region at least this long
DUMP_MAX_BYTES = 64 << 20


def load_workload(name: str, poses: int):
    if name.startswith("m3500"):
        d = H.PoseGraphData.load(os.path.join(ROOT, "tests", "golden", "m3500.npz"))
        label = "M3500 (3500 poses, 5453 xyt + 1 xytpos factors)"
    elif name == "manhattan_batch":
        d = datasets.manhattan_dense(poses, seed=1)
        label = f"synthetic Manhattan seed 1, {d.n_nodes} poses, {d.n_edges} xyt + 1 xytpos factors"
    elif name == "manhattan_replay":
        d = datasets.manhattan_sparse(poses, seed=1)
        label = f"synthetic Manhattan 5% closures seed 1, {d.n_nodes} poses, {d.n_edges} xyt + 1 xytpos factors"
    else:
        raise SystemExit(f"unknown workload {name}")
    return d, label


def data_kind(name: str) -> str:
    return "synthetic" if "manhattan" in name else "fixture M3500 (public dataset) + synthetic prior"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    def __init__(self, device: int, period_ms: int = 200):
        self.p = None
        self.device = device
        self.period_ms = period_ms
        self.path = os.path.join("/tmp", f"asam_clocks_{os.getpid()}.csv")

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.f = open(self.path, "w")
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", str(self.period_ms),
                                       "-i", str(self.device)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.p:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                t = [x.strip() for x in line.split(",")]
                if len(t) < 9:
                    continue
                sm.append(float(t[1]))
                mx.append(float(t[2]))
                for nm, v in zip(names, t[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(np.max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


def dist_setup(ngpus: int, backend: str | None = None):
    """One process per GPU (torchrun env).  backend "gloo" is used by the CPU tests."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    backend = backend or os.environ.get("ASAM_BENCH_BACKEND", "nccl")
    if world > 1:
        import torch
        import torch.distributed as dist
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend)
        return world, rank, local, dist
    return 1, 0, local, None


def barrier_max(dist, local, value: float) -> float:
    """Barrier, then the maximum of `value` over all ranks (device-side for NCCL)."""
    if dist is None:
        return value
    import torch
    cuda = dist.get_backend() == "nccl"
    dev = torch.device("cuda", local) if cuda else torch.device("cpu")
    t = torch.tensor([value], dtype=torch.float64, device=dev)
    dist.barrier()
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if cuda:
        torch.cuda.synchronize()
    return float(t.item())


def aggregate_rate(dist, local, world: int, steps_this_rank: int, seconds_this_rank: float) -> float:
    """Whole-job rate: every rank runs `steps_this_rank` steps of its own replica; the job takes as
    long as the slowest rank (replicas only, SURVEY.md section 8e)."""
    return world * steps_this_rank / barrier_max(dist, local, seconds_this_rank)


# ----------------------------------------------------------------------------------------------
# the reference on host cores (reference arm / cpu_baseline legs)
# ----------------------------------------------------------------------------------------------
def time_reference_batch(d, calls: int, warm: int = 1, impl: str = "reference", keep_states: bool = False):
    h = H.Harness(impl)
    h.load_full(d)
    init = d.init.copy()
    ms, first = [], None
    for i in range(warm + calls):
        h.set_states(init)
        t = h.batch()
        if i == 0 and keep_states:
            first = h.states()
        if i >= warm:
            ms.append(t)
    h.close()
    return (np.array(ms), first) if keep_states else np.array(ms)


BULK_START = 2000  # replay windows that start later are reached by one batch solve, not by replay


def replay_seek(h, d, s_begin: int):
    """Bring harness `h` to the state "first s_begin poses solved".  Small offsets replay the demo
    protocol from pose 0; large ones (SURVEY.md section 8d: a full CPU replay of 100 k poses takes
    hours) load the first s_begin poses at once, start them at the generator's ground truth (what a
    replay from pose 0 would have tracked: dead-reckoning over 50 k poses is metres off and
    Gauss-Newton diverges from there, the linear systems become numerically meaningless) and run
    two batch solves -- identical for both arms."""
    h.replay_begin(d)
    if s_begin <= BULK_START:
        h.replay_to(s_begin, want_chi2=False)
    else:
        sub = d.head(s_begin)
        h.load_full(sub)
        if sub.truth is not None:
            h.set_states(sub.truth)
        h.batch()
        h.batch()


def time_reference_replay(d, s_begin: int, steps: int, impl: str = "reference"):
    h = H.Harness(impl)
    replay_seek(h, d, s_begin)
    _, ms, info = h.replay_to(s_begin + steps, want_chi2=False)
    h.close()
    return ms, info


BUCKETS = ("naffected_le5", "naffected_6_50", "naffected_gt50", "batch_escalation")


def step_buckets(info) -> np.ndarray:
    """Bucket index per replay step: by naffected (search_tree_t.naffected after the step); a step that
    escalated to a batch solve leaves a fresh tree behind (naffected == 0, aprilsam.c:613-657) and is
    counted apart."""
    na = info[:, 0].astype(np.int64)
    b = np.where(na <= 5, 0, np.where(na <= 50, 1, 2))
    b[na == 0] = 3
    return b


def bucket_latency(ms, info) -> dict:
    b = step_buckets(info)
    out = {}
    for i, name in enumerate(BUCKETS):
        sel = ms[b == i]
        out[name] = {"steps": int(sel.size), "median_us": float(np.median(sel) * 1e3) if sel.size else None,
                     "mean_us": float(np.mean(sel) * 1e3) if sel.size else None}
    return out


def replay_start(args, d, name: str) -> int:
    if name == "m3500_replay":
        return 1
    return max(1, min(args.replay_from, d.n_nodes - 1))


def reference_record(args, name: str, d, label: str, steps: int, warmup: int, wallclock: bool = False) -> dict:
    """One workload on the unmodified reference (oracle/_ref), 1 thread."""
    if name.endswith("_batch"):
        ms = time_reference_batch(d, steps, warmup)
        sample = f"{steps} april_graph_cholesky calls on the full graph after {warmup} untimed"
        rec_extra = {}
    else:
        s0 = replay_start(args, d, name)
        ms, info = time_reference_replay(d, s0, steps)
        sample = f"demo replay steps [{s0}, {s0 + len(ms)})" + ("" if s0 <= BULK_START else f"; first {s0} poses loaded at once at ground truth + two batch solves")
        rec_extra = {"latency_by_bucket": bucket_latency(ms, info)}
        if wallclock and H.available("reference_wallclock"):
            wms, _ = time_reference_replay(d, s0, steps, impl="reference_wallclock")
            rec_extra["cpu_baseline_wallclock"] = {
                "value": len(wms) / (float(wms.sum()) / 1e3), "unit": "solves/s", "cores": 1, "kind": "reference",
                "sample": sample + "; the reference AS SHIPPED (wall-clock escalation heuristic aprilsam.c:556-559 active: "
                                   "non-deterministic, not a parity reference)"}
    total_s = float(ms.sum()) / 1e3
    val = len(ms) / total_s
    rec = {"workload": name, "graph": label, "value": val, "unit": "solves/s", "steps": int(len(ms)), "warmup": warmup,
           "ms_per_step": float(ms.mean()), "data": data_kind(name),
           "cpu_baseline": {"value": val, "unit": "solves/s", "cores": 1, "kind": "reference", "sample": sample},
           "e2e": {"value": val, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    rec.update(rec_extra)
    return rec


def run_reference(args, names, world, rank):
    if rank != 0:
        return
    if not H.available("reference"):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built (needs /root/reference at build time)"}))
        return
    recs = {}
    for i, name in enumerate(names):
        d, label = load_workload(name, args.poses)
        if i == 0:
            steps, warm = args.steps, args.warmup
        elif name == "m3500_batch":
            steps, warm = 100, 2
        elif name == "m3500_replay":
            steps, warm = d.n_nodes - 1, 0
        else:
            steps, warm = 60, 0
        recs[name] = reference_record(args, name, d, label, steps, warm, wallclock=(i > 0 or len(names) == 1))
    head = recs[names[0]]
    line = {"metric": METRIC, "value": head["value"], "unit": "solves/s", "impl": "reference", "n_gpus": args.gpus,
            "steps": head["steps"], "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": "strong" if names[0] == "manhattan_batch" and args.shard != "off" else "weak", "vs_baseline": None,
            "dtype": "f64", "data": head["data"], "config": {"workload": names[0], "graph": head["graph"]},
            "cpu_baseline": head["cpu_baseline"], "e2e": head["e2e"], "gpu_launches": 0}
    for k in ("latency_by_bucket", "cpu_baseline_wallclock"):
        if k in head:
            line[k] = head[k]
    if len(names) > 1:
        line["workloads"] = {n: recs[n] for n in names[1:]}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
# b200 arm
# ----------------------------------------------------------------------------------------------
class Ctx:
    """What every workload of one run shares."""

    def __init__(self, args, world, rank, local, dist):
        self.args, self.world, self.rank, self.local, self.dist = args, world, rank, local, dist
        self.L = capi.lib()
        self.hbm_peak, self.peak_src = peaks()
        self.fp64_peak_tf = None
        self.traffic = {}
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                self.traffic = json.load(f)
        except Exception:
            pass


def roofline_entries(ctx: Ctx, name: str, pinfo: dict, kern_ms) -> list:
    """SURVEY.md section 8d: algorithmic bytes per launch / live CUDA-event time of the kernel."""
    N, S, F = pinfo["N"], pinfo["n_slots"], pinfo["n_factors"]
    nnz_l = 9 * (pinfo["nnz_l_blocks"] - N) + 6 * N
    nnz_a = 6 * N + 9 * S
    idx = pinfo["nnz_l_blocks"]  # one 32-bit row index per 3x3 block row of L (supernodal: fewer)
    alg = {"k_linearize": 368 * F,
           "k_factor": 8 * nnz_a + 16 * nnz_l,
           "k_backsolve": 8 * nnz_l + 4 * idx + 24 * 3 * N}
    tr = ctx.traffic.get(name, {})
    out = []
    for i, k in enumerate(("k_linearize", "k_factor", "k_backsolve")):
        t = float(np.median(kern_ms[:, i])) * 1e-3 if len(kern_ms) else 0.0
        if t <= 0:
            continue
        ach = alg[k] / t / 1e9
        e = {"kernel": k + (" (+leaf kernel on large graphs)" if k != "k_linearize" else ""), "bound": "hbm", "achieved": ach,
             "peak": ctx.hbm_peak, "unit": "GB/s", "frac": ach / ctx.hbm_peak, "peak_source": ctx.peak_src,
             "algorithmic_bytes_per_launch": int(alg[k]), "avg_launch_ms": t * 1e3,
             "traffic": tr.get(k, {}).get("bytes") if isinstance(tr.get(k), dict) else (tr.get("bytes") if k == "k_factor" else None),
             "traffic_source": tr.get("source")}
        if k == "k_factor":
            e.update({"flops_per_launch": pinfo["flops"], "fp64_tflops": pinfo["flops"] / t / 1e12,
                      "fp64_peak_tflops": ctx.fp64_peak_tf,
                      "fp64_peak_source": "measured live (asam_measure_fp64_peak: DFMA loop, 512 thr/SM); tcgen05 has no FP64 kind",
                      "fp64_frac": (pinfo["flops"] / t / 1e12 / ctx.fp64_peak_tf) if ctx.fp64_peak_tf else None,
                      "note": "latency-bound: the dependent chain of supernode levels / panel steps sets the time (DESIGN.md section 4)"})
        out.append(e)
    return out


def bench_batch(ctx: Ctx, name: str, d, label: str, K: int, W: int, sharded: bool, with_cpu: bool) -> dict:
    L, dist, local, world, rank = ctx.L, ctx.dist, ctx.local, ctx.world, ctx.rank
    init = d.init.copy()
    h = H.Harness("b200")
    h.load_full(d)
    t0 = time.perf_counter()
    h.batch()  # cold call: ordering + symbolic analysis + plan upload (+ CUDA context on the first workload)
    cold_ms = (time.perf_counter() - t0) * 1e3
    first_states = h.states()
    dev = L.asam_dbg_dev_of_graph(h.graph_ptr())
    pinfo = capi.plan_info(L.asam_dbg_plan_of_param(h.param_ptr()))
    L.asam_set_timing(dev, 1)
    if ctx.fp64_peak_tf is None:
        tf = C.c_double()
        capi.check(L.asam_measure_fp64_peak(dev, C.byref(tf)), "asam_measure_fp64_peak")
        ctx.fp64_peak_tf = tf.value
    jobs = 1 if sharded else world

    # ---- e2e: through the public API, host structs in, host structs out ----------------------
    e2e_ms, kern = [], []
    launches0 = h2d0 = d2h0 = 0
    for i in range(W + K):
        h.set_states(init)  # scaffolding (the same first Gauss-Newton iteration every step), not timed
        if i == W:
            barrier_max(dist, local, 0.0)
            launches0, h2d0, d2h0 = capi.counters(dev)
        elif sharded:
            # the ranks of a sharded solve meet inside the call (NCCL exchange): without this, a rank's timed call would
            # also wait for the slowest rank's set_states() above
            barrier_max(dist, local, 0.0)
        t = h.batch()
        if i >= W:
            e2e_ms.append(t)
            kern.append(capi.kernel_ms(dev))
    launches1, h2d1, d2h1 = capi.counters(dev)
    e2e_val = aggregate_rate(dist, local, jobs, len(e2e_ms), float(np.sum(e2e_ms)) / 1e3)
    kern = np.array(kern)
    e2e_states = h.states()

    # ---- e2e with the plan rebuilt on every call (ordering + symbolic, like the reference) ---------
    n_unc = max(3, min(K, int(1.0 / max(cold_ms * 1e-3, 1e-3)) + 3)) if not sharded else 3
    unc_ms = []
    prof0 = (C.c_double * 24)()
    L.asam_dbg_profile(prof0, 1)
    for i in range(n_unc + 1):
        h.set_states(init)
        h.invalidate_plan()
        t = h.batch()
        if i >= 1:
            unc_ms.append(t)
        else:
            L.asam_dbg_profile(prof0, 1)
    prof = (C.c_double * 24)()
    L.asam_dbg_profile(prof, 1)
    plan_ms = prof[12] / max(n_unc, 1)
    unc_val = aggregate_rate(dist, local, jobs, len(unc_ms), float(np.sum(unc_ms)) / 1e3)

    # ---- device-resident: same pipeline, inputs already in HBM, CUDA events per step ----------
    h.set_states(init)
    h.batch()
    N, S, F = pinfo["N"], pinfo["n_slots"], pinfo["n_factors"]
    ms = C.c_float()
    dev_ms = []
    launches_a = capi.counters(dev)[0]
    for i in range(W + K):
        if i == W:
            launches_a = capi.counters(dev)[0]
        capi.check(L.asam_l2_flush(dev), "l2_flush")
        capi.check(L.asam_timer_start(dev), "timer")
        capi.check(L.asam_hessian_reset(dev, N, S, N, 1e-4), "reset")
        capi.check(L.asam_linearize(dev, 0, F, None), "linearize")
        capi.check(L.asam_factor_full(dev), "factor")
        capi.check(L.asam_backsolve_full(dev), "backsolve")
        capi.check(L.asam_timer_stop(dev, C.byref(ms)), "timer")
        if i >= W:
            dev_ms.append(ms.value)
    launches_dev = capi.counters(dev)[0] - launches_a
    st = C.c_int()
    L.asam_factor_status(dev, C.byref(st))
    if st.value != 0:
        raise SystemExit(f"bench.py: factorisation status {st.value}")
    step = np.empty((N, 3), dtype=np.float64)
    capi.check(L.asam_download_x(dev, 0, N, step.ctypes.data_as(C.POINTER(C.c_double))), "asam_download_x")
    value = aggregate_rate(dist, local, jobs, len(dev_ms), float(np.sum(dev_ms)) / 1e3)
    h.close()

    rec = {"workload": name, "graph": label, "value": value, "unit": "solves/s", "steps": K, "warmup": W,
           "ms_per_step": float(np.mean(dev_ms)), "data": data_kind(name),
           "e2e": {"value": e2e_val, "unit": "solves/s", "ms_per_step": float(np.mean(e2e_ms)),
                   "h2d_bytes_per_step": (h2d1 - h2d0) // max(len(e2e_ms), 1),
                   "d2h_bytes_per_step": (d2h1 - d2h0) // max(len(e2e_ms), 1)},
           "e2e_uncached": {"value": unc_val, "unit": "solves/s", "ms_per_step": float(np.mean(unc_ms)), "calls": len(unc_ms),
                            "plan_build_ms_per_call": plan_ms,
                            "note": "ordering + symbolic analysis + plan upload redone on every call (aprilsam_b200_invalidate_plan), "
                                    "as the reference does; like-for-like with cpu_baseline"},
           "gpu_launches": int(launches_dev),
           "kernel_ms": {"k_linearize": float(np.median(kern[:, 0])), "k_factor": float(np.median(kern[:, 1])),
                         "k_backsolve": float(np.median(kern[:, 2]))},
           "roofline_kernels": roofline_entries(ctx, name, pinfo, kern),
           "plan": {k: pinfo[k] for k in ("N", "nsn", "n_slots", "n_levels", "max_m", "nnz_l_blocks")},
           "cold_first_call_ms": cold_ms,
           "cache": "L2 flushed (384 MiB overwrite) between timed device-resident steps"}
    # ---- cpu baseline + parity against it (rank 0, N = 1) ----------------------------------------
    if with_cpu and rank == 0 and world == 1 and H.available("reference"):
        probe, ref_first = time_reference_batch(d, 1, 0, keep_states=True)
        calls = int(max(2, min(300, 12e3 / max(probe[0], 1e-3))))
        ms_ref = time_reference_batch(d, calls, 0)
        rec["cpu_baseline"] = {"value": calls / (float(ms_ref.sum()) / 1e3), "unit": "solves/s", "cores": 1, "kind": "reference",
                               "sample": f"{calls} april_graph_cholesky calls of the same graph (oracle/_ref, 1 thread: the reference has no threads)"}
        scale = max(1.0, float(np.abs(ref_first).max()))
        rec["parity"] = {"vs_reference_first_iteration_max_rel": float(np.abs(first_states - ref_first).max() / scale),
                         "tolerance": 1e-6}
    rec["_first_states"] = first_states
    rec["_outputs"] = {"states": e2e_states, "step": step}
    return rec


def bench_replay(ctx: Ctx, name: str, d, label: str, K: int, W: int, with_cpu: bool) -> dict:
    L, dist, local, world, rank = ctx.L, ctx.dist, ctx.local, ctx.world, ctx.rank
    s0 = replay_start(ctx.args, d, name)
    K = min(K, d.n_nodes - s0 - W)
    h = H.Harness("b200")
    replay_seek(h, d, s0)
    dev = L.asam_dbg_dev_of_graph(h.graph_ptr())
    h.replay_to(s0 + W, want_chi2=False)
    barrier_max(dist, local, 0.0)
    launches0, h2d0, d2h0 = capi.counters(dev)
    small0 = int(L.asam_small_steps(dev))
    sp = (C.c_double * 7)()
    L.asam_small_step_profile(dev, sp, 1)
    _, ms, info = h.replay_to(s0 + W + K, want_chi2=False)
    launches1, h2d1, d2h1 = capi.counters(dev)
    n_small = int(L.asam_small_steps(dev)) - small0
    L.asam_small_step_profile(dev, sp, 0)
    chi2_end = h.chi2()
    end_states = h.states()
    h.close()
    val = aggregate_rate(dist, local, world, len(ms), float(np.sum(ms)) / 1e3)
    n = max(len(ms), 1)
    rec = {"workload": name, "graph": label, "value": val, "unit": "solves/s", "steps": int(len(ms)), "warmup": W,
           "ms_per_step": float(np.mean(ms)), "data": data_kind(name),
           "window": f"replay steps [{s0 + W}, {s0 + W + len(ms)})" + ("" if s0 <= BULK_START else f"; first {s0} poses loaded at once at ground truth + two batch solves"),
           "e2e": {"value": val, "unit": "solves/s", "ms_per_step": float(np.mean(ms)), "h2d_bytes_per_step": (h2d1 - h2d0) // n,
                   "d2h_bytes_per_step": (d2h1 - d2h0) // n},
           "gpu_launches": int(launches1 - launches0),
           "latency_by_bucket": bucket_latency(ms, info),
           "fused_small_steps": {"count": n_small,
                                 "note": "steps with naffected <= 5 run as ONE launch (k_step): uploads fetched over PCIe by the kernel, "
                                         "linearize + partial re-factorisation + pruned back-substitution, results through pinned memory",
                                 "mean_us": ({k: sp[i] / n_small for i, k in enumerate(
                                     ("fetch_scatter", "linearize", "factor", "backsolve", "write_results", "host_launch_call", "host_flag_wait"))}
                                             if n_small else None)},
           "roofline_kernels": None,
           "roofline_note": "incremental steps re-factor a handful of fronts (median naffected <= 5): launch + dependency latency, "
                            "not bytes; the per-bucket latencies above are the measure"}
    if with_cpu and rank == 0 and world == 1 and H.available("reference"):
        nref = len(ms) if d.n_nodes <= 5000 else min(len(ms), 100)
        rms, rinfo = time_reference_replay(d, s0, W + nref)
        rms, rinfo = rms[W:], rinfo[W:]
        rec["cpu_baseline"] = {"value": len(rms) / (float(rms.sum()) / 1e3), "unit": "solves/s", "cores": 1, "kind": "reference",
                               "sample": f"replay steps [{s0 + W}, {s0 + W + len(rms)}) (oracle/_ref, deterministic clock)",
                               "latency_by_bucket": bucket_latency(rms, rinfo)}
        same = min(len(rms), len(ms))
        rec["parity"] = {"naffected_equal_steps": int(np.sum(info[:same, 0] == rinfo[:same, 0])), "steps_compared": int(same)}
        if H.available("reference_wallclock"):
            wms, _ = time_reference_replay(d, s0, W + nref, impl="reference_wallclock")
            wms = wms[W:]
            rec["cpu_baseline_wallclock"] = {"value": len(wms) / (float(wms.sum()) / 1e3), "unit": "solves/s", "cores": 1,
                                             "kind": "reference",
                                             "sample": "same steps, the reference AS SHIPPED (wall-clock escalation heuristic "
                                                       "aprilsam.c:556-559 active; non-deterministic, speed reference only)"}
    rec["_chi2_end"] = chi2_end
    rec["_end_states"] = end_states
    rec["_outputs"] = {"states": end_states}
    return rec


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """DIR/<name>.npy in float64; above DUMP_MAX_BYTES in all, the same seeded fraction of every array's rows."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.size * 8 for a in arrays.values())
    frac = min(1.0, DUMP_MAX_BYTES / max(total, 1))
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if frac < 1.0:
            keep = np.sort(np.random.default_rng(0).choice(len(a), size=int(len(a) * frac), replace=False))
            a = a[keep]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_b200(args, names, world, rank, local, dist):
    L = capi.lib()
    if L.asam_device_count() <= 0:
        raise SystemExit("bench.py: no CUDA device; the b200 arm has no CPU fallback")
    ctx = Ctx(args, world, rank, local, dist)
    sampler = ClockSampler(local, period_ms=int(os.environ.get("ASAM_CLOCK_PERIOD_MS", "200")))
    recs = {}
    sharded_head = False
    if rank == 0:
        sampler.start()
    for i, name in enumerate(names):
        d, label = load_workload(name, args.poses)
        is_batch = name.endswith("_batch")
        sharded = world > 1 and is_batch and (args.shard == "on" or (args.shard == "auto" and name == "manhattan_batch"))
        if sharded:
            capi.comm_init_torch(dist, local)
            capi.check(L.asam_comm_set_sharding(1), "asam_comm_set_sharding")
        if i == 0:
            K, W = args.steps, args.warmup
            sharded_head = sharded
        elif name == "m3500_batch":
            K, W = max(args.steps, 1500), max(args.warmup, 5)
        elif name == "m3500_replay":
            K, W = d.n_nodes, 0
        else:
            K, W = 1000, args.warmup
        if is_batch:
            rec = bench_batch(ctx, name, d, label, K, W, sharded, with_cpu=not args.no_cpu_baseline)
        else:
            rec = bench_replay(ctx, name, d, label, K, W, with_cpu=not args.no_cpu_baseline)
        if sharded:
            # in-line parity of the sharded solve: the same graph, one GN iteration, on this rank's GPU alone
            capi.check(L.asam_comm_set_sharding(0), "asam_comm_set_sharding")
            if rank == 0:
                with H.Harness("b200") as h1:
                    h1.load_full(d)
                    h1.batch()
                    single = h1.states()
                scale = max(1.0, float(np.abs(single).max()))
                rec.setdefault("parity", {})["sharded_vs_single_gpu_max_rel"] = float(np.abs(rec["_first_states"] - single).max() / scale)
                rec["parity"]["tolerance"] = 1e-6
            barrier_max(dist, local, 0.0)
        recs[name] = rec
    clocks = sampler.stop() if rank == 0 else {}
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {f"{n}_{k}": v for n, r in recs.items() for k, v in r["_outputs"].items()})
    for r in recs.values():
        for k in [k for k in r if k.startswith("_")]:
            del r[k]
    head = recs[names[0]]
    is_batch = names[0].endswith("_batch")
    par = (f"elimination-tree shards x{world}, top of the tree replicated, NCCL broadcast of shard root fronts and solution "
           f"segments") if sharded_head else f"replicas x{world}"
    line = {"metric": METRIC, "value": head["value"], "unit": "solves/s", "n_gpus": world, "steps": head["steps"],
            "warmup": head["warmup"], "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": "strong" if sharded_head else "weak", "vs_baseline": None, "dtype": "f64", "data": head["data"],
            "config": {"workload": names[0], "graph": head["graph"], "parallelism": par,
                       "cache": head.get("cache", "working set grows each step"), "plan": head.get("plan"),
                       "cold_first_call_ms": head.get("cold_first_call_ms"),
                       "sub_workloads": names[1:]},
            "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
            "roofline": (next((e for e in head["roofline_kernels"] if e["kernel"].startswith("k_factor")), None)
                         if head.get("roofline_kernels") else
                         {"kernel": "k_factor", "bound": "hbm", "achieved": None, "peak": ctx.hbm_peak, "unit": "GB/s", "frac": None,
                          "traffic": None, "peak_source": ctx.peak_src, "note": head.get("roofline_note")}),
            "cpu_baseline": head.get("cpu_baseline"), "clocks": clocks}
    for k in ("e2e_uncached", "kernel_ms", "roofline_kernels", "parity", "latency_by_bucket", "cpu_baseline_wallclock", "window"):
        if head.get(k) is not None:
            line[k] = head[k]
    if len(names) > 1:
        line["workloads"] = {n: recs[n] for n in names[1:]}
    print(json.dumps(line))


def main():
    os.environ.setdefault("NCCL_DEBUG", "WARN")  # (NCCL's version banner would otherwise share stdout with the JSON line)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all"] + ALL)
    ap.add_argument("--poses", type=int, default=100000)
    ap.add_argument("--replay-from", type=int, default=50000, help="manhattan_replay: first timed step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the arrays the last timed step of every workload computed as DIR/<workload>_<array>.npy")
    ap.add_argument("--shard", choices=["auto", "on", "off"], default="auto",
                    help="--gpus N > 1: shard the elimination tree of ONE solve over the GPUs (NCCL) instead of "
                         "running N replicas; auto = on for manhattan_batch (SURVEY.md section 8e)")
    args = ap.parse_args()
    names = ALL if args.workload == "all" else [args.workload]
    if args.impl == "reference":
        world = int(os.environ.get("WORLD_SIZE", "1"))
        rank = int(os.environ.get("RANK", "0"))
        run_reference(args, names, world, rank)
        return
    if args.warmup < 3:
        args.warmup = 3
    world, rank, local, dist = dist_setup(args.gpus)
    try:
        run_b200(args, names, world, rank, local, dist)
    finally:
        if dist is not None:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
