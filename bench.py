#!/usr/bin/env python
"""bench.py -- pivots/sec on the synthetic dense 2000x2000 fp64 LP (BASELINE.json configs[2]).

A "step" is one complete `Tableau.simplex()` of the 2001x2001 tableau (phase 1 + phase 2, about
8k pivots under the reference's partial-pricing rule).  `value` = pivots/s with the initial
tableau already resident in HBM (each step restores it device-to-device, then solves);
`e2e` = the same solve through the reference-facing call with HOST buffers: H2D upload of the
tableau from pinned memory, solve, D2H read-back of the RHS column and basis arrays, all inside
the timed region.  L2 is flushed between timed steps (the 32 MB tableau is smaller than L2; inside
a step the tableau legitimately stays L2-resident because every pivot rewrites all of it).

  python bench.py --gpus N --steps K --warmup W            # B200 arm
  python bench.py ... --dump-outputs DIR                    # B200 arm, then the last timed step's outputs as
        DIR/<name>.npy (final tableau, basis maps, status; e2e read-back; MIP solution), inputs fixed by --seed
  python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the oracle restatement of the
        reference's TypeScript path (Node.js is not available), single thread, bounded sample.

LP does not shard (SURVEY.md 8e "replicas only"): with N > 1 every rank solves its own replica
and `value` is the aggregate (weak scaling, no data-path collective).

The line also carries a `mip` block: BASELINE.json configs[4] (0/1 knapsack, 1024 binaries x 512 constraints,
seed 12345) through Model.solve() -- the path that DOES shard: each round's open nodes are dealt over the N
ranks, node LPs run in HBM node slots (jslp_slots.cuh), summaries are all-gathered and the incumbent bound
all-reduced over NCCL inside the library.  The instance has no incumbent within thousands of nodes under the
reference's best-first rule (scripts/knap_explore.py: 6000 nodes, none), so no `tolerance` terminates it in
bench time; the run is capped at --mip-nodes committed nodes and says so (strong scaling: the work is fixed).
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "pivots_per_sec_dense_lp_2000x2000_fp64"
UNIT = "pivots/s"
DUMP_BYTES = 64_000_000  # --dump-outputs budget over all files, .npy headers included


def lp_status_array(st):
    """What an LP solve reports besides the tableau, as float64 (the integers are exact)."""
    import numpy as np
    return np.array([st.feasible, st.bounded, st.evaluation, st.evaluation_raw, st.phase1_pivots, st.phase2_pivots],
                    dtype=np.float64)


def write_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each array as out_dir/<name>.npy in float64, DUMP_BYTES in all.  The budget is shared out smallest array
    first; an array larger than its share is replaced by a fixed seeded sample of its elements (row-major flat order),
    whose flat indices go to <name>_index.npy.  Same arguments, same files: two builds compare output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    header = 128  # numpy writes a 128-byte header for these 1-D / 2-D float64 arrays
    left, items = DUMP_BYTES, sorted(arrays.items(), key=lambda kv: np.asarray(kv[1]).size)
    for i, (name, a) in enumerate(items):
        a = np.asarray(a, dtype=np.float64)
        share = left // (len(items) - i)
        if a.nbytes + header <= share:
            np.save(os.path.join(out_dir, f"{name}.npy"), a)
            left -= a.nbytes + header
            continue
        n = (share - 2 * header) // 16  # value + index per sampled element
        idx = np.sort(np.random.default_rng(0).choice(a.size, size=n, replace=False))
        np.save(os.path.join(out_dir, f"{name}.npy"), a.reshape(-1)[idx])
        np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))
        left -= 16 * n + 2 * header


def algorithmic_bytes_per_pivot(H: int, W: int) -> int:
    """SURVEY.md 8d: read+write every element, pricing scan, ratio test, row/column staging."""
    return 16 * H * W + 8 * W + 16 * H + 8 * (H + W)


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples nvidia-smi clocks/throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic():
    """DRAM / L2 bytes per launch of k_pivot_step from the committed warm-cache ncu capture
    (scripts/ncu_summary.py writes profiles/r02_k_pivot_step_ncu.json); None when there is no capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_k_pivot_step_ncu.json")) as f:
            return json.load(f)
    except Exception:
        return None


def l2_copy_peak(ctx, nbytes: int):
    """L2-resident copy bandwidth [GB/s, read + write], measured live with the library's own 128-bit copy loop
    ping-ponging between two buffers of the tableau's size (2 x 32 MB stay in the 126 MB L2) -- the roof the
    in-solve streaming phase runs under: its working set, the two tableau buffers, lives in L2."""
    import ctypes as C
    from jslpsolver_b200 import _lib
    out = C.c_double()
    _lib.check(ctx.lib.jslp_debug_copy_gbs(ctx.handle, int(nbytes), 50, C.byref(out)))
    return out.value


def run_mip_leg(args, torch, dist, rank, world, outputs=None):
    """BASELINE configs[4] through the public Model.solve(); returns the `mip` block (rank 0) or None.  With
    `outputs`, the last repetition's solution is added to it."""
    import numpy as np
    import jslpsolver_b200 as J
    from jslpsolver_b200 import problems
    model = problems.knapsack_mip_model(1024, 512, seed=12345)
    K = args.mip_spec if args.mip_spec > 0 else 32 * world

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    best = None
    for rep in range(1 + args.mip_reps):  # first repetition = warm-up (graph capture, slot allocation, NCCL init)
        inst = J.Model().loadJson(model)
        inst.max_nodes = args.mip_nodes
        inst.tableau.distributed = world > 1
        inst.tableau.max_spec_batch = K
        barrier()
        t0 = time.perf_counter()
        sol = inst.solve()       # presolve, tableau build, H2D upload, branch and cut, read-back
        torch.cuda.synchronize()
        wall_ms = 1e3 * (time.perf_counter() - t0)
        barrier()
        b = inst.tableau.lastBnbStatus
        v = torch.tensor([wall_ms, b.gpu_ms, b.host_root_ms, b.host_eval_ms - b.host_root_ms + b.host_commit_ms],
                         dtype=torch.float64, device="cuda")
        c = torch.tensor([float(b.nodes_evaluated), float(b.slot_pivots), b.slot_bytes, float(b.kernel_launches)],
                         dtype=torch.float64, device="cuda")
        sl = torch.tensor([b.slot_ms], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(v, op=dist.ReduceOp.MAX)
            dist.all_reduce(c, op=dist.ReduceOp.SUM)
            dist.all_reduce(sl, op=dist.ReduceOp.MAX)
        wall, gpu_ms, root_ms, node_ms = v.tolist()
        node_lps, slot_pivots, slot_bytes, launches = c.tolist()
        rec = {"total_ms": wall, "gpu_ms": gpu_ms, "root_ms": root_ms, "node_phase_ms": node_ms,
               "committed_nodes": b.iterations, "node_lps_all_ranks": int(node_lps), "rounds": b.rounds,
               "pivots_committed": b.pivots, "result": sol.evaluation, "collectives_per_rank": b.collectives,
               "nodes_pruned": b.nodes_pruned, "slot_pivots": int(slot_pivots), "slot_ms_max_rank": sl.item(),
               "slot_bytes": slot_bytes, "launches": int(launches)}
        if outputs is not None and rep == args.mip_reps:  # read back before the tableau is closed
            values = sol.generateSolutionSet()
            outputs.update(mip_solution=np.array([values.get(v.id, 0.0) for v in inst.variables]),
                           mip_rhs=inst.tableau.rhs_column(), mip_var_index_by_row=inst.tableau.varIndexByRow,
                           mip_status=np.array([sol.feasible, sol.bounded, sol.evaluation, b.iterations, b.pivots],
                                               dtype=np.float64))
        inst.tableau.close()
        if rep > 0 and (best is None or rec["total_ms"] < best["total_ms"]):
            best = rec
    if rank != 0:
        return None
    peak, peak_src = measured_peak()
    r = best
    non_root = max(1, r["node_lps_all_ranks"] - world)  # every rank solves the root itself
    slot_gbs = r["slot_bytes"] / (r["slot_ms_max_rank"] * 1e-3) / 1e9 if r["slot_ms_max_rank"] > 0 else None
    try:  # DRAM / L2 bytes per launch of the slot batch from the committed warm-cache ncu capture
        with open(os.path.join(ROOT, "profiles", "r02_slot_batch_ncu.json")) as f:
            slot_ncu = json.load(f)
    except Exception:
        slot_ncu = None
    out = {
        "workload": f"0/1 knapsack 1024 binaries x 512 constraints (root tableau 1537x1025, 12.6 MB), seed 12345, "
                    f"BASELINE.json configs[4]; Model.solve() capped at {args.mip_nodes} committed nodes (no incumbent "
                    f"exists within thousands of nodes: a tolerance cannot end it); best of {args.mip_reps}",
        "n_gpus": world, "spec_width": K, "scaling": "strong",
        "total_ms": r["total_ms"], "branch_and_cut_ms": r["gpu_ms"], "root_lp_ms": r["root_ms"],
        "node_phase_ms": r["node_phase_ms"], "host_front_end_ms": r["total_ms"] - r["gpu_ms"],
        "committed_nodes": r["committed_nodes"], "node_lps": r["node_lps_all_ranks"], "rounds": r["rounds"],
        "node_lps_per_s": non_root / (r["node_phase_ms"] * 1e-3),
        "committed_per_s": (r["committed_nodes"] - 1) / (r["node_phase_ms"] * 1e-3),
        "whole_solve_node_lps_per_s": r["node_lps_all_ranks"] / (r["total_ms"] * 1e-3),
        "pivots_committed": r["pivots_committed"], "pivots_per_s": r["pivots_committed"] / (r["total_ms"] * 1e-3),
        "result": r["result"], "collectives_per_rank": r["collectives_per_rank"], "nodes_pruned": r["nodes_pruned"],
        "gpu_launches": r["launches"],
        "roofline": {"bound": "hbm", "kernel": "k_pivot_step<256,2,flat8> over node slots (grid (G+2) x B)",
                     "achieved": slot_gbs, "peak": peak * world, "unit": "GB/s",
                     "frac": (slot_gbs / (peak * world)) if slot_gbs else None,
                     "traffic": slot_ncu["dram_bytes_per_launch"] if slot_ncu else None,
                     "l2_bytes_per_launch": slot_ncu["lts_bytes_per_launch"] if slot_ncu else None,
                     "traffic_source": slot_ncu["source"] if slot_ncu else None,
                     "timing": "total_ms = wall clock of Model.solve() between barriers, slowest rank (presolve + tableau "
                               "build in the Python host mirror = host_front_end_ms, upload, branch and cut, read-back); "
                               "branch_and_cut_ms = CUDA events around jslp_branch_and_cut (root LP + node phase + final "
                               "re-solve)",
                     "note": "algorithmic bytes of the pivots executed in node slots (16 x rows x stride each, all "
                             "ranks) / wall time of the slot-batch graphs incl. restore, cut rows, idle slot steps "
                             "and host polls (slowest rank).  One launch of 5 slots moves 126 MB algorithmically; `traffic` is what "
                             "DRAM saw per launch in the warm-cache ncu capture (reads are served from L2 thanks to the "
                             "dead-load hint, every written line is written back once)"},
    }
    try:
        with open(os.path.join(ROOT, "profiles", f"r02_cpu_config5_cap{args.mip_nodes}.json")) as f:
            cpu = json.load(f)
        out["cpu_reference"] = {"seconds": cpu["seconds"], "node_lps_per_s": cpu["node_lps_per_s"],
                                "pivots_per_s": cpu["pivots_per_s"], "cores": 1, "kind": "port",
                                "where": "oracle/ C restatement, same capped run, measured once in the build "
                                         "container (scripts/cpu_config5.py); same pivots: "
                                         + str(cpu["pivots"] == r["pivots_committed"])}
    except Exception:
        out["cpu_reference"] = None
    return out


def cpu_sample(it, pivots: int, check_cycles: bool = True):
    """The reference's CPU path restated (oracle/, single thread) on the first `pivots` pivots; with check_cycles
    the literal O(k^2)-per-pivot checkForCycles scan (simplex.ts:415-440, the reference's default) is included."""
    from oracle import ref_model
    t = ref_model.OracleTableau(it.matrix, it.varIndexByRow, it.varIndexByCol, check_cycles=check_cycles, fast_cycles=False)
    t.set_pivot_limit(pivots)
    t0 = time.perf_counter()
    st = t.simplex()
    dt = time.perf_counter() - t0
    return st.totalPivots, dt


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    from jslpsolver_b200 import problems
    it = problems.dense_packing_lp_tableau(args.size, args.size, args.seed)
    sample = args.cpu_pivots
    for _ in range(args.warmup):
        cpu_sample(it, max(10, sample // 10))
    tot_p, tot_t = 0, 0.0
    for _ in range(args.steps):
        p, dt = cpu_sample(it, sample)
        tot_p += p
        tot_t += dt
    value = tot_p / tot_t
    cores = os.cpu_count()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": f"first {sample} pivots of the same {args.size}x{args.size} solve per step; "
                                   f"oracle/ C restatement of the reference's single-threaded TypeScript path "
                                   f"(no Node.js on this image); box has {cores} host cores, the reference can use 1"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args):
    n = args.size
    return {"workload": f"synthetic dense packing LP {n}x{n} fp64 (tableau {n + 1}x{n + 1}, seed {args.seed}, "
                        f"a~U{{1..20}}, b~U{{100..500}}, c~U{{1..50}}), BASELINE.json configs[2]; one step = one full "
                        f"simplex() solve",
            "l2": "flushed between timed steps (256 MiB write); tableau is L2-resident within a solve",
            "parallelism": "replicas (LP does not shard)", "check_cycles": True}


def run_b200(args, rank: int, world: int, local_rank: int):
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 arm has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from jslpsolver_b200 import _lib, problems
    from jslpsolver_b200.tableau import DeviceContext, GpuTableau

    # one explicit stream for everything: the library launches on it, torch events are recorded on it
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = DeviceContext(local_rank, stream.cuda_stream)
    it = problems.dense_packing_lp_tableau(args.size, args.size, args.seed)
    H, W = it.matrix.shape
    # pinned host buffers: the e2e arm uploads from these every step
    pin_M = torch.from_numpy(it.matrix).pin_memory()
    pin_vr = torch.from_numpy(it.varIndexByRow).pin_memory()
    pin_vc = torch.from_numpy(it.varIndexByCol).pin_memory()
    g = GpuTableau(1e-8, context=ctx)
    g.upload(pin_M.numpy(), pin_vr.numpy(), pin_vc.numpy(), row_capacity=H)
    if args.engine:
        g.set_option(_lib.OPT_ENGINE, args.engine)
    if args.batch:
        g.set_option(_lib.OPT_BATCH, args.batch)
    g.save()  # device-resident initial tableau
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        g.restore()
        g.simplex()
        return g.lastStatus

    out_rhs = torch.empty(H, dtype=torch.float64).pin_memory()
    out_vr = torch.empty(H, dtype=torch.int32).pin_memory()
    out_vc = torch.empty(W, dtype=torch.int32).pin_memory()

    def step_e2e():
        L = ctx.lib
        _lib.check(L.jslp_tab_upload(g.handle, pin_M.data_ptr(), pin_vr.data_ptr(), pin_vc.data_ptr(), None, W + H - 2,
                                     None, 0, 0, None))
        g.simplex()
        _lib.check(L.jslp_download(g.handle, None, out_rhs.data_ptr(), None, out_vr.data_ptr(), out_vc.data_ptr(),
                                   None, None, None))
        return g.lastStatus

    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = ctx.launches
    ms, pivots, solve_ms = 0.0, 0, 0.0
    last = None
    for _ in range(args.steps):
        flush.fill_(1)  # L2 flush between timed steps (outside the timed events)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        last = step_resident()
        e1.record(stream)
        e1.synchronize()
        ms += e0.elapsed_time(e1)
        solve_ms += last.gpu_ms
        pivots += last.phase1_pivots + last.phase2_pivots
    launches = ctx.launches - launches0
    clocks = sampler.stop()
    barrier()
    outputs = {} if args.dump_outputs and rank == 0 else None
    if outputs is not None:  # the last timed step's tableau, read back before the e2e arm overwrites it
        outputs.update(lp_matrix=g.matrix2d(), lp_var_index_by_row=g.varIndexByRow,
                       lp_var_index_by_col=g.varIndexByCol, lp_status=lp_status_array(last))

    # e2e: host buffers in, host buffers out, copies inside the timed region
    for _ in range(min(args.warmup, 2)):
        step_e2e()
    barrier()
    e_ms, e_pivots = 0.0, 0
    for _ in range(args.steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        st = step_e2e()
        e1.record(stream)
        e1.synchronize()
        e_ms += e0.elapsed_time(e1)
        e_pivots += st.phase1_pivots + st.phase2_pivots
    barrier()
    if outputs is not None:
        outputs.update(e2e_rhs=out_rhs.numpy().copy(), e2e_var_index_by_row=out_vr.numpy().copy(),
                       e2e_var_index_by_col=out_vc.numpy().copy(), e2e_status=lp_status_array(st))

    l2_gbs = l2_copy_peak(ctx, H * W * 8) if rank == 0 else None
    mip = None
    if args.mip_nodes > 0:
        try:
            mip = run_mip_leg(args, torch, dist, rank, world, outputs)
        except Exception as e:  # the LP headline must not be lost to a failure of the secondary block
            if world > 1:
                raise           # ... but a rank that drops out of the collectives must not leave the others waiting
            mip = {"error": f"{type(e).__name__}: {e}"}

    t = torch.tensor([ms, e_ms], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([pivots, e_pivots, launches], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    ms_max, e_ms_max = t.tolist()
    tot_pivots, tot_e_pivots, tot_launches = cnt.tolist()

    if rank == 0:
        value = tot_pivots / (ms_max * 1e-3)
        e2e_value = tot_e_pivots / (e_ms_max * 1e-3)
        peak, peak_src = measured_peak()
        bpp = algorithmic_bytes_per_pivot(H, W)
        # dominant kernel = k_pivot_step, one launch per pivot: average launch duration over the
        # event-timed solve region of this rank (launch gaps and the host polls are inside it, so
        # this is a conservative per-launch figure)
        per_launch_us = 1e3 * ms / max(1, pivots)
        achieved = bpp / (per_launch_us * 1e-6) / 1e9
        ncu = ncu_traffic() if args.size == 2000 else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args),
            "pivots_per_step": pivots / args.steps,
            "final": {"feasible": bool(last.feasible), "bounded": bool(last.bounded), "evaluation": last.evaluation,
                      "phase1_pivots": last.phase1_pivots, "phase2_pivots": last.phase2_pivots,
                      "engine": last.engine},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         # dram__bytes_read.sum + dram__bytes_write.sum per launch, read from the committed
                         # warm-cache capture (ncu --cache-control none, mid-solve launches); null without one
                         "traffic": ncu["dram_bytes_per_launch"] if ncu else None,
                         "traffic_source": ncu["source"] if ncu else None,
                         "l2_bytes_per_launch": ncu.get("lts_bytes_per_launch") if ncu else None,
                         "peak_source": peak_src, "kernel": "k_pivot_step<256,2,4,prefetch> (ping-pong)",
                         "bytes_per_launch": bpp, "avg_launch_us": per_launch_us,
                         "l2": {"peak": l2_gbs, "unit": "GB/s", "frac": achieved / l2_gbs if l2_gbs else None,
                                "how": "library's 128-bit copy loop ping-ponging between two tableau-sized buffers (L2-resident), measured in this run"},
                         "note": "achieved = algorithmic bytes (SURVEY 8d: 16HW+8W+16H+8(H+W)) x pivots / event-timed "
                                 "solve time, launch gaps and host polls included.  What this number is: algorithmic "
                                 "bytes over the HBM *copy* peak for a working set (two 32 MB ping-pong buffers) that "
                                 "lives in the 126 MB L2 during a solve -- DRAM traffic is a fraction of the algorithmic "
                                 "bytes (`traffic`), the binding roof of the streaming phase is L2 bandwidth (`l2`)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(H * W * 8 + (H + W) * 4),
                    "d2h_bytes_per_step": int(H * 8 + (H + W) * 4), "ms_per_step": e_ms_max / args.steps},
            "gpu_launches": int(tot_launches), "clocks": clocks,
        }
        if mip is not None:
            line["mip"] = mip
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
            line["outputs"] = {"dir": args.dump_outputs, "arrays": sorted(outputs)}
        if world == 1 and not args.no_cpu:
            p, dt = cpu_sample(it, args.cpu_pivots)
            p2, dt2 = cpu_sample(it, args.cpu_pivots, check_cycles=False)
            line["cpu_baseline"] = {
                "value": p / dt, "unit": UNIT, "cores": 1, "kind": "port",
                "value_without_cycle_check": p2 / dt2,
                "sample": f"first {p} pivots of the same solve ({dt:.1f} s with the reference's default literal "
                          f"checkForCycles scan -- cheap this early in a solve, it grows as k^2 --, {dt2:.1f} s with "
                          f"options.exitOnCycles false); oracle/ C restatement, 1 thread (the reference is "
                          f"single-threaded; box has {os.cpu_count()} host cores; no Node.js on the box)"}
        print(json.dumps(line), flush=True)
    if dist is not None:
        from jslpsolver_b200 import distributed as D
        D.destroy_communicators()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=int, default=2000)
    ap.add_argument("--seed", type=int, default=12345)
    ap.add_argument("--engine", type=int, default=0)
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--cpu-pivots", type=int, default=1500)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--mip-nodes", type=int, default=1000, help="committed-node cap of the MIP block (0 = skip it)")
    ap.add_argument("--mip-spec", type=int, default=0, help="speculation width K (0 = 32 per GPU)")
    ap.add_argument("--mip-reps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed paths returned in their last step to DIR/<name>.npy (float64, 64 MB "
                         "at most) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the B200 arm's outputs")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
