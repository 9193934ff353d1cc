#!/usr/bin/env python
"""bench.py — registrations/sec of the TEASER++ solve() hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--config C2]   # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...         # the reference algorithm on the host cores

--config selects one of the BASELINE.json configurations (SURVEY §8d); the default, C2, is the one the metric is
quoted on.  All use fixed scale (what every reference example uses) unless --estimate-scaling is given.
    C1      bunny, N=1889, 1700 outlier draws (teaser_cpp_ply; README's 0.787 s datum)       single problem
    C2      N=5000, 95 % outliers, "ball" outlier model                                        batch/GPU, weak scaling
    C2scale N=5000, 80 % outliers, ball, estimate_scaling=true (SURVEY §8 f-1)                batch 16/GPU, weak scaling
    C2cube  N=5000, 95 % outliers, "in-cube" outliers (real branch-and-bound in the clique)   batch/GPU, weak scaling
    C3      N=10000, 99 % outliers, in-cube (max-clique stress)                                batch/GPU, weak scaling
    C4      4096 problems x N=2000, 90 % outliers, sharded b mod G                            fixed batch, strong scaling
    C5      256 problems x N=8000, 97 % outliers (3DMatch shape), sharded b mod G             fixed batch, strong scaling

A "step" = one pass of solve() over this rank's batch.
  value : registrations/s with the inputs already resident in HBM (tzr_solve_batch_dev), CUDA-event timed, no host
          synchronisation between steps (stage events are kept by the library and read after the loop).
  e2e   : same metric through the host-pointer C-ABI call (tzr_solve_batch): page-locked host inputs are copied
          host->device inside the timed region, solutions + clique index sets are read back; `pageable` repeats it
          from ordinary (numpy) host memory.
  latency : one problem through tzr_solve (the drop-in solve() shape), p50 over >= 20 calls.
Inputs per step are larger than L2 for the batch configs; for the small ones an L2 flush (256 MB write) runs
between steps and is excluded from the per-stage kernel times but not from ms_per_step — see config.l2.

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (see dump_outputs), so that two builds
run with the same arguments, and therefore on the same seeded inputs, can be compared output for output.
"""
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

CONFIGS = {
    # name: (synth cfg, n, default batch per GPU (weak) or total batch (strong), scaling, description)
    "C1": dict(n=1889, batch=1, scaling="weak", desc="C1 bunny: N=1889 correspondences, 1700 outlier draws (teaser_cpp_ply), nb=0.001"),
    "C2": dict(n=5000, batch=1024, scaling="weak", desc="C2: N=5000 correspondences, 95% outliers (ball)"),
    "C2scale": dict(n=5000, batch=16, scaling="weak", estimate_scaling=True,
                    desc="C2scale: N=5000 correspondences, 80% outliers (ball) — C2's geometry at the highest outlier ratio "
                         "where the reference's TLS scale estimator still finds the scale with this outlier model (oracle: "
                         "s_hat = 7.6 instead of 1 at 90 % and 95 %, the planted inliers are then lost by reference and GPU alike)"),
    "C2cube": dict(n=5000, batch=256, scaling="weak", desc="C2cube: N=5000 correspondences, 95% outliers (in-cube)"),
    "C3": dict(n=10000, batch=32, scaling="weak", desc="C3: N=10000 correspondences, 99% outliers (in-cube, max-clique stress)"),
    "C3ball": dict(n=10000, batch=64, scaling="weak", desc="C3ball: N=10000 correspondences, 99% outliers (ball)"),
    "C4": dict(n=2000, batch=4096, scaling="strong", desc="C4: 4096 problems x N=2000, 90% outliers (ball), sharded b mod G"),
    "C5": dict(n=8000, batch=256, scaling="strong", desc="C5: 256 problems x N=8000, 97% outliers (3DMatch shape), sharded b mod G"),
}


def bytes_graph(n):
    """Algorithmic bytes of the graph stage per problem (SURVEY §8d): read src+dst (FP64), write the full
    symmetric bitset (rows padded to 64-bit words) and the degree vector."""
    return 48 * n + 8 * n * ((n + 63) // 64) + 4 * n


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        s = sorted(sm)  # median of the upper half = clocks under load (the sampler also sees idle gaps)
        return {"sm_mhz": float(np.median(s[len(s) // 2:])), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


def problem(cfg, b, synth):
    if cfg == "C1":
        return synth.bunny_problem(os.path.join(synth.GOLDEN_DIR, "bun_zipper_res3.ply"), seed=1889 + b)
    return synth.config_problem(cfg, b)


def make_batch(cfg, idx, synth):
    n = CONFIGS[cfg]["n"]
    src = np.empty((len(idx), n, 3))
    dst = np.empty((len(idx), n, 3))
    inl, nb = [], None
    for k, b in enumerate(idx):
        pr = problem(cfg, int(b), synth)
        src[k], dst[k] = pr["src"], pr["dst"]
        inl.append(pr["inliers"])
        nb = pr["noise_bound"]
    return src, dst, inl, nb


def solver_params(mod, cfg, nb, estimate_scaling):
    # C1: teaser_cpp_ply.cc:76-88 (cost threshold 0.005); the others: registration-benchmark.cc:193 (1e-12)
    return mod.default_params(noise_bound=nb, cbar2=1.0, estimate_scaling=1 if estimate_scaling else 0,
                              rotation_estimation_algorithm=0, rotation_gnc_factor=1.4, rotation_max_iterations=100,
                              rotation_cost_threshold=0.005 if cfg == "C1" else 1e-12, rotation_tim_graph=0,
                              inlier_selection_mode=0)


DUMP_BUDGET_BYTES = 63_000_000  # array data; leaves room for the .npy headers under 64 MB in all
# every solution field except stage_ms, which holds timings rather than results
DUMP_FIELDS = ("valid", "clique_size", "scale", "translation", "rotation", "clique_proven_optimal", "gnc_iterations",
               "gnc_cost", "n_rotation_inliers", "n_translation_inliers", "n_edges")


def dump_outputs(out_dir, sols, clq, problems):
    """Writes one step's results of tzr_solve_batch_dev as out_dir/<name>.npy: each field of DUMP_FIELDS in float64
    (rotation as (B, 3, 3) matrices, gnc_cost -1 where the record holds +inf), clique (B, N) float32 with the clique's
    indices and -1 past clique_size, and problem, the synth problem number of each row.  Every value is finite.  A batch
    over DUMP_BUDGET_BYTES is cut to a sample of rows drawn with a fixed seed from the batch shape alone, so that every
    build dumps the same problems."""
    B, n = clq.shape
    per_problem = 4 * n + 8 * (1 + sum(int(np.prod(sols.dtype[f].shape)) for f in DUMP_FIELDS))
    keep = DUMP_BUDGET_BYTES // per_problem
    rows = np.arange(B) if keep >= B else np.sort(np.random.default_rng(0).choice(B, size=keep, replace=False))
    sols, clq = sols[rows], clq[rows]
    arrays = {f: sols[f].astype(np.float64) for f in DUMP_FIELDS}
    arrays["rotation"] = arrays["rotation"].reshape(-1, 3, 3).transpose(0, 2, 1)  # records are column-major
    # GNC-TLS reports +inf when it stops before its first cost evaluation (every squared residual below half the squared
    # noise bound, registration.cc:791-792,814-825); costs are sums of squares, so -1 marks that case in a finite array
    arrays["gnc_cost"][np.isposinf(arrays["gnc_cost"])] = -1.0
    arrays["clique"] = np.where(np.arange(n) < sols["clique_size"][:, None], clq, -1).astype(np.float32)
    arrays["problem"] = np.asarray(problems, dtype=np.float64)[rows]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))


def workload_string(cfg, estimate_scaling, extra=""):
    sc = "unknown scale (estimate_scaling=true, the Params default)" if estimate_scaling else "fixed scale"
    return f"{CONFIGS[cfg]['desc']}, {sc}, GNC-TLS, PMC_EXACT{extra}"


ORC_STAGES = ("tims", "scale_test", "graph", "clique", "rotation", "translation", "total")


def oracle_threads(orc, want):
    """Set and report the OpenMP thread count of the CPU restatement explicitly (torchrun exports OMP_NUM_THREADS=1)."""
    L = orc.lib()
    if hasattr(L, "orc_set_num_threads"):
        L.orc_set_num_threads(int(want))
    return int(L.orc_num_threads())


def cpu_sample(cfg, estimate_scaling, synth, seed0, max_problems, budget_s, threads):
    """Times the CPU restatement of the reference algorithm (oracle) on a bounded sample of the workload.
    Returns dict(value, cores, done, seconds, stage_ms (mean per problem), p50_ms)."""
    import oracle_lib as orc
    cores = oracle_threads(orc, threads)
    pr = problem(cfg, seed0, synth)
    p = solver_params(orc, cfg, pr["noise_bound"], estimate_scaling)
    orc.solve(pr["src"], pr["dst"], p)  # warm-up (page faults, thread pool)
    done, t_total, times = 0, 0.0, []
    stage = np.zeros(7)
    for i in range(max_problems):
        pr = problem(cfg, seed0 + 1 + i, synth)
        t0 = time.perf_counter()
        out = orc.solve(pr["src"], pr["dst"], p)
        dt = time.perf_counter() - t0
        t_total += dt
        times.append(dt * 1e3)
        stage += np.asarray(out.get("stage_ms", np.zeros(8)))[:7]
        done += 1
        if t_total > budget_s:
            break
    return dict(value=done / t_total, cores=cores, done=done, seconds=t_total,
                stage_ms={k: float(v / done) for k, v in zip(ORC_STAGES, stage)}, p50_ms=float(np.median(times)))


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port; the true reference cannot be compiled here:
    Eigen/PMC absent) on the host cores, same workload/metric.  Rank 0 only."""
    if rank != 0:
        return
    synth = importlib.import_module("teaser-plusplus_b200.synth")
    cfg = args.config
    threads = os.cpu_count() or 1
    per_step = max(1, args.ref_problems_per_step)
    # bounded: at most steps*per_step problems or ~90 s of CPU work
    s = cpu_sample(cfg, args.estimate_scaling, synth, 0, args.steps * per_step, 90.0, threads)
    v = s["value"]
    steps_done = max(1, s["done"] // per_step)
    line = {
        "impl": "reference", "metric": "registrations/sec", "value": v, "unit": "registrations/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * s["seconds"] / steps_done,
        "higher_is_better": True, "scaling": CONFIGS[cfg]["scaling"], "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_string(cfg, args.estimate_scaling),
                   "sample": f"{per_step} problem(s) per step on the host cores"},
        "cpu_baseline": {"value": v, "unit": "registrations/s", "cores": s["cores"], "kind": "port",
                         "omp_threads_set_explicitly": True, "host_cpus": os.cpu_count(),
                         "sample": f"{s['done']} problems of the {cfg} workload ({s['seconds']:.1f} s), solved back to "
                                   f"back with OpenMP on {s['cores']} threads (reference restatement; Eigen/PMC "
                                   f"unavailable so the true reference cannot be built)",
                         "stage_ms_per_problem": s["stage_ms"], "latency_ms_p50": s["p50_ms"],
                         "note": "serial stages of the reference (scale test registration.cc:427-443, graph loop "
                                 ":614-619) bound the multi-thread speed-up; see stage_ms_per_problem"},
        "e2e": {"value": v, "unit": "registrations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if cfg == "C1":
        line["cpu_baseline"]["upstream_published"] = {"seconds": 0.787, "source": "reference README.md:75-77 (teaser_cpp_ply, "
                                                      "unspecified CPU); timed like teaser_cpp_ply.cc:91-93"}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--estimate-scaling", action="store_true")
    ap.add_argument("--batch", type=int, default=0, help="problems per step per GPU (weak configs) / in total (C4, C5)")
    ap.add_argument("--ref-problems-per-step", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parity-problems", type=int, default=16)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy "
                                                          "(DIR/rank<r>/ when several ranks run)")
    args = ap.parse_args()
    if CONFIGS[args.config].get("estimate_scaling"):
        args.estimate_scaling = True

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    use_dist = world > 1
    if use_dist:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    capi = importlib.import_module("teaser-plusplus_b200.capi")
    synth = importlib.import_module("teaser-plusplus_b200.synth")
    shard = importlib.import_module("teaser-plusplus_b200.shard")
    cfg = args.config
    C = CONFIGS[cfg]
    n = C["n"]
    W = max(args.warmup, 3)
    K = args.steps
    strong = C["scaling"] == "strong"
    Btot = args.batch or C["batch"]
    if strong:   # fixed batch, problem b on rank b mod G (SURVEY §8d C4/C5)
        idx = shard.shard_indices(Btot, rank, world)
        global_batch = Btot
    else:        # every rank its own batch (weak scaling)
        idx = np.arange(Btot, dtype=np.int64) + rank * 100000
        global_batch = Btot * world
    B = len(idx)

    # ---- synthetic inputs: pinned host copies + device copies
    src_h, dst_h, inliers, nb = make_batch(cfg, idx, synth)
    src_pin = torch.empty((B, n, 3), dtype=torch.float64, pin_memory=True)
    dst_pin = torch.empty((B, n, 3), dtype=torch.float64, pin_memory=True)
    src_pin.numpy()[...] = src_h
    dst_pin.numpy()[...] = dst_h
    src_d = src_pin.cuda(non_blocking=False)
    dst_d = dst_pin.cuda(non_blocking=False)
    sol_d = torch.zeros(B * capi.SOLUTION_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    clq_d = torch.zeros((B, n), dtype=torch.int32, device="cuda")
    params = solver_params(capi, cfg, nb, args.estimate_scaling)
    ctx = capi.Context(local_rank)
    base_flags = int(os.environ.get("TZR_FLAGS", "0"))  # debug / A-B switches of the library (1024 = tensor-core graph
    # kernel, 2048 = one-MUFU CUDA-core variant)
    ctx.set_flags(base_flags)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    # L2 flush between steps for working sets that would otherwise sit in the 126 MB L2
    step_bytes = B * (48 * n + n * ((n + 127) // 128) * 16)
    flush = None
    if step_bytes < 512e6:
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def step_dev():
        ctx.solve_batch_dev(params, B, n, src_d.data_ptr(), dst_d.data_ptr(), sol_d.data_ptr(), clq_d.data_ptr())

    src_np, dst_np = src_pin.numpy(), dst_pin.numpy()  # page-locked host buffers
    h_sols = np.zeros(B, dtype=capi.SOLUTION_DTYPE)
    h_clq = np.zeros((B, n), dtype=np.int32)

    def step_host(s=src_np, d=dst_np):
        # the public host-pointer call: H2D of this step's inputs, all kernels, D2H of solutions + clique sets
        return ctx.solve_batch_array(s, d, params, cliques_out=h_clq, sols_out=h_sols)

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up
    for _ in range(W):
        step_dev()
    ctx.synchronize()
    sols = np.frombuffer(sol_d.cpu().numpy().tobytes(), dtype=capi.SOLUTION_DTYPE)
    clq = clq_d.cpu().numpy()
    n_ok = sum(int(np.array_equal(clq[b, :sols[b]["clique_size"]], inliers[b])) for b in range(B))
    n_sub = sum(int(np.isin(inliers[b], clq[b, :sols[b]["clique_size"]]).all()) for b in range(B))
    # one untimed step with the debug counters on: exact re-checks of the graph filter, clique search nodes
    ctx.set_flags(base_flags | 4)
    step_dev()
    ctx.synchronize()
    counters = ctx.debug_counters()
    ctx.set_flags(base_flags)
    step_dev()
    ctx.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- timed region 1: device-resident inputs, no host synchronisation between steps
    barrier()
    l0 = ctx.kernel_launches()
    ctx.stage_log(True)
    ev_begin, ev_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev_begin.record(stream)
        for _ in range(K):
            if flush is not None:
                flush.fill_(1)
            step_dev()
        ev_end.record(stream)
        ev_end.synchronize()
        t_dev = ev_begin.elapsed_time(ev_end)
    stage_sum, n_calls = ctx.stage_log_read()
    ctx.stage_log(False)
    barrier()
    launches = ctx.kernel_launches() - l0
    if args.dump_outputs:  # sol_d / clq_d hold the last timed step's results; nothing after this writes them
        dump_sols = np.frombuffer(sol_d.cpu().numpy().tobytes(), dtype=capi.SOLUTION_DTYPE)
        dump_clq = clq_d.cpu().numpy()
    t_flush = 0.0
    if flush is not None:  # the flush writes are inside ev_begin..ev_end: measure them alone and take them out
        with torch.cuda.stream(stream):
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(stream)
            for _ in range(K):
                flush.fill_(1)
            f1.record(stream)
            f1.synchronize()
            t_flush = f0.elapsed_time(f1)
    t_dev_net = max(t_dev - t_flush, 1e-6)
    # ---- timed region 2: end to end through the host-pointer C-ABI (pinned, then pageable host memory)
    for _ in range(2):
        step_host()
    barrier()
    t_e2e = 0.0
    for _ in range(K):
        t0 = time.perf_counter()
        hsols, hcl = step_host()
        t_e2e += (time.perf_counter() - t0) * 1e3
    barrier()
    e2e_ok = sum(int(np.array_equal(hcl[b, :hsols[b]["clique_size"]], inliers[b])) for b in range(B))
    src_pg, dst_pg = np.array(src_h, copy=True), np.array(dst_h, copy=True)  # ordinary pageable numpy memory
    step_host(src_pg, dst_pg)
    barrier()
    t_pg = 0.0
    for _ in range(K):
        t0 = time.perf_counter()
        step_host(src_pg, dst_pg)
        t_pg += (time.perf_counter() - t0) * 1e3
    barrier()
    # ---- single-problem latency through tzr_solve (the shape of the reference's solve())
    lat = []
    for r in range(max(20, 3)):
        b = r % B
        t0 = time.perf_counter()
        g1 = ctx.solve(src_h[b], dst_h[b], params)
        lat.append((time.perf_counter() - t0) * 1e3)
    lat_stage = ctx.last_stage_ms()
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"),
                     dump_sols, dump_clq, idx)

    tt = torch.tensor([t_dev_net, t_e2e, t_pg], dtype=torch.float64, device="cuda")
    if use_dist:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_dev_max, t_e2e_max, t_pg_max = float(tt[0]), float(tt[1]), float(tt[2])

    if rank == 0:
        value = global_batch * K / (t_dev_max * 1e-3)
        e2e = global_batch * K / (t_e2e_max * 1e-3)
        e2e_pg = global_batch * K / (t_pg_max * 1e-3)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
        g_ms = stage_sum["graph"] / max(n_calls, 1)   # graph stage per step (operand tiles + graph kernels), CUDA events
        achieved = bytes_graph(n) * B / (g_ms * 1e-3) / 1e9
        traffic = None
        try:  # measured once with `ncu --set full`, scaled to this launch's batch
            prof = json.load(open(os.path.join(ROOT, "profiles", "graph_kernel_traffic.json")))
            if prof.get("n") == n:
                traffic = prof.get("dram_bytes_per_problem") * B
        except Exception:
            pass
        kern = ("graph_tc_kernel (+ tc_prep_kernel, tc_patch_kernel)" if base_flags & 1024 else
                "graph_strip3_kernel (+ tc_patch_kernel)" if base_flags & 2048 else "graph_strip2_kernel")
        line = {
            "metric": "registrations/sec", "value": value, "unit": "registrations/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": t_dev_max / K, "higher_is_better": True, "scaling": C["scaling"],
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": workload_string(cfg, args.estimate_scaling,
                                            f"; {'total batch ' + str(global_batch) + ' sharded b mod G' if strong else 'batch ' + str(B) + ' problems/step/GPU'}"),
                "name": cfg, "global_batch": global_batch,
                "parallelism": f"batch sharded over {world} GPU(s), no collective",
                "l2": (f"inputs larger than L2: {step_bytes / 1e6:.0f} MB of points + adjacency per step (L2 = 126 MB); no flush"
                       if flush is None else
                       f"working set {step_bytes / 1e6:.0f} MB per step: 256 MB L2 flush between steps (its {t_flush / K:.3f} ms "
                       f"per step is subtracted from ms_per_step)"),
                "dtype_note": "FP64 predicate/GNC/TLS; the graph stage classifies pairs with an FP32 interval test on centred "
                              "float copies and re-checks the undecided band in exact FP64 (bit-identical bitset)",
            },
            "e2e": {"value": e2e, "unit": "registrations/s", "h2d_bytes_per_step": int(2 * B * n * 24),
                    # what tzr_solve_batch copies back: the solution records + the used prefix of every clique row
                    "d2h_bytes_per_step": int(B * capi.SOLUTION_DTYPE.itemsize + B * int(hsols["clique_size"].max()) * 4),
                    "ms_per_step": t_e2e_max / K, "host_memory": "page-locked, contiguous (zero-staging DMA)",
                    "pageable": {"value": e2e_pg, "ms_per_step": t_pg_max / K,
                                 "host_memory": "ordinary numpy arrays (staged through the context's pinned buffer)"}},
            "latency": {"single_problem_ms_p50": float(np.median(lat)), "single_problem_ms_min": float(np.min(lat)),
                        "calls": len(lat), "api": "tzr_solve (host pointers in, solution + clique + masks out)",
                        "stage_ms_last_call": lat_stage},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": kern,
                         "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_kind": peak_kind,
                         "algorithmic_bytes_per_launch": bytes_graph(n) * B, "kernel_ms": g_ms,
                         "note": "graph stage = O(N^2) pair classification; SURVEY §8d defines its roofline against HBM "
                                 "(algorithmic bytes: points in, packed bitset + degrees out).  The binding resource is "
                                 "the per-pair arithmetic (issue 78 %, XU 64 %, FMA pipe 58 % in the ncu capture), not DRAM"},
            "stage_ms_per_step": {k_: v / max(n_calls, 1) for k_, v in stage_sum.items()},
            "counters": {"graph_exact_rechecks_per_problem": counters["filter_rechecks"] / B,
                         "clique_search_nodes_per_problem": counters["clique_nodes"] / B},
            "parity": {"timed_batch_clique_equals_planted_inliers": f"{n_ok}/{B}",
                       "timed_batch_planted_inliers_subset_of_clique": f"{n_sub}/{B}",
                       "e2e_batch_clique_equals_planted_inliers": f"{e2e_ok}/{B}",
                       "note": "ground-truth check, not parity: with in-cube / permuted outliers some outliers are consistent "
                               "with every inlier, so the maximum clique is a strict superset of the planted set (C3: 105 vs "
                               "100); parity is vs_oracle below"},
        }
        if args.estimate_scaling:
            # SURVEY §8f-1: the K-element TLS is "HBM-bound for real": sort traffic ~ 4 passes x 2K end points x 12 B.
            # The scale stage (TIM ratios, radix sort of the 2K end points, scans, arg-min) is what the "prep" stage
            # timer covers in this mode (the centring kernel is < 1 % of it).
            Kp = n * (n - 1) // 2
            sbytes = 4 * 2 * Kp * 12 * B
            s_ms = line["stage_ms_per_step"]["prep"]
            line["roofline_scale_stage"] = {
                "bound": "hbm", "kernel": "scale_pairs + cub::DeviceRadixSort (library) + tls_scan kernels",
                "achieved": sbytes / (s_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": sbytes / (s_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": sbytes, "kernel_ms": s_ms,
                "parity": "n > 256: scale to 1e-9 relative (running sums associated differently from the reference's "
                          "sequential sweep), inlier graph identical except pairs whose predicate margin is below the "
                          "scale difference (tests/test_gpu_parity.py::test_unknown_scale_large_n); n <= 256: bit-exact"}
        # rotation / translation error vs the oracle on identical inputs (metric's second half) + CPU baseline
        if args.parity_problems > 0 or not args.no_cpu_baseline:
            import oracle_lib as orc
            threads = oracle_threads(orc, os.cpu_count() or 1)
        if args.parity_problems > 0:
            errs, t_par = [], time.perf_counter()
            for b in range(min(B, args.parity_problems)):
                o = orc.solve(src_h[b], dst_h[b], solver_params(orc, cfg, nb, args.estimate_scaling))
                Rg = capi.rotation_from_solution_record(sols[b])
                errs.append((synth.angular_error(o["R"], Rg), float(np.linalg.norm(o["t"] - sols[b]["translation"])),
                             bool(np.array_equal(o["clique"], clq[b, :sols[b]["clique_size"]])),
                             abs(float(o["scale"]) - float(sols[b]["scale"]))))
                if time.perf_counter() - t_par > 90.0:
                    break
            line["parity"]["vs_oracle"] = {"rot_err_rad_max": max(e[0] for e in errs),
                                           "trans_err_m_max": max(e[1] for e in errs),
                                           "scale_err_max": max(e[3] for e in errs),
                                           "clique_identical": all(e[2] for e in errs), "problems": len(errs)}
        if not args.no_cpu_baseline:
            if world == 1:
                s = cpu_sample(cfg, args.estimate_scaling, synth, 777, 24, 20.0, threads)
                line["cpu_baseline"] = {"value": s["value"], "unit": "registrations/s", "cores": s["cores"], "kind": "port",
                                        "sample": f"{s['done']} problems of the same {cfg} workload ({s['seconds']:.1f} s), "
                                                  f"OpenMP on {s['cores']} host threads (set explicitly), reference "
                                                  f"restatement (Eigen/PMC unavailable)",
                                        "stage_ms_per_problem": s["stage_ms"], "latency_ms_p50": s["p50_ms"]}
        print(json.dumps(line), flush=True)
    ctx.close()
    if use_dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
