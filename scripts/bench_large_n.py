"""Throughput and stage times of problems above and around the 32 768-correspondence clique-kernel limit (ball model,
inputs resident in HBM, tzr_solve_batch_dev).  Above 32 768 the clique stage runs the large-n front end (greedy clique
and (L-1)-core peel on the full graph) and the existing search on the compacted core; the call waits once on the host
for the batch's largest core.

    python scripts/bench_large_n.py [--steps 3] [--warmup 1] [--out profiles/r03_bench_large_n.json]

Per (n, outlier ratio, B): registrations/s (host clock around the timed steps, which end in a device synchronise),
per-stage ms (graph kernels | degrees + clique front end + search | rotation + translation), the graph stage against the HBM byte model of bench.py, and the
device memory the context holds (cudaMemGetInfo before the context exists and after the largest run).  The card name
and power limit are read in the same run."""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def bytes_graph(n):
    """bench.py's algorithmic bytes of the graph stage per problem: src+dst in (FP64), bitset + degrees out."""
    return 48 * n + 8 * n * ((n + 63) // 64) + 4 * n


def card_info():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim, clk = [x.strip() for x in out.split(",")]
        return dict(name=name, power_limit=plim, sm_max_clock=clk)
    except Exception as e:  # the numbers are then reported without it
        return dict(name=None, power_limit=None, error=str(e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--sizes", default="32768,40000,65536,131072")
    ap.add_argument("--ratios", default="0.95,0.99")
    ap.add_argument("--batches", default="1,4")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_bench_large_n.json"))
    args = ap.parse_args()

    import torch
    capi = importlib.import_module("teaser-plusplus_b200.capi")
    synth = importlib.import_module("teaser-plusplus_b200.synth")
    torch.cuda.init()
    free0, total = torch.cuda.mem_get_info(0)
    ctx = capi.Context(0)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    rows = []
    for n in [int(x) for x in args.sizes.split(",")]:
        for ratio in [float(x) for x in args.ratios.split(",")]:
            for B in [int(x) for x in args.batches.split(",")]:
                prs = [synth.make_problem(n, ratio, 7000 + 100 * b + n % 97, "ball") for b in range(B)]
                src = torch.tensor(np.stack([q["src"] for q in prs]), device="cuda")
                dst = torch.tensor(np.stack([q["dst"] for q in prs]), device="cuda")
                sol = torch.zeros(B * capi.SOLUTION_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
                p = capi.default_params(noise_bound=prs[0]["noise_bound"], estimate_scaling=0,
                                        rotation_cost_threshold=1e-12)

                def step():
                    ctx.solve_batch_dev(p, B, n, src.data_ptr(), dst.data_ptr(), sol.data_ptr())

                for _ in range(args.warmup):
                    step()
                ctx.synchronize()
                ctx.stage_log(True)
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    step()
                ctx.synchronize()
                wall = (time.perf_counter() - t0) * 1e3 / args.steps
                sums, calls = ctx.stage_log_read()
                ctx.stage_log(False)
                stage = {k: v / max(calls, 1) for k, v in sums.items()}
                sols = np.frombuffer(sol.cpu().numpy().tobytes(), dtype=capi.SOLUTION_DTYPE)
                ok = all(int(s["clique_size"]) == len(q["inliers"]) and bool(s["valid"]) for s, q in zip(sols, prs))
                step_ms = sum(stage.values())
                g_ms = stage["graph"]
                row = dict(n=n, outlier_ratio=ratio, B=B, steps=calls,
                           registrations_per_s=B / (wall * 1e-3), step_ms_host_clock=wall,
                           stage_ms=dict(prep=stage["prep"], graph=g_ms, degrees_clique=stage["clique"],
                                         rot_trans=stage["rot_trans"], sum=step_ms),
                           graph_hbm=dict(algorithmic_bytes=bytes_graph(n) * B,
                                          achieved_gbs=bytes_graph(n) * B / (g_ms * 1e-3) / 1e9 if g_ms > 0 else None,
                                          peak_gbs=peak, frac=(bytes_graph(n) * B / (g_ms * 1e-3) / 1e9 / peak) if g_ms > 0 else None,
                                          pairs_per_s=B * n * (n - 1) / 2 / (g_ms * 1e-3) if g_ms > 0 else None),
                           cliques_equal_planted_inliers=ok)
                rows.append(row)
                print(json.dumps(row), flush=True)
                del src, dst, sol
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free1, _ = torch.cuda.mem_get_info(0)
    out = dict(card=card_info(), torch_device=torch.cuda.get_device_name(0),
               device_memory=dict(total_bytes=total, context_workspace_bytes_after_largest_run=free0 - free1,
                                  note="cudaMemGetInfo before the context was created and after the last run "
                                       "(the workspace is grow-only; torch's cached input tensors are freed)"),
               timing="host clock around `steps` back-to-back tzr_solve_batch_dev calls after `warmup`, ending in a "
                      "stream synchronise; stage times "
                      "from the context's stage log (CUDA events); inputs resident in HBM, no L2 flush (one "
                      "bitset is >= 128 MB from n = 32 768 on, more than the 126 MB L2)",
               rows=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
