"""One n = 40 000 problem through every kernel of the large-n clique path (meant to run under compute-sanitizer):
PMC_EXACT solve (greedy clique, core peel, compaction, search on the core, map back), KCORE_HEU and PMC_HEU."""
import importlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
capi = importlib.import_module("teaser-plusplus_b200.capi")
synth = importlib.import_module("teaser-plusplus_b200.synth")

ctx = capi.Context(0)
pr = synth.make_problem(40000, 0.95, 17, "ball")
for mode, thr in ((0, 0.5), (2, 0.01), (1, 0.5)):
    g = ctx.solve(pr["src"], pr["dst"], capi.default_params(noise_bound=pr["noise_bound"], estimate_scaling=0,
                                                            inlier_selection_mode=mode, kcore_heuristic_threshold=thr))
    print("mode", mode, "valid", g["valid"], "clique", len(g["clique"]), "proven", g["proven"])
ctx.close()
