"""Model type `reinforce` fused in the persistent kernel (pdp_set_reinforce) against the step loop it replaces, and its
solved counts on the cells of tools/prof_rollback.py (profiles/r4_rollback.json).

Speed: seeded random 3-SAT at alpha 4.2, B x n in --speed-sizes; ReinforceSurveyPropagatorSolver.forward (pi 0.01,
decimation_probability 0.5, no WalkSAT) for --speed-T iterations, without a termination callback and with the trainer's:
fused on the blocked passes (the default), fused on the generic passes (PDP_B200_SP_FLAGS=1) and step by step (forced by a
coin source drawing what the step loop draws), each twice, alternating; device-synchronised wall time per iteration, the
coin draws before and after the run included.
Solved: the batches of prof_rollback.py (same seeds), ReinforceSurveyPropagatorSolver.forward with the trainer's
termination for T iterations and W WalkSAT flips (the product path: coins, fused loop, WalkSAT); iterations, problems
retired by the survey test, problems still running at the iteration budget, problems solved (CNF check of the final
prediction), next to the SID and rollback rows of profiles/r4_rollback.json for the same cells.  The card's name and power
limit are printed with the numbers.

    python tools/prof_reinforce.py [--out profiles/r5_reinforce.json] [--speed-sizes 100000,1000000] [--T 2000] [--W 100]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from pdp_solver_b200 import cnfgen  # noqa: E402
from pdp_solver_b200.nn import solver as S  # noqa: E402
from tools.prof_sid import card  # noqa: E402

PI, P_DEC = 0.01, 0.5


def standard_termination(active, prediction, sat_problem):
    raise RuntimeError("the trainer's termination is evaluated inside the library")


standard_termination._pdp_standard_termination = True


def speed(tensors, T, path, terminate, W=0):
    gm, bvm, bfm, ef = tensors
    model = S.ReinforceSurveyPropagatorSolver(gm.device, "r", pi=PI, decimation_probability=P_DEC, local_search_iterations=W)
    if path == "step loop":
        model._decimator._coin_source = lambda: torch.rand(1, device=gm.device).item()
    os.environ["PDP_B200_SP_FLAGS"] = "1" if path == "fused generic" else "0"
    torch.manual_seed(0)
    init = model.get_init_state(gm, bvm, bfm, ef, None, False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with torch.no_grad():
        (vp, _), _ = model(init_state=init, graph_map=gm, batch_variable_map=bvm, batch_function_map=bfm,
                           edge_feature=ef.reshape(-1, 1), meta_data=None, is_training=False, iteration_num=T,
                           check_termination=standard_termination if terminate else None, simplify=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    os.environ.pop("PDP_B200_SP_FLAGS")
    solved, _ = model.last_problem._ctx.cnf_eval(vp.reshape(-1))
    _, _, freeze = model.last_problem._ctx.problem_flags()
    return dict(iterations=int(model.last_iterations.item()), forward_s=round(dt, 4), ms_per_iteration=round(1e3 * dt / T, 3),
                prediction_sum=float(vp.sum().item()), solved=int((solved > 0.5).sum().item()),
                freeze_iter=freeze.cpu().numpy().tolist())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--speed-sizes", default="100000,1000000")
    ap.add_argument("--speed-T", type=int, default=50)
    ap.add_argument("--sizes", default="100000,1000000")
    ap.add_argument("--alphas", default="4.0,4.2")
    ap.add_argument("--T", type=int, default=2000)
    ap.add_argument("--W", type=int, default=100)
    ap.add_argument("--B", type=int, default=8)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_reinforce.py measures on the GPU; no CUDA device")
    res = {"card": card(), "speed": [], "cells": []}
    print(json.dumps(res["card"]), flush=True)
    dev = torch.device("cuda:0")
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "r4_rollback.json")) as fh:
        r4 = json.load(fh)["cells"]
    for n in [int(x) for x in a.speed_sizes.split(",") if x]:
        batch = cnfgen.random_batch(a.B, n, 3, 4.2, 1000 + n // 1000 + 42)
        tensors = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in batch]
        speed(tensors, 2, "fused blocked", False)   # warm-up: module load, allocator
        speed(tensors, 2, "fused generic", False)
        for terminate in (False, True):
            for path in ("fused blocked", "fused generic", "step loop") * 2:
                row = dict(B=a.B, n=n, alpha=4.2, path=path, T=a.speed_T, check_termination="trainer's" if terminate else None)
                row.update(speed(tensors, a.speed_T, path, terminate))
                res["speed"].append(row)
                print(json.dumps(row), flush=True)
    for n in [int(x) for x in a.sizes.split(",") if x]:
        for alpha in [float(x) for x in a.alphas.split(",")]:
            batch = cnfgen.random_batch(a.B, n, 3, alpha, 1000 + n // 1000 + int(alpha * 10))   # prof_rollback.py's seeds
            tensors = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in batch]
            row = dict(B=a.B, n=n, alpha=alpha, model="reinforce", pi=PI, decimation_probability=P_DEC, T=a.T, W=a.W)
            row.update(speed(tensors, a.T, "fused blocked", True, W=a.W))
            res["cells"].append(row)
            print(json.dumps(row), flush=True)
            for r in r4:   # SP-inspired decimation and conflict rollback on the same cell
                if r["n"] == n and r["alpha"] == alpha and r["W"] == a.W and r["T"] == a.T:
                    res["cells"].append(dict(r, model="p-d-p SID", source="profiles/r4_rollback.json"))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
