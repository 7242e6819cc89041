"""Conflict rollback for SP-inspired decimation at the sizes of tools/prof_sid.py: seeded random 3-SAT batches of
8 x n = 100 000 and 8 x n = 1 000 000 at alpha 4.0 / 4.2, decimation fractions f in {0.01, 0.04}, rollback off and on,
T iterations, then random fill and WalkSAT with W flips.  Per cell: device-synchronised forward wall time (SP +
decimation, then fill + WalkSAT), iterations executed, decimation steps and decimation fixes (the trace, undone fixes
included), decimation fixes kept (distinct traced variables still fixed at the end), rollbacks and problems with one,
problems that ended trivial, in an SP contradiction or in a unit-propagation conflict (with rollback on: a conflict of a
one-variable step, which stands), problems still running at the iteration budget, and problems solved (CNF check of the
final prediction).  The card's name and power limit are printed with the numbers.

    python tools/prof_rollback.py [--out profiles/r4_rollback.json] [--sizes 100000,1000000] [--T 2000] [--W 100,10000]
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
from pdp_solver_b200.engine import Context  # noqa: E402
from tools.prof_sid import card  # noqa: E402

FLAG_TRIVIAL, FLAG_SOLVED, FLAG_CONTRADICTION, FLAG_UP_CONFLICT = 1, 2, 4, 8


def cell(tensors, B, f, rollback, T, W):
    gm, bvm, bfm, ef = tensors
    ctx = Context(gm, bvm, bfm, ef, batch_size=B)
    ctx.set_decimation_fraction(f)
    if rollback:
        ctx.enable_conflict_rollback()
    ctx.enable_trace(min(ctx.V, 1 << 24))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ctx.simplify()
    ctx.load_state_const(1.0 / 3.0, 1.0 / 3.0, 1.0 / 3.0, 0.5, 0.0)
    it = ctx.sp_run(T, 0.02, 100, True, sync=True)
    t1 = time.perf_counter()
    masks = ctx.get_masks()
    n_act = ctx.count_active_variables()
    if n_act:
        ctx.random_fill(torch.rand(n_act, device=gm.device))
    pred, _ = ctx.walksat(W, 0.05, None, None, seed=1, sync=True)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    solved, _ = ctx.cnf_eval(pred)
    flags, _, _ = ctx.problem_flags()
    count, _ = ctx.rollbacks()
    tr = ctx.trace()
    fl = flags.cpu().numpy()
    cnt = count.cpu().numpy()
    av = masks["av"].cpu().numpy()
    kept = int((av[np.unique(tr[:, 1].numpy())] == 0).sum()) if tr.shape[0] else 0
    row = dict(f=f, rollback=bool(rollback), T=T, W=W, forward_s=round(t2 - t0, 4), sp_decimation_s=round(t1 - t0, 4),
               fill_walksat_s=round(t2 - t1, 4), iterations=int(it),
               decimation_steps=int(np.unique(tr[:, 0].numpy()).shape[0]) if tr.shape[0] else 0,
               decimation_fixes=int(tr.shape[0]), fixes_kept=kept, rollbacks=int(cnt.sum()),
               problems_rolled_back=int((cnt > 0).sum()), active_variables_left=int(n_act),
               trivial=int(((fl & FLAG_TRIVIAL) != 0).sum()), contradiction=int(((fl & FLAG_CONTRADICTION) != 0).sum()),
               up_conflict=int(((fl & FLAG_UP_CONFLICT) != 0).sum()),
               at_budget=int(masks["active"].cpu().numpy().astype(bool).sum()), solved=int((solved > 0.5).sum().item()))
    del ctx
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="100000,1000000")
    ap.add_argument("--alphas", default="4.0,4.2")
    ap.add_argument("--fractions", default="0.01,0.04")
    ap.add_argument("--T", type=int, default=2000)
    ap.add_argument("--W", default="100,10000")
    ap.add_argument("--B", type=int, default=8)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_rollback.py measures on the GPU; no CUDA device")
    res = {"card": card(), "cells": []}
    print(json.dumps(res["card"]), flush=True)
    dev = torch.device("cuda:0")
    for n in [int(x) for x in a.sizes.split(",")]:
        for alpha in [float(x) for x in a.alphas.split(",")]:
            batch = cnfgen.random_batch(a.B, n, 3, alpha, 1000 + n // 1000 + int(alpha * 10))   # prof_sid.py's seeds
            tensors = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in batch]
            for f in [float(x) for x in a.fractions.split(",")]:
                for rollback in (False, True):
                    for W in [int(x) for x in a.W.split(",")]:
                        row = dict(B=a.B, n=n, alpha=alpha)
                        row.update(cell(tensors, a.B, f, rollback, a.T, W))
                        res["cells"].append(row)
                        print(json.dumps(row), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
