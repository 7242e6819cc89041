#!/usr/bin/env python3
"""bench.py -- SATYR p-d-p hot path on B200: SP edge-updates/s (+ CNFs solved/s), % of HBM roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[3], the configuration the metric is quoted on at 1/2/4/8 B200): the
p-d-p model (Survey Propagation + sequential decimation) plus 100 iterations of WalkSAT on uniform
random 3-SAT with n = 1,000,000 variables at m/n = 4.2, `--problems` (default 8) problems per GPU,
T = 100 iterations.  One step = one whole forward() of SurveyPropagatorSolver over that batch: graph
ingest, simplify, T x [SP sweep, decimation statistics/decisions, termination check], random fill,
WalkSAT, solution merge.  Weak scaling: every rank owns its own problems, no data-path collective.

`value`  : device-resident inputs; SP edge-updates (sum over problems of executed iterations x edges)
           divided by the time of the whole step, max over ranks.
`e2e`    : the same through the public API with HOST (pinned) batch tensors; H2D of the batch and D2H
           of the prediction + verdicts are inside the timed region.
`roofline`: the persistent SP kernel (k_sp_run) timed alone with CUDA events on its stream.
`--impl reference`: the UNMODIFIED reference (baseline/_ref or /root/reference, loaded through oracle/compat.py) on
           the host cores: its own `model(...)` forward with use_cuda=False (== satyr.py --cpu_mode,
           src/pdp/factorgraph/base.py:280-305), torch threads = cpu_count as the reference sets them, on a
           bounded sample of the workload (one smaller problem, few iterations; set-up, loop and WalkSAT timed
           separately and the whole-step figure rebuilt for the workload's T and W).  The C oracle port is the
           fallback when the reference tree is absent (`kind: "port"`).
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last step of the `value` leg returned to its caller
           (prediction, solved, unsat_clauses) as DIR/<name>.npy.  The inputs are a function of the arguments (seeded
           generator, seeded WalkSAT draws), so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALG_BYTES_PER_EDGE_UPDATE = 20.0   # SURVEY.md section 8d: q_u r + eta r + index r + eta' w + q_u' w
DUMP_BYTES = 60 * 10 ** 6          # --dump-outputs: array bytes in all, under 64 MB with the .npy headers


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config3", choices=["config0", "config1", "config2", "config3", "config4"],
                    help="BASELINE.json configs[i]; config3 (default) is the configuration the metric is quoted on")
    ap.add_argument("--problems", type=int, default=8, help="problems per GPU")
    ap.add_argument("--n", type=int, default=1000000)
    ap.add_argument("--k", type=int, default=3)
    ap.add_argument("--alpha", type=float, default=4.2)
    ap.add_argument("--iterations", type=int, default=100)
    ap.add_argument("--walksat", type=int, default=100)
    ap.add_argument("--epsilon", type=float, default=0.5)
    ap.add_argument("--tolerance", type=float, default=0.02)
    ap.add_argument("--t_max", type=int, default=100)
    ap.add_argument("--seed", type=int, default=4000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config0", action="store_true", help="skip the CNFs-solved/s measurement on BASELINE.json configs[0]")
    ap.add_argument("--cpu-problem-n", type=int, default=100000, help="n of the CPU sample problem (0: --n)")
    ap.add_argument("--cpu-iterations", type=int, default=3)
    ap.add_argument("--cpu-walksat", type=int, default=2)
    ap.add_argument("--cpu-port", action="store_true", help="time the C oracle port even when the reference is present")
    ap.add_argument("--strong-problems", type=int, default=64, help="problems of the fixed batch of the strong-scaling line (0: skip it)")
    ap.add_argument("--strong-n", type=int, default=0, help="variables per problem of that batch (0: --n)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="B200 arm: write the outputs of the last timed step as DIR/<name>.npy (an output too large for the "
                         "%d-byte budget is replaced by a fixed, seeded sample of its elements)" % DUMP_BYTES)
    return ap.parse_args()


def dump_outputs(out_dir, outputs):
    """outputs: name -> 1-D float32 / float64 numpy array.  Smallest first, each is written whole while it fits in what is
    left of DUMP_BYTES; one that does not is cut to the elements at sorted indices drawn by numpy's default_rng(0)."""
    os.makedirs(out_dir, exist_ok=True)
    room = DUMP_BYTES
    for name, x in sorted(outputs.items(), key=lambda kv: kv[1].nbytes):
        keep = room // x.itemsize
        if x.size > keep:
            x = x[np.sort(np.random.default_rng(0).choice(x.size, keep, replace=False))]
        room -= x.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), x)


def config_of(a):
    """the `config` object of the JSON line: a function of the arguments only, identical in both arms"""
    m = int(a.n * a.alpha)
    E, V, F = a.k * m * a.problems, a.n * a.problems, m * a.problems
    from pdp_solver_b200.nn import solver as pdp_solver
    return {"workload": workload_name(a), "model_type": "p-d-p", "edges_per_gpu": E, "variables_per_gpu": V,
            "clauses_per_gpu": F, "init": "deterministic (predict path)",
            "rng": "torch" if a.walksat * (V + a.problems) <= pdp_solver.TORCH_RNG_DRAW_LIMIT else "philox",
            "l2": "inputs larger than L2 (%.1f GB message+topology working set per GPU)" % (E * 48 / 1e9),
            "sharding": "problems sharded across ranks, no per-iteration collective"}


def workload_name(a):
    return "p-d-p SP + %d-iteration WalkSAT, random %d-SAT n=%d m/n=%.2f, %d problems/GPU, T=%d" % (
        a.walksat, a.k, a.n, a.alpha, a.problems, a.iterations)


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.samples.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx = max(mx, float(s[1]))
                for nme, v in zip(names, s[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU arm: the reference itself (oracle/ref_timing.py) or, when its tree is absent, the C oracle port
# --------------------------------------------------------------------------------------------------
def port_forward(batch, T, W, tol, t_max, eps, seed):
    """one forward() of the C oracle port; returns dict like ref_timing.timed_forward"""
    from oracle import pdp_oracle as po
    gm, bvm, bfm, ef = batch
    E = gm.shape[1]
    rng = np.random.default_rng(seed)
    t0 = time.perf_counter()
    o = po.Oracle(gm, bvm, bfm, ef, strict=False)
    o.simplify()
    o.set_state(*po.init_state(E, False))
    t1 = time.perf_counter()
    done = o.run(T, tol, t_max, True)
    t2 = time.perf_counter()
    n_act = o.count_active_variables()
    if n_act:
        o.random_fill(rng.random(n_act, dtype=np.float32))
    rv = rng.random((max(W, 1), o.V), dtype=np.float32)
    rc = rng.random((max(W, 1), o.B), dtype=np.float32)
    t3 = time.perf_counter()
    pred, _ = o.local_search(W, eps, rv, rc)
    t4 = time.perf_counter()
    solved, _ = o.cnf_eval(pred)
    t5 = time.perf_counter()
    return {"total_s": t5 - t0, "loop_s": t2 - t1, "walksat_s": t4 - t3, "setup_s": (t1 - t0) + (t3 - t2) + (t5 - t4),
            "iterations": int(done), "solved": int(solved.sum()), "edges": int(E)}


class CpuArm(object):
    """the reference's CPU path on a bounded sample of the workload"""

    def __init__(self, a):
        import torch
        from pdp_solver_b200 import cnfgen
        from oracle import ref_timing
        self.a = a
        self.n = a.cpu_problem_n or a.n
        self.batch = cnfgen.random_batch(1, self.n, a.k, a.alpha, a.seed + 999)
        self.kind = "reference" if (ref_timing.available() and not a.cpu_port) else "port"
        if self.kind == "reference":
            self.cores = ref_timing.pin_threads()
            self.model = ref_timing.build_model("p-d-p", torch.device("cpu"), a.cpu_walksat, a.epsilon, a.tolerance, a.t_max)
        else:
            from oracle import pdp_oracle as po
            po.build()
            po.set_num_threads(os.cpu_count() or 1)
            self.cores = po.num_threads()
        self.sample = ("1 problem of n=%d (workload: n=%d), T=%d SP iterations + %d WalkSAT iterations per step; set-up / "
                       "loop / WalkSAT timed separately; `value` = whole-step rate rebuilt for the workload's T=%d, W=%d "
                       "from the measured per-iteration costs") % (self.n, a.n, a.cpu_iterations, a.cpu_walksat, a.iterations, a.walksat)

    def step(self, seed):
        if self.kind == "reference":
            import torch
            from oracle import ref_timing
            return ref_timing.timed_forward(self.model, self.batch, self.a.cpu_iterations, torch.device("cpu"), seed=seed)
        a = self.a
        return port_forward(self.batch, a.cpu_iterations, a.cpu_walksat, a.tolerance, a.t_max, a.epsilon, seed)

    def summarize(self, runs):
        """per-iteration costs of the sample and the whole-step rate they give at the workload's T and W"""
        a = self.a
        E = runs[0]["edges"]
        it = sum(r["iterations"] for r in runs)
        loop = sum(r["loop_s"] for r in runs)
        s_it = loop / max(it, 1)
        s_ws = sum(r["walksat_s"] for r in runs) / max(a.cpu_walksat * len(runs), 1)
        setup = sum(r["setup_s"] for r in runs) / len(runs)
        step_s = setup + a.iterations * s_it + a.walksat * s_ws
        return {"value": E * a.iterations / step_s, "unit": "edge-updates/s", "cores": self.cores, "kind": self.kind,
                "sample": self.sample, "loop_edge_updates_per_s": E / s_it if s_it > 0 else None,
                "s_per_sp_iteration": s_it, "s_per_walksat_iteration": s_ws, "setup_s": setup,
                "sample_edges": E, "measured_step_s": sum(r["total_s"] for r in runs) / len(runs)}


def reference_gpu_probe(a):
    """second comparator: the reference's own CUDA branch (torch sparse on the same B200), one small forward"""
    try:
        import torch
        from oracle import ref_timing
        from pdp_solver_b200 import cnfgen
        if not (torch.cuda.is_available() and ref_timing.available()):
            return {"unavailable": "no CUDA device or no reference tree"}
        dev = torch.device("cuda", 0)
        n = a.cpu_problem_n or a.n
        batch = cnfgen.random_batch(1, n, a.k, a.alpha, a.seed + 999)
        model = ref_timing.build_model("p-d-p", dev, a.cpu_walksat, a.epsilon, a.tolerance, a.t_max)
        T = 10
        ref_timing.timed_forward(model, batch, 2, dev)
        r = ref_timing.timed_forward(model, batch, T, dev)
        s_it = r["loop_s"] / max(r["iterations"], 1)
        return {"what": "reference CUDA branch (torch sparse) on cuda:0, 1 problem n=%d, T=%d" % (n, T),
                "s_per_sp_iteration": s_it, "loop_edge_updates_per_s": r["edges"] / s_it if s_it > 0 else None,
                "setup_s": r["setup_s"], "s_per_walksat_iteration": r["walksat_s"] / max(a.cpu_walksat, 1)}
    except Exception as e:   # the reference's legacy sparse constructors may not survive this torch
        return {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:200])}


def run_reference_arm(a, rank, world):
    if rank != 0:
        return
    arm = CpuArm(a)
    for s in range(min(a.warmup, 1)):
        arm.step(a.seed)
    runs = []
    t0 = time.perf_counter()
    for s in range(a.steps):
        runs.append(arm.step(a.seed + s))
    wall = time.perf_counter() - t0
    cb = arm.summarize(runs)
    line = {"impl": "reference", "metric": "sp_edge_updates_per_s", "value": cb["value"], "unit": "edge-updates/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * wall / max(a.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(a), "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "edge-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "reference_gpu": reference_gpu_probe(a)}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------
def run_b200_arm(a, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from pdp_solver_b200 import cnfgen
    from pdp_solver_b200.nn import solver as pdp_solver
    from pdp_solver_b200.nn import util as pdp_util

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- synthetic batch (host, pinned) -----------------------------------------------------------
    batch = cnfgen.random_batch(a.problems, a.n, a.k, a.alpha, a.seed + 17 * rank)
    host = [torch.from_numpy(x).pin_memory() for x in batch]
    E, V, F, B = batch[0].shape[1], batch[1].shape[0], batch[2].shape[0], a.problems
    h2d_bytes = sum(int(t.numel() * t.element_size()) for t in host)
    resident = [t.to(dev, non_blocking=True) for t in host]
    edges_per_problem = torch.bincount(resident[1].long()[resident[0][0].long()], minlength=B).double()
    torch.cuda.synchronize()

    model = pdp_solver.SurveyPropagatorSolver(dev, "p-d-p", tolerance=a.tolerance, t_max=a.t_max,
                                              local_search_iterations=a.walksat, epsilon=a.epsilon)
    evaluator = pdp_util.SatCNFEvaluator(dev)

    def termination(active, prediction, sat_problem):   # evaluated inside the persistent kernel
        raise RuntimeError("unreachable")
    termination._pdp_standard_termination = True

    stats = {"updates": 0.0, "solved": 0, "launches": 0, "loop_ms": 0.0, "loop_updates": 0.0, "ws_ms": 0.0}
    out_h = {"pred": torch.empty(V, dtype=torch.float32).pin_memory(), "solved": torch.empty(B, dtype=torch.float32).pin_memory()}

    def one_step(tensors, from_host, timed):
        torch.manual_seed(1 + rank)
        if from_host and tensors[0].device.type == "cpu":     # (warm-up of the end-to-end leg)
            gm, bvm, bfm, ef = [t.to(dev, non_blocking=True) for t in tensors]
        else:
            gm, bvm, bfm, ef = tensors
        init = model.get_init_state(gm, bvm, bfm, ef, None, randomized=False, batch_replication=1)
        (pred, _), _ = model(init_state=init, graph_map=gm, batch_variable_map=bvm, batch_function_map=bfm,
                             edge_feature=ef, meta_data=None, is_training=False, iteration_num=a.iterations,
                             check_termination=termination, batch_replication=1)
        ctx = model.last_problem._ctx
        solved, n_unsat = ctx.cnf_eval(pred)
        if from_host:      # the step's result back to (pinned) host memory, then wait for it
            out_h["pred"].copy_(pred.reshape(-1), non_blocking=True)
            out_h["solved"].copy_(solved.reshape(-1), non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
        if timed:
            _, _, freeze = ctx.problem_flags()
            iters = int(model.last_iterations.item())
            per = torch.where(freeze >= 0, freeze, torch.full_like(freeze, iters)).double()
            upd = float((per * edges_per_problem).sum().item())
            stats["updates"] += upd
            stats["solved"] += int(solved.sum().item())
            stats["launches"] += ctx.launch_count() + 2   # + the evaluator's two kernels
            t = model.last_problem._ctx.timing
            if t:
                stats["loop_ms"] += t.get("sp_run", 0.0)
                stats["ws_ms"] += t.get("walksat", 0.0)
                stats["loop_updates"] += upd
        return {"prediction": pred, "solved": solved, "unsat_clauses": n_unsat}

    copy_stream = torch.cuda.Stream(dev)

    class Staged(object):
        """end-to-end leg: every step's batch is copied from pinned host memory inside the timed region, on a copy stream,
        into one of two device buffers (allocated once, before the clock starts: cudaMalloc is not part of a step) -- the
        copy of step i+1 runs under the kernels of step i (the same double buffering as
        FactorGraphTrainerBase._predict_epoch); the copy of step i+2 waits until step i has released its buffer"""

        def __init__(self, tensors):
            self.host = tensors
            with torch.cuda.stream(copy_stream):
                self.bufs = [[torch.empty(t.shape, dtype=t.dtype, device=dev) for t in tensors] for _ in range(2)]
            self.ready, self.freed = [None, None], [None, None]
            self.spans = []
            torch.cuda.synchronize()

        def copy_ms(self):
            "mean duration of one step's host-to-device copy on the copy stream (call after a synchronize)"
            return sum(b.elapsed_time(e) for b, e in self.spans) / max(len(self.spans), 1)

        def stage(self, k):
            with torch.cuda.stream(copy_stream):
                if self.freed[k & 1] is not None:
                    copy_stream.wait_event(self.freed[k & 1])
                begin = torch.cuda.Event(enable_timing=True)
                begin.record(copy_stream)
                for dst, src in zip(self.bufs[k & 1], self.host):
                    dst.copy_(src, non_blocking=True)
                self.ready[k & 1] = torch.cuda.Event(enable_timing=True)
                self.ready[k & 1].record(copy_stream)
                self.spans.append((begin, self.ready[k & 1]))

        def take(self, k):
            torch.cuda.current_stream(dev).wait_event(self.ready[k & 1])
            return self.bufs[k & 1]

        def release(self, k):
            self.freed[k & 1] = torch.cuda.Event()
            self.freed[k & 1].record(torch.cuda.current_stream(dev))

    def timed_region(tensors, from_host):
        for k in stats:
            stats[k] = 0 if isinstance(stats[k], int) else 0.0
        for _ in range(a.warmup):
            one_step(tensors, from_host, False)
        st = Staged(tensors) if from_host else None
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if from_host:
            st.stage(0)
            for i in range(a.steps):
                if i + 1 < a.steps:
                    st.stage(i + 1)
                one_step(st.take(i), True, True)
                st.release(i)
        else:
            for _ in range(a.steps):
                last = one_step(tensors, False, True)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if a.dump_outputs and not from_host and rank == 0:
            outputs.update({k: v.reshape(-1).cpu().numpy() for k, v in last.items()})
        copy_ms = st.copy_ms() if from_host else 0.0
        if world > 1:
            t = torch.tensor([ms, copy_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, copy_ms = [float(x) for x in t.tolist()]
            agg = torch.tensor([stats["updates"], stats["solved"], stats["launches"]], device=dev, dtype=torch.float64)
            dist.all_reduce(agg, op=dist.ReduceOp.SUM)
            tot_upd, tot_solved, tot_launch = [float(x) for x in agg.tolist()]
        else:
            tot_upd, tot_solved, tot_launch = stats["updates"], stats["solved"], stats["launches"]
        stats["h2d_ms"] = copy_ms
        return ms, tot_upd, tot_solved, tot_launch, dict(stats)

    os.environ["PDP_B200_TIMING"] = "1"
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    outputs = {}
    ms, upd, solved, launches, st = timed_region(resident, False)
    ms_e, upd_e, solved_e, _, st_e = timed_region(host, True)
    sampler.stop_flag = True
    if outputs:
        dump_outputs(a.dump_outputs, outputs)

    strong = None
    if a.strong_problems > 0:
        # rank 0 drives ALL the box's GPUs through the product's multi-GPU predict path; the other ranks free their
        # devices' SMs (no kernel, no NCCL call) and wait for a key in the rendezvous store
        store = dist.distributed_c10d._get_default_store() if world > 1 else None
        if rank == 0:
            try:
                del resident
                torch.cuda.empty_cache()
                strong = strong_scaling_line(a, world)
            except Exception as e:
                strong = {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:300])}
            if store is not None:
                store.set("pdp_strong_done", "1")
        else:
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            store.wait(["pdp_strong_done"])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    loop_s = st["loop_ms"] / 1e3
    achieved = ALG_BYTES_PER_EDGE_UPDATE * st["loop_updates"] / loop_s / 1e9 if loop_s > 0 else None
    # DRAM traffic of k_sp_run per launch: ncu --set full measured dram__bytes_read.sum + dram__bytes_write.sum per
    # edge-update on the same workload (profiles/k_sp_run_traffic.json), times the edge-updates of this launch
    traffic = None
    try:
        per = json.load(open(os.path.join(ROOT, "profiles", "k_sp_run_traffic.json"))).get("dram_bytes_per_edge_update")
        traffic = per * st["loop_updates"] / a.steps
    except Exception:
        pass

    line = {
        "metric": "sp_edge_updates_per_s", "value": upd / (ms / 1e3), "unit": "edge-updates/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(a),
        "cnfs_solved_per_s": solved / (ms / 1e3), "cnfs_per_s": world * B * a.steps / (ms / 1e3),
        "sp_loop_edge_updates_per_s_rank0": st["loop_updates"] / loop_s if loop_s > 0 else None,
        "phase_ms_per_step_rank0": {"sp_loop": st["loop_ms"] / a.steps, "walksat": st["ws_ms"] / a.steps,
                                    "other(ingest,simplify,fill,io)": (ms - st["loop_ms"] - st["ws_ms"]) / a.steps},
        "e2e": {"value": upd_e / (ms_e / 1e3), "unit": "edge-updates/s", "h2d_bytes_per_step": h2d_bytes * world,
                "d2h_bytes_per_step": (V * 4 + B * 4) * world, "ms_per_step": ms_e / a.steps,
                "cnfs_solved_per_s": solved_e / (ms_e / 1e3),
                # the copy of step i+1 runs on its own stream under the kernels of step i: its duration (max over ranks) and
                # rank 0's phases in this leg say whether the copy, or the kernels beside it, bend the end-to-end curve
                "h2d_ms_per_step_max_rank": st_e["h2d_ms"],
                "phase_ms_per_step_rank0": {"sp_loop": st_e["loop_ms"] / a.steps, "walksat": st_e["ws_ms"] / a.steps,
                                            "other(ingest,simplify,fill,io)": (ms_e - st_e["loop_ms"] - st_e["ws_ms"]) / a.steps}},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "k_sp_run (persistent SP propagate/decimate loop)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                     "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_edge_update": ALG_BYTES_PER_EDGE_UPDATE,
                     "edge_updates_per_launch": st["loop_updates"] / a.steps, "launch_ms": st["loop_ms"] / a.steps},
        "clocks": sampler.summary(),
    }
    if strong is not None:
        line["strong_scaling_fixed_batch"] = strong
    if not a.no_config0 and world == 1:
        line["config0_cnfs_solved"] = config0_solved(dev)
    if not a.no_cpu_baseline:
        arm = CpuArm(a)
        line["cpu_baseline"] = arm.summarize([arm.step(a.seed)])
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def strong_scaling_line(a, world):
    """A FIXED batch through the product's own multi-GPU predict path (FactorGraphTrainerBase._predict_epoch: one host
    process, one worker thread + copy/compute streams per device, DynamicBatchDivider-style segments handed out to the
    devices; replaces the reference's nn.DataParallel wrapper, src/pdp/factorgraph/base.py:96-97): `--strong-problems`
    problems of the workload's size, one per segment, pinned host tensors, H2D / D2H and the per-problem output text
    inside the timed region.  Runs in rank 0 on all `world` GPUs while the other ranks wait on the host."""
    import io
    import logging
    import torch
    from pdp_solver_b200 import cnfgen
    from pdp_solver_b200.trainer import SatFactorGraphTrainer
    n = a.strong_n or a.n
    cfg = {"model_type": "p-d-p", "model_name": "bench", "tolerance": a.tolerance, "t_max": a.t_max, "local_search_iteration": a.walksat,
           "epsilon": a.epsilon, "test_recurrence_num": a.iterations, "random_seed": a.seed, "gpus": world, "hidden_dim": 1,
           "test_batch_limit": 1 << 40, "batch_size": 1, "verbose": False}
    trainer = SatFactorGraphTrainer(cfg, True, logging.getLogger("bench"))
    distinct = []        # (eight distinct instances, cycled: generating 64 on the host would take a minute)
    for j in range(min(8, a.strong_problems)):
        gm, bvm, bfm, ef = cnfgen.random_batch(1, n, a.k, a.alpha, a.seed + 5000 + j)
        distinct.append([torch.from_numpy(np.ascontiguousarray(x)).pin_memory() for x in (gm, bvm, bfm, ef)])
    segs = []
    for j in range(a.strong_problems):
        t = distinct[j % len(distinct)]
        segs.append((t[0], t[1], t[2], t[3], None, torch.zeros(1, 1), [["s%d" % j]]))
    E = sum(int(sg[0].shape[1]) for sg in segs)

    def run():
        out = io.StringIO()
        t0 = time.perf_counter()
        trainer._predict_epoch(None, trainer._post_process_predictions, 1, out, segment_stream=iter(segs))
        for dev in trainer._devices:
            torch.cuda.synchronize(dev)
        return time.perf_counter() - t0, out.getvalue().count("\n")
    run()                      # warm-up: module loading, allocator, workspace sizes
    secs, lines = run()
    return {"workload": "%d problems of random %d-SAT n=%d m/n=%.2f (one per segment), p-d-p T=%d + %d WalkSAT iterations, through "
                        "FactorGraphTrainerBase._predict_epoch on %d GPU(s) of one process" % (a.strong_problems, a.k, n, a.alpha, a.iterations, a.walksat, world),
            "n_gpus": world, "seconds": secs, "cnfs_per_s": a.strong_problems / secs, "edge_updates_per_s": float(E) * a.iterations / secs,
            "output_lines": lines, "scaling": "strong", "timing": "host wall clock around the call, all devices synchronised"}


def config0_solved(dev):
    """The "CNFs solved/s" half of the metric on BASELINE.json configs[0] (the n = 1M problems of the main workload are
    never solved within T = 100): p-d-p on 5000 x random 3-SAT n = 100, m/n = 4.2, T = 1000, + 100 WalkSAT iterations,
    one whole forward() + CNF check, device-resident inputs, second of two runs."""
    import torch
    from pdp_solver_b200 import cnfgen
    from pdp_solver_b200.nn import solver as pdp_solver
    B, n, T, W = 5000, 100, 1000, 100
    gm, bvm, bfm, ef = [torch.from_numpy(x).to(dev) for x in cnfgen.random_batch(B, n, 3, 4.2, 1000)]
    model = pdp_solver.SurveyPropagatorSolver(dev, "p-d-p", tolerance=0.02, t_max=100, local_search_iterations=W, epsilon=0.5)

    def termination(active, prediction, sat_problem):
        raise RuntimeError("unreachable")
    termination._pdp_standard_termination = True
    out = None
    for rep in range(2):
        torch.manual_seed(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        init = model.get_init_state(gm, bvm, bfm, ef, None, randomized=False, batch_replication=1)
        (pred, _), _ = model(init_state=init, graph_map=gm, batch_variable_map=bvm, batch_function_map=bfm, edge_feature=ef,
                             meta_data=None, is_training=False, iteration_num=T, check_termination=termination, batch_replication=1)
        solved, _ = model.last_problem._ctx.cnf_eval(pred)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        k = int(solved.sum().item())
        out = {"workload": "p-d-p SP + %d-iteration WalkSAT, random 3-SAT n=%d m/n=4.20, batch %d, T=%d (BASELINE.json configs[0])" % (W, n, B, T),
               "cnfs_solved": k, "cnfs": B, "ms": ms, "cnfs_solved_per_s": k / (ms / 1e3), "cnfs_per_s": B / (ms / 1e3),
               "iterations": int(model.last_iterations.item())}
    return out


# --------------------------------------------------------------------------------------------------
# the other configurations of BASELINE.json as driver-parsable lines: `--workload config0|config1|config2|config4`
# --------------------------------------------------------------------------------------------------
def other_workload(a):
    """(name, model type, per-rank batch builder, T, W, replication list, metric, unit)"""
    from pdp_solver_b200 import cnfgen
    w = a.workload
    if w == "config0":
        return dict(name="p-d-p SP + 100-iteration WalkSAT, random 3-SAT n=100 m/n=4.20, batch 5000 per GPU, T=1000 (BASELINE.json configs[0])",
                    model="p-d-p", batch=lambda seed: cnfgen.random_batch(5000, 100, 3, 4.2, seed), T=1000, W=100, reps=[1],
                    metric="cnfs_solved_per_s", unit="CNFs/s", cpu=dict(B=20, n=100, k=3, alpha=4.2, T=1000, W=100))
    if w == "config1":
        return dict(name="p-nd-np (SP with neural decimator and predictor, random-init weights) random 3-SAT n=10000 m/n=4.20, 8 problems per GPU, T=20 (BASELINE.json configs[1])",
                    model="p-nd-np", batch=lambda seed: cnfgen.random_batch(8, 10000, 3, 4.2, seed), T=20, W=100, reps=[1],
                    metric="edge_updates_per_s", unit="edge-updates/s", cpu=dict(B=1, n=2000, k=3, alpha=4.2, T=3, W=2))
    if w == "config2":
        return dict(name="np-nd-np (fully neural PDP, random-init weights) random 4-SAT n=1000 m/n=9.00, 32 problems per GPU, T=20 (BASELINE.json configs[2])",
                    model="np-nd-np", batch=lambda seed: cnfgen.random_batch(32, 1000, 4, 9.0, seed), T=20, W=100, reps=[1],
                    metric="edge_updates_per_s", unit="edge-updates/s", cpu=dict(B=2, n=1000, k=4, alpha=9.0, T=3, W=2))

    def mixed(seed):      # mixed random 3-/5-SAT, n = 500 ... 50 000
        specs = [(500, 3, 4.0), (500, 5, 18.0), (5000, 3, 4.0), (5000, 5, 18.0), (50000, 3, 4.0), (50000, 5, 18.0)]
        return cnfgen.mixed_batch([sp for sp in specs for _ in range(2)], seed)
    return dict(name="p-d-p SP + 100-iteration WalkSAT with batch replication -b 1..64, mixed random 3-SAT (m/n=4.0) / 5-SAT (m/n=18) n=500..50000, 12 problems per GPU, T=600 (BASELINE.json configs[4])",
                model="p-d-p", batch=mixed, T=600, W=100, reps=[1, 8, 64], metric="edge_updates_per_s", unit="edge-updates/s",
                cpu=dict(B=2, n=500, k=3, alpha=4.2, T=50, W=10))


def build_b200_model(model_type, dev, W, a):
    import torch
    from pdp_solver_b200.nn import solver as S, util as U
    if model_type == "p-d-p":
        return S.SurveyPropagatorSolver(dev, "p-d-p", tolerance=a.tolerance, t_max=a.t_max, local_search_iterations=W, epsilon=a.epsilon)
    H, MH, AH, MAH, CH = 150, 100, 100, 50, 50
    torch.manual_seed(1)
    clf = U.Perceptron(H, CH, 1)
    if model_type == "p-nd-np":
        m = S.NeuralSurveyPropagatorSolver(dev, "m", 1, 0, H, MH, AH, MAH, 1, variable_classifier=clf, local_search_iterations=W, epsilon=a.epsilon)
    else:
        m = S.NeuralPropagatorDecimatorSolver(dev, "m", 1, 0, H, H, MH, AH, MAH, 1, variable_classifier=clf, local_search_iterations=W, epsilon=a.epsilon)
    return m.to(dev).eval()


def run_other_workload(a, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    spec = other_workload(a)
    if a.impl == "reference":
        if rank == 0:
            print(json.dumps(other_reference_line(a, spec, a.steps, min(a.warmup, 1))))
        return
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    batch = spec["batch"](a.seed + 17 * rank)
    host = [torch.from_numpy(np.ascontiguousarray(x)).pin_memory() for x in batch]
    E, V, B = batch[0].shape[1], batch[1].shape[0], int(batch[1].max()) + 1
    resident = [t.to(dev) for t in host]
    model = build_b200_model(spec["model"], dev, spec["W"], a)

    def termination(active, prediction, sat_problem):
        raise RuntimeError("unreachable")
    termination._pdp_standard_termination = True

    def forward(tensors, rep):
        gm, bvm, bfm, ef = tensors
        with torch.no_grad():
            init = model.get_init_state(gm, bvm, bfm, ef, None, randomized=False, batch_replication=rep)
            (pred, _), _ = model(init_state=init, graph_map=gm, batch_variable_map=bvm, batch_function_map=bfm, edge_feature=ef,
                                 meta_data=None, is_training=False, iteration_num=spec["T"], check_termination=termination,
                                 batch_replication=rep)
        from pdp_solver_b200.nn.util import cnf_eval_edges
        solved, n_unsat = cnf_eval_edges(pred, gm, bvm, bfm, ef, batch_size=B)
        return pred, solved, n_unsat

    outputs = {}

    def measure(rep, from_host):
        tot = {"solved": 0.0, "updates": 0.0}

        def step(timed):
            torch.manual_seed(1 + rank)
            tens = [t.to(dev, non_blocking=True) for t in host] if from_host else resident
            pred, solved, n_unsat = forward(tens, rep)
            if from_host:
                pred.cpu(); solved.cpu()
            if timed:
                tot["solved"] += float((solved > 0.5).sum().item())
                tot["updates"] += float(E) * rep * float(model.last_iterations.reshape(-1)[0].item())
            return {"prediction": pred, "solved": solved, "unsat_clauses": n_unsat}
        for _ in range(a.warmup):
            step(False)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.steps):
            last = step(True)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if a.dump_outputs and not from_host and rep == spec["reps"][0] and rank == 0:
            outputs.update({k: v.reshape(-1).cpu().numpy() for k, v in last.items()})
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            g = torch.tensor([tot["solved"], tot["updates"]], device=dev, dtype=torch.float64)
            dist.all_reduce(g, op=dist.ReduceOp.SUM)
            tot["solved"], tot["updates"] = [float(x) for x in g.tolist()]
        units = tot["solved"] if spec["metric"] == "cnfs_solved_per_s" else tot["updates"]
        return ms, units, tot

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    sweep = []
    for rep in spec["reps"]:
        ms, units, tot = measure(rep, False)
        ms_e, units_e, _ = measure(rep, True)
        sweep.append({"batch_replication": rep, "value": units / (ms / 1e3), "ms_per_step": ms / a.steps, "e2e_value": units_e / (ms_e / 1e3),
                      "e2e_ms_per_step": ms_e / a.steps, "cnfs_solved_per_step": tot["solved"] / a.steps,
                      "cnfs_per_s": world * B * a.steps / (ms / 1e3), "edge_updates_per_s": tot["updates"] / (ms / 1e3)})
    sampler.stop_flag = True
    if outputs:
        dump_outputs(a.dump_outputs, outputs)
    if rank == 0:
        head = sweep[0]
        h2d = sum(int(t.numel() * t.element_size()) for t in host)
        line = {"metric": spec["metric"], "value": head["value"], "unit": spec["unit"], "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if spec["model"] == "p-d-p" else "f32 (dense layers: tf32 x 3 split on tcgen05)", "data": "synthetic",
                "config": {"workload": spec["name"], "model_type": spec["model"], "edges_per_gpu": E, "variables_per_gpu": V, "problems_per_gpu": B,
                           "T": spec["T"], "walksat_iterations": spec["W"], "init": "deterministic (predict path)",
                           "l2": "flushed by the step itself: every step re-ingests its batch and rewrites its message arrays" if E * 48 < 126e6
                           else "inputs larger than L2", "sharding": "problems sharded across ranks, no per-iteration collective"},
                "e2e": {"value": head["e2e_value"], "unit": spec["unit"], "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": (V * 4 + B * 4) * world,
                        "ms_per_step": head["e2e_ms_per_step"]},
                "gpu_launches": int(model.last_problem._ctx.launch_count()) * a.steps, "replication_sweep": sweep if len(sweep) > 1 else None,
                "edge_updates_per_s": head["edge_updates_per_s"], "cnfs_per_s": head["cnfs_per_s"], "roofline": None, "clocks": sampler.summary()}
        if not a.no_cpu_baseline:
            line["cpu_baseline"] = other_reference_line(a, spec)["cpu_baseline"]
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def other_reference_line(a, spec, steps=1, warmup=0):
    """the reference's CPU path on a bounded sample of the workload (same model type, fewer / smaller problems, fewer iterations),
    `steps` timed forwards after `warmup` untimed ones.  Without the reference tree the C oracle port stands in for p-d-p, as
    in run_reference_arm; the neural model types have no port."""
    import torch
    from oracle import ref_timing
    from pdp_solver_b200 import cnfgen
    c = spec["cpu"]
    if ref_timing.available():
        kind, what = "reference", "the unmodified reference with use_cuda=False"
        cores = ref_timing.pin_threads()
        model = ref_timing.build_model(spec["model"], torch.device("cpu"), c["W"], a.epsilon, a.tolerance, a.t_max)
    elif spec["model"] == "p-d-p":
        from oracle import pdp_oracle as po
        kind, what = "port", "the C oracle port"
        po.build()
        po.set_num_threads(os.cpu_count() or 1)
        cores = po.num_threads()
    else:
        cb = {"unavailable": "reference tree absent (baseline/_ref)"}
        return {"impl": "reference", "metric": spec["metric"], "unit": spec["unit"], "cpu_baseline": cb}
    batch = cnfgen.random_batch(c["B"], c["n"], c["k"], c["alpha"], a.seed + 999)

    def forward():
        if kind == "reference":
            return ref_timing.timed_forward(model, batch, c["T"], torch.device("cpu"), seed=a.seed)
        return port_forward(batch, c["T"], c["W"], a.tolerance, a.t_max, a.epsilon, a.seed)
    for _ in range(warmup):
        forward()
    runs = [forward() for _ in range(steps)]
    r = {k: sum(x[k] for x in runs) for k in ("total_s", "loop_s", "setup_s", "iterations", "solved")}
    r["edges"] = runs[0]["edges"]
    if spec["metric"] == "cnfs_solved_per_s":
        value = r["solved"] / r["total_s"]
    else:
        value = r["edges"] * max(r["iterations"], 1) / r["total_s"]
    cb = {"value": value, "unit": spec["unit"], "cores": cores, "kind": kind,
          "sample": "%d problems of random %d-SAT n=%d m/n=%.2f, T=%d, %d WalkSAT iterations: %d forward(s) of %s, %.2f s (%d iterations executed, %d solved)"
                    % (c["B"], c["k"], c["n"], c["alpha"], c["T"], c["W"], steps, what, r["total_s"], r["iterations"], r["solved"]),
          "s_per_iteration": r["loop_s"] / max(r["iterations"], 1), "setup_s": r["setup_s"] / steps,
          "cnfs_per_s": c["B"] * steps / r["total_s"], "edge_updates_per_s": r["edges"] * max(r["iterations"], 1) / r["total_s"]}
    return {"impl": "reference", "metric": spec["metric"], "value": value, "unit": spec["unit"], "n_gpus": a.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": 1e3 * r["total_s"] / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": spec["name"], "model_type": spec["model"]}, "cpu_baseline": cb,
            "e2e": {"value": value, "unit": spec["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.workload != "config3":
        if world == 1 and a.gpus > 1 and a.impl != "reference":
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(a.gpus),
                   "--master-addr", "127.0.0.1", "--master-port", "29531"] + sys.argv
            sys.exit(subprocess.call(cmd))
        run_other_workload(a, rank, world, local_rank)
        return
    if a.impl == "reference":
        run_reference_arm(a, rank, world)
        return
    if world == 1 and a.gpus > 1:
        # launched without torchrun: re-launch one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(a.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29531"] + sys.argv
        sys.exit(subprocess.call(cmd))
    run_b200_arm(a, rank, world, local_rank)


if __name__ == "__main__":
    main()
