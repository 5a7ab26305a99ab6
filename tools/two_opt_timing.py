#!/usr/bin/env python
"""Timing of the 2-opt kernel (elg_two_opt) with CUDA events, one GPU call for every case:

  1. TSP100 / CVRP100: the best POMO row of each of 8000 aug-instances (1000 instances x 8), scaled metric;
  2. all 49 TSPLIB and 51 Set-X instances of tests/golden/lib, the drivers' greedy tours, rounded unscaled metric;
  3. synthetic TSP with N = 1000, 4000, 7000 (one instance x 8 augmentations), scaled metric, max_iterations 1000.

Tours come from greedy rollouts of the seeded synthetic checkpoint.  Every case is launched once to warm up, then timed
(the kernel is deterministic, so both launches do the same work).  Per case: ms per call, moves applied, us per move
(call time / largest per-tour move count: tours run side by side), pair evaluations per second (pairs the kernel swept,
counted on the host), cost or gap before and after.

    python tools/two_opt_timing.py [--out profiles/r03_two_opt] [--quick]"""
import argparse
import ctypes as C
import json
import os
import random
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
LIB = os.path.join(ROOT, "tests", "golden", "lib")
DEV = "cuda:0"


def pairs_swept(problem, row, n1, moves, max_iterations):
    """Pairs the kernel evaluates over the whole search of one tour (searches = moves + 1 unless the cap stopped it)."""
    n = len(row) if problem == "cvrp" else n1
    if problem == "cvrp":
        last = np.maximum.accumulate(np.where(row == 0, np.arange(n), -1))
        dmax = min(int((np.arange(n) - last).max()), n - 1)
    else:
        dmax = n - 1
    per = sum(n - d for d in range(2, dmax + 1))
    return per * (moves + (0 if moves >= max_iterations else 1))


def timed(problem, xy, rows, max_iterations, rounding):
    """-> (ms of the timed launch, tours, length, iterations)"""
    from elg_b200 import engine
    from elg_b200._lib import ELG_CVRP, ELG_TSP, check, lib
    engine.two_opt(problem, xy, rows, max_iterations=max_iterations, rounding=rounding)       # warm-up, argument checks
    R, L = rows.shape
    xy = xy.contiguous().float()
    t16 = rows.to(torch.int16).contiguous()
    length = torch.empty(R, dtype=torch.float32, device=DEV)
    iters = torch.empty(R, dtype=torch.int32, device=DEV)
    stream = torch.cuda.current_stream()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record(stream)
    check(lib.elg_two_opt(ELG_CVRP if problem == "cvrp" else ELG_TSP, C.c_void_p(xy.data_ptr()), int(xy.shape[0]),
                          int(xy.shape[1]), C.c_void_p(0), C.c_void_p(t16.data_ptr()), R, L, int(rounding), max_iterations,
                          C.c_void_p(iters.data_ptr()), C.c_void_p(length.data_ptr()), C.c_void_p(stream.cuda_stream)))
    ev1.record(stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1), t16.long(), length, iters


def summarize(case, problem, xy, rows, max_iterations, rounding, before, opt=None, n_aug=8):
    from elg_b200 import engine
    ms, out, length, iters = timed(problem, xy, rows, max_iterations, rounding)
    it = iters.cpu().numpy()
    r_np = rows.cpu().numpy()
    pairs = sum(pairs_swept(problem, r_np[r], int(xy.shape[1]), int(it[r]), max_iterations) for r in range(len(it)))
    inst_before = before.reshape(n_aug, -1).min(0)[0].cpu().numpy()
    inst_after = length.reshape(n_aug, -1).min(0)[0].cpu().numpy()
    row = dict(case=case, tours=len(it), N1=int(xy.shape[1]), L=int(rows.shape[1]), ms=ms, moves=int(it.sum()),
               max_moves=int(it.max()), capped=int((it >= max_iterations).sum()),
               us_per_move=1000 * ms / max(int(it.max()), 1), pair_evals_per_s=pairs / (ms / 1000),
               cost_before=float(inst_before.mean()), cost_after=float(inst_after.mean()))
    if opt is not None:
        row["gap_before"] = float(((inst_before - opt) / opt).mean())
        row["gap_after"] = float(((inst_after - opt) / opt).mean())
    assert torch.equal(length, engine.tour_length(xy, out[:, None], rounding=rounding)[:, 0])
    return row


def random_case(problem, N, n, M, seed):
    from elg_b200 import engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict, synthetic_tsp_batch
    if problem == "cvrp":
        b = synthetic_cvrp_batch(n, N, seed=seed)
        xy, dem = engine.load_problems("cvrp", b["loc"].to(DEV), b["depot"].to(DEV), b["demand"].to(DEV), aug=8)
    else:
        xy, dem = engine.load_problems("tsp", synthetic_tsp_batch(n, N, seed=seed).to(DEV), aug=8)
    h = engine.ModelHandle(problem, DEFAULT_MODEL_PARAMS[problem], synthetic_state_dict(problem, seed=1234, gain=3.0), DEV)
    batch = engine.encode(h, xy, dem)
    start = random.Random(seed).sample(range(N), M)
    tours16, reward, _, n_steps = engine.rollout(batch, M, start)
    T = int(n_steps.max()) if problem == "cvrp" else N
    best = reward.argmax(1)
    rows = tours16[torch.arange(xy.shape[0], device=DEV), best, :T].long()
    return xy, rows, -reward.max(1)[0]


def library_case(kind):
    """Every instance of the set through its driver (greedy, x8, rounded unscaled metric) -> list of summaries."""
    import library_parity as lp
    from elg_b200 import engine
    problem = "tsp" if kind == "tsplib" else "cvrp"
    with open(os.path.join(LIB, kind + "_ref.json")) as f:
        ref = json.load(f)
    z = np.load(os.path.join(LIB, kind + "_inputs.npz"))
    model = lp._model(problem, ref)
    cfg = lp._config(problem)
    if problem == "cvrp":
        from elg_b200.cvrp.test_vrplib import VRPLib_Tester
        tester = VRPLib_Tester(cfg, model=model)
    else:
        from elg_b200.tsp.test_tsplib import TSPLib_Tester
        tester = TSPLib_Tester(cfg, model=model)
    rows_out = []
    for r in ref["instances"]:
        name = r["instance"]
        random.seed(ref["seed"])
        res = {}
        if problem == "cvrp":
            cap, opt = z[name + "/capopt"]
            inst = {"node_coord": z[name + "/coord"].astype(np.float64), "demand": z[name + "/demand"].astype(np.float64),
                    "capacity": float(cap), "depot": np.array([0])}
            sols, rewards = tester.test_on_one_ins(name=name, result_dict=res, instance=inst, solution=float(opt))
            c = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None].to(DEV)
            xy = engine.load_problems("cvrp", c[:, 1:], c[:, 0], torch.zeros(1, c.shape[1] - 1, device=DEV), aug=8)[0]
        else:
            opt = float(z[name + "/opt"])
            sols, rewards = tester.test_on_one_ins(name, res, [z[name + "/coord"], opt])
            xy = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None].to(DEV)
        B = rewards.shape[0]
        rows = sols[torch.arange(B, device=DEV), rewards.argmax(1)]
        rows_out.append(summarize(name, problem, xy, rows, 1000, True, -rewards.max(1)[0], opt=float(opt)))
        print(json.dumps(rows_out[-1]), flush=True)
    return rows_out


def markdown(device, power, cases, lib):
    out = ["# 2-opt local search on the GPU (`elg_two_opt`)", "",
           "Measured on %s, power limit %s, with `tools/two_opt_timing.py` (CUDA events around one launch after a warm-up "
           "launch of the same work).  Tours are the greedy rollouts of the seeded synthetic checkpoint (gain 3), best POMO "
           "row of every aug-instance, so they are far from 2-opt-optimal.  `us/move` is the call time over the largest "
           "per-tour move count (tours are refined side by side).  Pair evaluations count the pairs the kernel sweeps "
           "(cvrp: the diagonals up to the longest route); cost is the best over the 8 augmentations, averaged over "
           "instances." % (device, power), "",
           "| case | tours | N1 | L | max_iterations | ms / call | moves (sum) | max moves / tour | tours at the cap | us / move | pair evals / s | cost before | cost after |",
           "|---|---|---|---|---|---|---|---|---|---|---|---|---|"]
    for c in cases:
        out.append("| %s | %d | %d | %d | %d | %.2f | %d | %d | %d | %.1f | %.3g | %.4f | %.4f |" % (
            c["case"], c["tours"], c["N1"], c["L"], c["max_iterations"], c["ms"], c["moves"], c["max_moves"], c["capped"],
            c["us_per_move"], c["pair_evals_per_s"], c["cost_before"], c["cost_after"]))
    for kind, rows in lib.items():
        if not rows:
            continue
        tot = sum(r["ms"] for r in rows)
        out += ["", "## %s: %d instances, rounded unscaled metric, max_iterations 1000" % (kind, len(rows)), "",
                "Total kernel time %.1f ms; moves %d; mean gap %.2f %% before, %.2f %% after." % (
                    tot, sum(r["moves"] for r in rows), 100 * np.mean([r["gap_before"] for r in rows]),
                    100 * np.mean([r["gap_after"] for r in rows])), "",
                "| instance | N1 | L | ms | moves (8 tours) | max moves | us / move | pair evals / s | gap before | gap after |",
                "|---|---|---|---|---|---|---|---|---|---|"]
        for r in rows:
            out.append("| %s | %d | %d | %.2f | %d | %d | %.1f | %.3g | %.2f %% | %.2f %% |" % (
                r["case"], r["N1"], r["L"], r["ms"], r["moves"], r["max_moves"], r["us_per_move"], r["pair_evals_per_s"],
                100 * r["gap_before"], 100 * r["gap_after"]))
    return "\n".join(out) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_two_opt"))
    ap.add_argument("--quick", action="store_true", help="small sizes only (rehearsal)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    device = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip() or "not reported"
    except OSError:
        power = "not reported"
    cases = []
    plan = ([("tsp", 100, 1000, 100, 1000), ("cvrp", 100, 1000, 100, 1000)] if not args.quick else
            [("tsp", 100, 16, 100, 1000), ("cvrp", 100, 16, 100, 1000)])
    plan += [("tsp", N, 1, 128, 1000) for N in ((1000, 4000, 7000) if not args.quick else (1000,))]
    for problem, N, n, M, cap in plan:
        xy, rows, before = random_case(problem, N, n, M, seed=N)
        c = summarize("%s%d x %d" % (problem.upper(), N, 8 * n), problem, xy, rows, cap, False, before)
        c["max_iterations"] = cap
        cases.append(c)
        print(json.dumps(c), flush=True)
    lib = {} if args.quick else {k: library_case(k) for k in ("tsplib", "setx")}
    md = markdown(device, power, cases, lib)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out + ".md", "w") as f:
        f.write(md)
    with open(args.out + ".json", "w") as f:
        json.dump({"device": device, "power_limit": power, "cases": cases, "library": lib}, f, indent=1)
    print(md)


if __name__ == "__main__":
    main()
