#!/usr/bin/env python
"""Timing of the GPU local searches with CUDA events, one GPU call per search.  Every case is one launch through the C
ABI between two events, after a warm-up call of the same search (2-opt: the same work; the other two: one move).

  --search two_opt  (elg_two_opt -> profiles/r03_two_opt):
      TSP100 / CVRP100, the best POMO row of each of 8000 aug-instances (1000 instances x 8), scaled metric; synthetic
      TSP with N = 1000, 4000, 7000 (one instance x 8 augmentations), scaled metric; all 49 TSPLIB and 51 Set-X
      instances of tests/golden/lib, the drivers' greedy tours, rounded unscaled metric.
  --search cvrp_ls  (elg_cvrp_local_search_ex, --max-segment 1 -> profiles/r04_cvrp_local_search):
      CVRP100 x 8000 and CVRP1000 x 8 rows, scaled metric; all 51 Set-X instances, rounded unscaled metric, with the gap
      after 2-opt on the same rows beside it.  With --max-segment 2 or 3 (Or-opt chains of up to that many customers ->
      profiles/r07_cvrp_or_opt) the same cases, each also run with max_segment 1 on the same rows.
  --search tsp_ls   (elg_tsp_local_search, max_segment 3, with elg_two_opt timed on the same tours beside it
                     -> profiles/r05_tsp_local_search):
      TSP100 x 8000, TSP1000 x 8 and TSP4000 x 8 tours, scaled metric; all 49 TSPLIB instances, rounded unscaled metric.

Tours come from greedy rollouts of the seeded synthetic checkpoint; max_iterations is 1000.  Per case: ms per call,
moves applied, us per move (call time over the largest per-tour move count: tours run side by side, one CTA each),
pair evaluations per second (pairs the kernel sweeps, counted on the host; see each markdown header), cost or gap
before and after.  --quick runs small sizes only (a rehearsal).

    python tools/local_search_timing.py --search {two_opt,cvrp_ls,tsp_ls} [--max-segment {1,2,3}] [--quick] [--out PREFIX]"""
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
MAX_IT = 1000
MAX_SEGMENT = 3
OUT = {"two_opt": "r03_two_opt", "cvrp_ls": "r04_cvrp_local_search", "tsp_ls": "r05_tsp_local_search"}


def timed(kernel, xy, rows, max_iterations, rounding, warmup_iterations, dem=None, cap=None, max_segment=1):
    """kernel 'tsp' / 'cvrp' (elg_two_opt), 'tsp_ls' or 'cvrp_ls' (max_segment) -> (ms of the timed launch, tours,
    length, iterations)"""
    from elg_b200 import engine
    from elg_b200._lib import ELG_CVRP, ELG_TSP, check, lib
    if kernel == "tsp_ls":                              # warm-up, argument checks
        engine.tsp_local_search(xy, rows, max_iterations=warmup_iterations, max_segment=MAX_SEGMENT, rounding=rounding)
    elif kernel == "cvrp_ls":
        engine.cvrp_local_search(xy, rows, dem, cap, max_iterations=warmup_iterations, rounding=rounding,
                                 max_segment=max_segment)
    else:
        engine.two_opt(kernel, xy, rows, max_iterations=warmup_iterations, rounding=rounding)
    R, L = rows.shape
    xy = xy.contiguous().float()
    t16 = rows.to(torch.int16).contiguous()
    length = torch.empty(R, dtype=torch.float32, device=DEV)
    iters = torch.empty(R, dtype=torch.int32, device=DEV)
    stream = torch.cuda.current_stream()
    p = lambda t: C.c_void_p(t.data_ptr())
    B, N1, s, null = int(xy.shape[0]), int(xy.shape[1]), C.c_void_p(stream.cuda_stream), C.c_void_p(0)
    if kernel == "cvrp_ls":
        units = torch.round(dem.double() * cap).to(torch.int32).contiguous()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record(stream)
    if kernel == "tsp_ls":
        check(lib.elg_tsp_local_search(p(xy), B, N1, null, p(t16), R, L, MAX_SEGMENT, int(rounding), max_iterations,
                                       p(iters), p(length), s))
    elif kernel == "cvrp_ls":
        check(lib.elg_cvrp_local_search_ex(p(xy), B, N1, p(units), int(cap), null, p(t16), R, L, max_segment,
                                           int(rounding), max_iterations, p(iters), p(length), s))
    else:
        check(lib.elg_two_opt(ELG_CVRP if kernel == "cvrp" else ELG_TSP, p(xy), B, N1, null, p(t16), R, L, int(rounding),
                              max_iterations, p(iters), p(length), s))
    ev1.record(stream)
    torch.cuda.synchronize()
    out = t16.long()
    assert torch.equal(length, engine.tour_length(xy, out[:, None], rounding=rounding)[:, 0])
    return ev0.elapsed_time(ev1), out, length, iters


def random_rows(problem, N, n, M, seed, capacity=None):
    """Greedy rollout of n random instances x 8 -> (xy, demand | None, best POMO row of every aug-instance, its cost)"""
    from elg_b200 import engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict, synthetic_tsp_batch
    if problem == "cvrp":
        b = synthetic_cvrp_batch(n, N, seed=seed, capacity=capacity)
        xy, dem = engine.load_problems("cvrp", b["loc"].to(DEV), b["depot"].to(DEV), b["demand"].to(DEV), aug=8)
    else:
        xy, dem = engine.load_problems("tsp", synthetic_tsp_batch(n, N, seed=seed).to(DEV), aug=8)
    h = engine.ModelHandle(problem, DEFAULT_MODEL_PARAMS[problem], synthetic_state_dict(problem, seed=1234, gain=3.0), DEV)
    start = random.Random(seed).sample(range(N), M)
    tours16, reward, _, n_steps = engine.rollout(engine.encode(h, xy, dem), M, start)
    T = int(n_steps.max()) if problem == "cvrp" else N
    rows = tours16[torch.arange(xy.shape[0], device=DEV), reward.argmax(1), :T].long()
    return xy, dem, rows, -reward.max(1)[0]


def library_rows(kind, names=None):
    """Every instance of the set ('tsplib' / 'setx', or those named) through its driver (greedy, x8, rounded unscaled
    metric) -> yields (name, xy, normalised demand | None, capacity | None, best rows, their cost, optimal cost)"""
    import library_parity as lp
    from elg_b200 import engine
    problem = "tsp" if kind == "tsplib" else "cvrp"
    with open(os.path.join(LIB, kind + "_ref.json")) as f:
        ref = json.load(f)
    z = np.load(os.path.join(LIB, kind + "_inputs.npz"))
    if problem == "cvrp":
        from elg_b200.cvrp.test_vrplib import VRPLib_Tester
        tester = VRPLib_Tester(lp._config(problem), model=lp._model(problem, ref))
    else:
        from elg_b200.tsp.test_tsplib import TSPLib_Tester
        tester = TSPLib_Tester(lp._config(problem), model=lp._model(problem, ref))
    for r in ref["instances"]:
        name = r["instance"]
        if names and name not in names:
            continue
        random.seed(ref["seed"])
        if problem == "cvrp":
            cap, opt = z[name + "/capopt"]
            inst = {"node_coord": z[name + "/coord"].astype(np.float64), "demand": z[name + "/demand"].astype(np.float64),
                    "capacity": float(cap), "depot": np.array([0])}
            sols, rewards = tester.test_on_one_ins(name=name, result_dict={}, instance=inst, solution=float(opt))
            c = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None].to(DEV)
            d = torch.tensor(z[name + "/demand"], dtype=torch.float32)[None].to(DEV) / float(cap)
            xy, dem = engine.load_problems("cvrp", c[:, 1:], c[:, 0], d[:, 1:], aug=8)
            cap = int(cap)
        else:
            opt = float(z[name + "/opt"])
            sols, rewards = tester.test_on_one_ins(name, {}, [z[name + "/coord"], opt])
            xy, dem, cap = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None].to(DEV), None, None
        rows = sols[torch.arange(rewards.shape[0], device=DEV), rewards.argmax(1)]
        yield name, xy, dem, cap, rows, -rewards.max(1)[0], float(opt)


def per_instance(cost, n_aug=8):
    """(aug*n,) costs -> (n,) best over the augmentations, on the host"""
    return cost.reshape(n_aug, -1).min(0)[0].cpu().numpy()


# ------------------------------------------------------------------------------------------------ two_opt


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


def two_opt_summary(case, problem, xy, rows, max_iterations, rounding, before, opt=None):
    ms, out, length, iters = timed(problem, xy, rows, max_iterations, rounding, max_iterations)
    it = iters.cpu().numpy()
    r_np = rows.cpu().numpy()
    pairs = sum(pairs_swept(problem, r_np[r], int(xy.shape[1]), int(it[r]), max_iterations) for r in range(len(it)))
    inst_before, inst_after = per_instance(before), per_instance(length)
    row = dict(case=case, tours=len(it), N1=int(xy.shape[1]), L=int(rows.shape[1]), ms=ms, moves=int(it.sum()),
               max_moves=int(it.max()), capped=int((it >= max_iterations).sum()),
               us_per_move=1000 * ms / max(int(it.max()), 1), pair_evals_per_s=pairs / (ms / 1000),
               cost_before=float(inst_before.mean()), cost_after=float(inst_after.mean()))
    if opt is not None:
        row["gap_before"] = float(((inst_before - opt) / opt).mean())
        row["gap_after"] = float(((inst_after - opt) / opt).mean())
    return row


def two_opt_run(quick):
    cases = []
    plan = ([("tsp", 100, 1000, 100, 1000), ("cvrp", 100, 1000, 100, 1000)] if not quick else
            [("tsp", 100, 16, 100, 1000), ("cvrp", 100, 16, 100, 1000)])
    plan += [("tsp", N, 1, 128, 1000) for N in ((1000, 4000, 7000) if not quick else (1000,))]
    for problem, N, n, M, cap in plan:
        xy, _, rows, before = random_rows(problem, N, n, M, seed=N)
        c = two_opt_summary("%s%d x %d" % (problem.upper(), N, 8 * n), problem, xy, rows, cap, False, before)
        c["max_iterations"] = cap
        cases.append(c)
        print(json.dumps(c), flush=True)
    lib = {}
    for kind in (() if quick else ("tsplib", "setx")):
        lib[kind] = []
        for name, xy, _, _, rows, before, opt in library_rows(kind):
            lib[kind].append(two_opt_summary(name, "tsp" if kind == "tsplib" else "cvrp", xy, rows, MAX_IT, True, before,
                                             opt=opt))
            print(json.dumps(lib[kind][-1]), flush=True)
    return {"cases": cases, "library": lib}


def two_opt_markdown(device, power, cases, library):
    out = ["# 2-opt local search on the GPU (`elg_two_opt`)", "",
           "Measured on %s, power limit %s, with `tools/local_search_timing.py --search two_opt` (CUDA events around one "
           "launch after a warm-up launch of the same work).  Tours are the greedy rollouts of the seeded synthetic "
           "checkpoint (gain 3), best POMO row of every aug-instance, so they are far from 2-opt-optimal.  `us/move` is the "
           "call time over the largest per-tour move count (tours are refined side by side).  Pair evaluations count the "
           "pairs the kernel sweeps (cvrp: the diagonals up to the longest route); cost is the best over the 8 "
           "augmentations, averaged over instances." % (device, power), "",
           "| case | tours | N1 | L | max_iterations | ms / call | moves (sum) | max moves / tour | tours at the cap | us / move | pair evals / s | cost before | cost after |",
           "|---|---|---|---|---|---|---|---|---|---|---|---|---|"]
    for c in cases:
        out.append("| %s | %d | %d | %d | %d | %.2f | %d | %d | %d | %.1f | %.3g | %.4f | %.4f |" % (
            c["case"], c["tours"], c["N1"], c["L"], c["max_iterations"], c["ms"], c["moves"], c["max_moves"], c["capped"],
            c["us_per_move"], c["pair_evals_per_s"], c["cost_before"], c["cost_after"]))
    for kind, rows in library.items():
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
    return out


# ------------------------------------------------------------------------------------------------ cvrp_ls


def cvrp_ls_summary(case, xy, rows, dem, cap, rounding, before, opt=None, max_segment=1):
    from elg_b200 import engine
    ms, out, length, iters = timed("cvrp_ls", xy, rows, MAX_IT, rounding, 1, dem, cap, max_segment)
    it = iters.cpu().numpy()
    pos = torch.arange(out.shape[1], device=out.device)
    P = (torch.where(out != 0, pos, 0).max(1)[0] + 1).cpu().numpy()      # used positions: up to the last customer
    pairs = sum(int(P[r]) ** 2 * (int(it[r]) + (0 if it[r] >= MAX_IT else 1)) for r in range(len(it)))
    routes = lambda t: ((t[:, :-1] == 0) & (t[:, 1:] != 0)).sum(1).float()
    inst_before, inst_after = per_instance(before), per_instance(length)
    row = dict(case=case, rows=len(it), N1=int(xy.shape[1]), L=int(rows.shape[1]), ms=ms, moves=int(it.sum()),
               max_moves=int(it.max()), capped=int((it >= MAX_IT).sum()),
               us_per_move=1000 * ms / max(int(it.max()), 1), pair_evals_per_s=pairs / (ms / 1000),
               routes_before=float(routes(rows).mean()), routes_after=float(routes(out).mean()),
               cost_before=float(inst_before.mean()), cost_after=float(inst_after.mean()))
    if opt is not None:
        row["gap_before"] = float(((inst_before - opt) / opt).mean())
        row["gap_after"] = float(((inst_after - opt) / opt).mean())
        if max_segment == 1:
            two = engine.two_opt("cvrp", xy, rows, max_iterations=MAX_IT, rounding=rounding)[1]
            row["gap_after_2opt"] = float(((per_instance(two) - opt) / opt).mean())
    if max_segment > 1:
        row["max_segment"] = max_segment
    return row


def cvrp_ls_run(quick, max_segment=1):
    """max_segment 1: the r04 cases.  Above 1: each case with max_segment and with 1 on the same rows, as a pair
    {"case", "or_opt": summary, "relocate": summary}."""
    def run(case, xy, rows, dem, cap, rounding, before, opt=None):
        if max_segment == 1:
            return cvrp_ls_summary(case, xy, rows, dem, cap, rounding, before, opt)
        return {"case": case, "or_opt": cvrp_ls_summary(case, xy, rows, dem, cap, rounding, before, opt, max_segment),
                "relocate": cvrp_ls_summary(case, xy, rows, dem, cap, rounding, before, opt, 1)}
    cases = []
    for N, n, cap in ([(100, 16, 50), (1000, 1, 250)] if quick else [(100, 1000, 50), (1000, 1, 250)]):
        xy, dem, rows, before = random_rows("cvrp", N, n, min(N, 100), seed=N, capacity=float(cap))
        cases.append(run("CVRP%d x %d" % (N, 8 * n), xy, rows, dem, cap, False, before))
        print(json.dumps(cases[-1]), flush=True)
    setx = []
    for name, xy, dem, cap, rows, before, opt in library_rows("setx", ["X-n101-k25", "X-n200-k36"] if quick else None):
        setx.append(run(name, xy, rows, dem, cap, True, before, opt=opt))
        print(json.dumps(setx[-1]), flush=True)
    return {"cases": cases, "setx": setx}


def cvrp_or_opt_markdown(device, power, cases, setx):
    seg = (cases or setx)[0]["or_opt"]["max_segment"]
    out = ["# Or-opt in the CVRP local search on the GPU (`elg_cvrp_local_search_ex`, max_segment %d)" % seg, "",
           "Measured on %s, power limit %s, with `tools/local_search_timing.py --search cvrp_ls --max-segment %d` (CUDA "
           "events around one launch after a one-move warm-up launch).  Rows are the greedy rollouts of the seeded "
           "synthetic checkpoint (gain 3), best POMO row of every aug-instance, the cases of `r04`.  Every case runs "
           "max_segment %d (Or-opt chains of up to %d customers) and max_segment 1 (relocate of one customer only, the "
           "search of `r04`) on the same rows.  max_iterations is %d.  `us/move` is the call time over the largest "
           "per-row move count.  Cost is the best over the 8 augmentations, averaged over instances; routes are averaged "
           "over rows." % (device, power, seg, seg, seg, MAX_IT), "",
           "| case | max_segment | rows | N1 | ms / call | moves (sum) | max moves / row | rows at the cap | us / move | routes before | routes after | cost before | cost after |",
           "|---|---|---|---|---|---|---|---|---|---|---|---|---|"]
    for pair in cases:
        for c, s in ((pair["relocate"], 1), (pair["or_opt"], seg)):
            out.append("| %s | %d | %d | %d | %.2f | %d | %d | %d | %.1f | %.1f | %.1f | %.4f | %.4f |" % (
                pair["case"], s, c["rows"], c["N1"], c["ms"], c["moves"], c["max_moves"], c["capped"], c["us_per_move"],
                c["routes_before"], c["routes_after"], c["cost_before"], c["cost_after"]))
    if setx:
        mean = lambda k, key: 100 * np.mean([r[k][key] for r in setx])
        above = [r["case"] for r in setx if r["or_opt"]["gap_after"] > r["relocate"]["gap_after"]]
        out += ["", "## Set-X: %d instances, rounded unscaled metric" % len(setx), "",
                "Total kernel time %.1f ms with max_segment %d (%d moves), %.1f ms with max_segment 1 (%d moves).  Mean gap "
                "%.2f %% before, %.2f %% after max_segment 1, %.2f %% after max_segment %d.  max_segment %d ends below "
                "max_segment 1 on %d instances, equal on %d, above on %d%s." % (
                    sum(r["or_opt"]["ms"] for r in setx), seg, sum(r["or_opt"]["moves"] for r in setx),
                    sum(r["relocate"]["ms"] for r in setx), sum(r["relocate"]["moves"] for r in setx),
                    mean("or_opt", "gap_before"), mean("relocate", "gap_after"), mean("or_opt", "gap_after"), seg, seg,
                    sum(r["or_opt"]["gap_after"] < r["relocate"]["gap_after"] for r in setx),
                    sum(r["or_opt"]["gap_after"] == r["relocate"]["gap_after"] for r in setx), len(above),
                    (" (%s)" % ", ".join(above)) if above else ""), "",
                "| instance | N1 | ms max_segment 1 | ms max_segment %d | moves 1 (8 rows) | moves %d | us / move 1 | us / move %d | routes after 1 | routes after %d | gap before | gap after 1 | gap after %d |" % (seg, seg, seg, seg, seg),
                "|---|---|---|---|---|---|---|---|---|---|---|---|---|"]
        for r in setx:
            a, b = r["relocate"], r["or_opt"]
            out.append("| %s | %d | %.2f | %.2f | %d | %d | %.1f | %.1f | %.1f | %.1f | %.2f %% | %.2f %% | %.2f %% |" % (
                r["case"], a["N1"], a["ms"], b["ms"], a["moves"], b["moves"], a["us_per_move"], b["us_per_move"],
                a["routes_after"], b["routes_after"], 100 * a["gap_before"], 100 * a["gap_after"], 100 * b["gap_after"]))
    return out


def cvrp_ls_markdown(device, power, cases, setx):
    out = ["# Capacity-aware CVRP local search on the GPU (`elg_cvrp_local_search`)", "",
           "Measured on %s, power limit %s, with `tools/local_search_timing.py --search cvrp_ls` (CUDA events around one "
           "launch after a one-move warm-up launch).  Rows are the greedy rollouts of the seeded synthetic checkpoint "
           "(gain 3), best POMO row of every aug-instance.  max_iterations is %d.  `us/move` is the call time over the "
           "largest per-row move count (rows are refined side by side, one CTA each).  Pair evaluations count P^2 position "
           "pairs per search (each pair covers up to four move types) with P the used positions of the output row, a lower "
           "bound.  Cost is the best over the 8 augmentations, averaged over instances; routes are averaged over rows." % (
               device, power, MAX_IT), "",
           "| case | rows | N1 | L | ms / call | moves (sum) | max moves / row | rows at the cap | us / move | pair evals / s | routes before | routes after | cost before | cost after |",
           "|---|---|---|---|---|---|---|---|---|---|---|---|---|---|"]
    for c in cases:
        out.append("| %s | %d | %d | %d | %.2f | %d | %d | %d | %.1f | %.3g | %.1f | %.1f | %.4f | %.4f |" % (
            c["case"], c["rows"], c["N1"], c["L"], c["ms"], c["moves"], c["max_moves"], c["capped"], c["us_per_move"],
            c["pair_evals_per_s"], c["routes_before"], c["routes_after"], c["cost_before"], c["cost_after"]))
    if setx:
        tot = sum(r["ms"] for r in setx)
        out += ["", "## Set-X: %d instances, rounded unscaled metric" % len(setx), "",
                "Total kernel time %.1f ms; moves %d; mean gap %.2f %% before, %.2f %% after the local search, %.2f %% after "
                "2-opt (elg_two_opt, max_iterations %d) on the same rows." % (
                    tot, sum(r["moves"] for r in setx), 100 * np.mean([r["gap_before"] for r in setx]),
                    100 * np.mean([r["gap_after"] for r in setx]), 100 * np.mean([r["gap_after_2opt"] for r in setx]),
                    MAX_IT), "",
                "| instance | N1 | L | ms | moves (8 rows) | max moves | rows at the cap | us / move | pair evals / s | routes before | routes after | gap before | gap after 2-opt | gap after local search |",
                "|---|---|---|---|---|---|---|---|---|---|---|---|---|---|"]
        for r in setx:
            out.append("| %s | %d | %d | %.2f | %d | %d | %d | %.1f | %.3g | %.1f | %.1f | %.2f %% | %.2f %% | %.2f %% |" % (
                r["case"], r["N1"], r["L"], r["ms"], r["moves"], r["max_moves"], r["capped"], r["us_per_move"],
                r["pair_evals_per_s"], r["routes_before"], r["routes_after"], 100 * r["gap_before"],
                100 * r["gap_after_2opt"], 100 * r["gap_after"]))
    return out


# ------------------------------------------------------------------------------------------------ tsp_ls


def tsp_ls_summary(case, xy, rows, rounding, before, opt=None):
    N1 = int(xy.shape[1])
    row = dict(case=case, tours=int(rows.shape[0]), N1=N1)
    inst_before = per_instance(before)
    row["cost_before"] = float(inst_before.mean())
    if opt is not None:
        row["gap_before"] = float(((inst_before - opt) / opt).mean())
    for kernel, per_search in (("2opt", (N1 - 1) * (N1 - 2) // 2), ("ls", N1 * N1)):
        ms, out, length, iters = timed("tsp_ls" if kernel == "ls" else "tsp", xy, rows, MAX_IT, rounding, 1)
        it = iters.cpu().numpy()
        searches = int(it.sum()) + int((it < MAX_IT).sum())
        inst_after = per_instance(length)
        row.update({kernel + "_ms": ms, kernel + "_moves": int(it.sum()), kernel + "_max_moves": int(it.max()),
                    kernel + "_capped": int((it >= MAX_IT).sum()), kernel + "_us_per_move": 1000 * ms / max(int(it.max()), 1),
                    kernel + "_pair_evals_per_s": searches * per_search / (ms / 1000),
                    kernel + "_cost_after": float(inst_after.mean())})
        if opt is not None:
            row[kernel + "_gap_after"] = float(((inst_after - opt) / opt).mean())
    return row


def tsp_ls_run(quick):
    cases = []
    for N, n, M in ([(100, 16, 100), (1000, 1, 128)] if quick else [(100, 1000, 100), (1000, 1, 128), (4000, 1, 128)]):
        xy, _, rows, before = random_rows("tsp", N, n, M, seed=N)
        cases.append(tsp_ls_summary("TSP%d x %d" % (N, 8 * n), xy, rows, False, before))
        print(json.dumps(cases[-1]), flush=True)
    lib = []
    for name, xy, _, _, rows, before, opt in library_rows("tsplib", ["eil51", "a280"] if quick else None):
        lib.append(tsp_ls_summary(name, xy, rows, True, before, opt=opt))
        print(json.dumps(lib[-1]), flush=True)
    return {"cases": cases, "tsplib": lib}


def tsp_ls_markdown(device, power, cases, lib):
    out = ["# TSP local search with 2-opt and Or-opt on the GPU (`elg_tsp_local_search`)", "",
           "Measured on %s, power limit %s, with `tools/local_search_timing.py --search tsp_ls` (CUDA events around one "
           "launch after a one-move warm-up launch).  Tours are the greedy rollouts of the seeded synthetic checkpoint "
           "(gain 3), best POMO row of every aug-instance.  max_iterations is %d, max_segment %d.  Each case runs the "
           "2-opt + Or-opt search (`ls`) and 2-opt alone (`elg_two_opt`, `2opt`) on the same tours.  `us/move` is the call "
           "time over the largest per-tour move count (tours are refined side by side, one CTA each).  Pair evaluations "
           "count the position pairs of every search: N1^2 for `ls` (each pair covers up to six variants), (N1-1)(N1-2)/2 "
           "for `2opt`.  Cost is the best over the 8 augmentations, averaged over instances." % (
               device, power, MAX_IT, MAX_SEGMENT), "",
           "| case | tours | N1 | kernel | ms / call | moves (sum) | max moves / tour | tours at the cap | us / move | pair evals / s | cost before | cost after |",
           "|---|---|---|---|---|---|---|---|---|---|---|---|"]
    for c in cases:
        for k, label in (("2opt", "2-opt"), ("ls", "2-opt + or-opt")):
            out.append("| %s | %d | %d | %s | %.2f | %d | %d | %d | %.1f | %.3g | %.4f | %.4f |" % (
                c["case"], c["tours"], c["N1"], label, c[k + "_ms"], c[k + "_moves"], c[k + "_max_moves"], c[k + "_capped"],
                c[k + "_us_per_move"], c[k + "_pair_evals_per_s"], c["cost_before"], c[k + "_cost_after"]))
    if lib:
        mean = lambda key: 100 * np.mean([r[key] for r in lib])
        out += ["", "## TSPLIB: %d instances, rounded unscaled metric" % len(lib), "",
                "Kernel time %.1f ms for 2-opt + Or-opt (%d moves), %.1f ms for 2-opt alone (%d moves).  Mean gap "
                "%.2f %% before, %.2f %% after 2-opt alone, %.2f %% after 2-opt + Or-opt; the search ends below 2-opt "
                "alone on %d instances, equal on %d, above on %d." % (
                    sum(r["ls_ms"] for r in lib), sum(r["ls_moves"] for r in lib), sum(r["2opt_ms"] for r in lib),
                    sum(r["2opt_moves"] for r in lib), mean("gap_before"), mean("2opt_gap_after"), mean("ls_gap_after"),
                    sum(r["ls_gap_after"] < r["2opt_gap_after"] for r in lib),
                    sum(r["ls_gap_after"] == r["2opt_gap_after"] for r in lib),
                    sum(r["ls_gap_after"] > r["2opt_gap_after"] for r in lib)), "",
                "| instance | N1 | ms 2-opt | ms 2-opt + or-opt | moves 2-opt (8 tours) | moves 2-opt + or-opt | us / move 2-opt | us / move 2-opt + or-opt | gap before | gap after 2-opt | gap after 2-opt + or-opt |",
                "|---|---|---|---|---|---|---|---|---|---|---|"]
        for r in lib:
            out.append("| %s | %d | %.2f | %.2f | %d | %d | %.1f | %.1f | %.2f %% | %.2f %% | %.2f %% |" % (
                r["case"], r["N1"], r["2opt_ms"], r["ls_ms"], r["2opt_moves"], r["ls_moves"], r["2opt_us_per_move"],
                r["ls_us_per_move"], 100 * r["gap_before"], 100 * r["2opt_gap_after"], 100 * r["ls_gap_after"]))
    return out


SEARCHES = {"two_opt": (two_opt_run, two_opt_markdown), "cvrp_ls": (cvrp_ls_run, cvrp_ls_markdown),
            "tsp_ls": (tsp_ls_run, tsp_ls_markdown)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--search", required=True, choices=sorted(SEARCHES))
    ap.add_argument("--out", help="output prefix for .md / .json (default: profiles/ r03 / r04 / r05 of the search)")
    ap.add_argument("--max-segment", type=int, choices=(1, 2, 3), default=1,
                    help="cvrp_ls: longest Or-opt chain; above 1 also runs 1 on the same rows (profiles/r07_cvrp_or_opt)")
    ap.add_argument("--quick", action="store_true", help="small sizes only (rehearsal)")
    args = ap.parse_args()
    if args.max_segment > 1 and args.search != "cvrp_ls":
        ap.error("--max-segment is an option of --search cvrp_ls")
    or_opt = args.max_segment > 1
    out_prefix = args.out or os.path.join(ROOT, "profiles", "r07_cvrp_or_opt" if or_opt else OUT[args.search])
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    device = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip() or "not reported"
    except OSError:
        power = "not reported"
    run, markdown = SEARCHES[args.search]
    if or_opt:
        result, markdown = cvrp_ls_run(args.quick, args.max_segment), cvrp_or_opt_markdown
    else:
        result = run(args.quick)
    md = "\n".join(markdown(device, power, *result.values())) + "\n"
    os.makedirs(os.path.dirname(os.path.abspath(out_prefix)), exist_ok=True)
    with open(out_prefix + ".md", "w") as f:
        f.write(md)
    with open(out_prefix + ".json", "w") as f:
        json.dump(dict(device=device, power_limit=power, **result), f, indent=1)
    print(md)


if __name__ == "__main__":
    main()
