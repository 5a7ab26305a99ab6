#!/usr/bin/env python
"""Timing of the capacity-aware CVRP local search (elg_cvrp_local_search) with CUDA events, one GPU call for every case:

  1. CVRP100: the best POMO row of each of 8000 aug-instances (1000 instances x 8), scaled metric;
  2. CVRP1000: one instance x 8 augmentations, scaled metric;
  3. all 51 Set-X instances of tests/golden/lib, the driver's greedy rows, rounded unscaled metric, with the gap after
     2-opt (elg_two_opt) on the same rows beside it.

Rows come from greedy rollouts of the seeded synthetic checkpoint; max_iterations is 1000 throughout.  Every case is
launched once with max_iterations 1 to warm up, then timed.  Per case: ms per call, moves applied, us per move (call time
over the largest per-row move count: rows run side by side), position pairs evaluated per second (P^2 pairs per search,
each pair covering up to four move types, with P the used positions of the output row: P only shrinks during a search,
so the count is a lower bound), cost or gap before and after.

    python tools/cvrp_ls_timing.py [--out profiles/r04_cvrp_local_search] [--quick]"""
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


def timed(xy, rows, dem, cap, rounding):
    """-> (ms of the timed launch, rows, length, iterations)"""
    from elg_b200 import engine
    from elg_b200._lib import check, lib
    engine.cvrp_local_search(xy, rows, dem, cap, max_iterations=1, rounding=rounding)     # warm-up, argument checks
    R, L = rows.shape
    xy = xy.contiguous().float()
    units = torch.round(dem.double() * cap).to(torch.int32).contiguous()
    t16 = rows.to(torch.int16).contiguous()
    length = torch.empty(R, dtype=torch.float32, device=DEV)
    iters = torch.empty(R, dtype=torch.int32, device=DEV)
    stream = torch.cuda.current_stream()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p = lambda t: C.c_void_p(t.data_ptr())
    torch.cuda.synchronize()
    ev0.record(stream)
    check(lib.elg_cvrp_local_search(p(xy), int(xy.shape[0]), int(xy.shape[1]), p(units), int(cap), C.c_void_p(0), p(t16),
                                    R, L, int(rounding), MAX_IT, p(iters), p(length), C.c_void_p(stream.cuda_stream)))
    ev1.record(stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1), t16.long(), length, iters


def summarize(case, xy, rows, dem, cap, rounding, before, opt=None, n_aug=8):
    from elg_b200 import engine
    ms, out, length, iters = timed(xy, rows, dem, cap, rounding)
    it = iters.cpu().numpy()
    pos = torch.arange(out.shape[1], device=out.device)
    P = (torch.where(out != 0, pos, 0).max(1)[0] + 1).cpu().numpy()      # used positions: up to the last customer
    pairs = sum(int(P[r]) ** 2 * (int(it[r]) + (0 if it[r] >= MAX_IT else 1)) for r in range(len(it)))
    routes = lambda t: ((t[:, :-1] == 0) & (t[:, 1:] != 0)).sum(1).float()
    inst_before = before.reshape(n_aug, -1).min(0)[0].cpu().numpy()
    inst_after = length.reshape(n_aug, -1).min(0)[0].cpu().numpy()
    row = dict(case=case, rows=len(it), N1=int(xy.shape[1]), L=int(rows.shape[1]), ms=ms, moves=int(it.sum()),
               max_moves=int(it.max()), capped=int((it >= MAX_IT).sum()),
               us_per_move=1000 * ms / max(int(it.max()), 1), pair_evals_per_s=pairs / (ms / 1000),
               routes_before=float(routes(rows).mean()), routes_after=float(routes(out).mean()),
               cost_before=float(inst_before.mean()), cost_after=float(inst_after.mean()))
    if opt is not None:
        row["gap_before"] = float(((inst_before - opt) / opt).mean())
        row["gap_after"] = float(((inst_after - opt) / opt).mean())
        two = engine.two_opt("cvrp", xy, rows, max_iterations=MAX_IT, rounding=rounding)[1]
        row["gap_after_2opt"] = float(((two.reshape(n_aug, -1).min(0)[0].cpu().numpy() - opt) / opt).mean())
    assert torch.equal(length, engine.tour_length(xy, out[:, None], rounding=rounding)[:, 0])
    return row


def random_case(N, n, cap, seed):
    from elg_b200 import engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict
    b = synthetic_cvrp_batch(n, N, seed=seed, capacity=float(cap))
    xy, dem = engine.load_problems("cvrp", b["loc"].to(DEV), b["depot"].to(DEV), b["demand"].to(DEV), aug=8)
    h = engine.ModelHandle("cvrp", DEFAULT_MODEL_PARAMS["cvrp"], synthetic_state_dict("cvrp", seed=1234, gain=3.0), DEV)
    start = random.Random(seed).sample(range(N), min(N, 100))
    tours16, reward, _, n_steps = engine.rollout(engine.encode(h, xy, dem), len(start), start)
    rows = tours16[torch.arange(xy.shape[0], device=DEV), reward.argmax(1), :int(n_steps.max())].long()
    return xy, dem, rows, -reward.max(1)[0]


def setx_case(names=None):
    """Every Set-X instance through its driver (greedy, x8, rounded unscaled metric) -> list of summaries."""
    import library_parity as lp
    from elg_b200 import engine
    from elg_b200.cvrp.test_vrplib import VRPLib_Tester
    with open(os.path.join(LIB, "setx_ref.json")) as f:
        ref = json.load(f)
    z = np.load(os.path.join(LIB, "setx_inputs.npz"))
    tester = VRPLib_Tester(lp._config("cvrp"), model=lp._model("cvrp", ref))
    out = []
    for r in ref["instances"]:
        name = r["instance"]
        if names and name not in names:
            continue
        random.seed(ref["seed"])
        cap, opt = z[name + "/capopt"]
        inst = {"node_coord": z[name + "/coord"].astype(np.float64), "demand": z[name + "/demand"].astype(np.float64),
                "capacity": float(cap), "depot": np.array([0])}
        sols, rewards = tester.test_on_one_ins(name=name, result_dict={}, instance=inst, solution=float(opt))
        c = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None].to(DEV)
        d = torch.tensor(z[name + "/demand"], dtype=torch.float32)[None].to(DEV) / float(cap)
        xy, dem = engine.load_problems("cvrp", c[:, 1:], c[:, 0], d[:, 1:], aug=8)
        rows = sols[torch.arange(8, device=DEV), rewards.argmax(1)]
        out.append(summarize(name, xy, rows, dem, int(cap), True, -rewards.max(1)[0], opt=float(opt)))
        print(json.dumps(out[-1]), flush=True)
    return out


def markdown(device, power, cases, setx):
    out = ["# Capacity-aware CVRP local search on the GPU (`elg_cvrp_local_search`)", "",
           "Measured on %s, power limit %s, with `tools/cvrp_ls_timing.py` (CUDA events around one launch after a "
           "one-move warm-up launch).  Rows are the greedy rollouts of the seeded synthetic checkpoint (gain 3), best POMO "
           "row of every aug-instance.  max_iterations is %d.  `us/move` is the call time over the largest per-row move "
           "count (rows are refined side by side, one CTA each).  Pair evaluations count P^2 position pairs per search "
           "(each pair covers up to four move types) with P the used positions of the output row, a lower bound.  Cost is "
           "the best over the 8 augmentations, averaged over instances; routes are averaged over rows." % (
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
    return "\n".join(out) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_cvrp_local_search"))
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
    plan = [(100, 16, 50), (1000, 1, 250)] if args.quick else [(100, 1000, 50), (1000, 1, 250)]
    cases = []
    for N, n, cap in plan:
        xy, dem, rows, before = random_case(N, n, cap, seed=N)
        cases.append(summarize("CVRP%d x %d" % (N, 8 * n), xy, rows, dem, cap, False, before))
        print(json.dumps(cases[-1]), flush=True)
    setx = setx_case(["X-n101-k25", "X-n200-k36"] if args.quick else None)
    md = markdown(device, power, cases, setx)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out + ".md", "w") as f:
        f.write(md)
    with open(args.out + ".json", "w") as f:
        json.dump({"device": device, "power_limit": power, "cases": cases, "setx": setx}, f, indent=1)
    print(md)


if __name__ == "__main__":
    main()
