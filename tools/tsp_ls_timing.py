#!/usr/bin/env python
"""Timing of the TSP local search with 2-opt and Or-opt moves (elg_tsp_local_search) with CUDA events, one GPU call for
every case, with 2-opt alone (elg_two_opt) timed on the same tours beside it:

  1. TSP100: the best POMO row of each of 8000 aug-instances (1000 instances x 8), scaled metric;
  2. TSP1000 and TSP4000: one instance x 8 augmentations, scaled metric;
  3. all 49 TSPLIB instances of tests/golden/lib, the driver's greedy tours, rounded unscaled metric.

Tours come from greedy rollouts of the seeded synthetic checkpoint; max_iterations is 1000 and max_segment 3 throughout.
Every kernel is launched once with max_iterations 1 to warm up, then timed.  Per case and kernel: ms per call, moves
applied, us per move (call time over the largest per-tour move count: tours run side by side), position pairs evaluated
per second (searches x the pairs one search sweeps: N1^2 for the local search, each pair covering up to six variants;
(N1-1)(N1-2)/2 for 2-opt), cost or gap before and after.

    python tools/tsp_ls_timing.py [--out profiles/r05_tsp_local_search] [--quick]"""
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


def timed(kernel, xy, rows, rounding):
    """kernel 'ls' (elg_tsp_local_search) or '2opt' (elg_two_opt) -> (ms of the timed launch, tours, length, iterations)"""
    from elg_b200 import engine
    from elg_b200._lib import ELG_TSP, check, lib
    if kernel == "ls":                                  # warm-up, argument checks
        engine.tsp_local_search(xy, rows, max_iterations=1, max_segment=MAX_SEGMENT, rounding=rounding)
    else:
        engine.two_opt("tsp", xy, rows, max_iterations=1, rounding=rounding)
    R, L = rows.shape
    xy = xy.contiguous().float()
    t16 = rows.to(torch.int16).contiguous()
    length = torch.empty(R, dtype=torch.float32, device=DEV)
    iters = torch.empty(R, dtype=torch.int32, device=DEV)
    stream = torch.cuda.current_stream()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p = lambda t: C.c_void_p(t.data_ptr())
    B, N1, s = int(xy.shape[0]), int(xy.shape[1]), C.c_void_p(stream.cuda_stream)
    torch.cuda.synchronize()
    ev0.record(stream)
    if kernel == "ls":
        check(lib.elg_tsp_local_search(p(xy), B, N1, C.c_void_p(0), p(t16), R, L, MAX_SEGMENT, int(rounding), MAX_IT,
                                       p(iters), p(length), s))
    else:
        check(lib.elg_two_opt(ELG_TSP, p(xy), B, N1, C.c_void_p(0), p(t16), R, L, int(rounding), MAX_IT, p(iters),
                              p(length), s))
    ev1.record(stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1), t16.long(), length, iters


def summarize(case, xy, rows, rounding, before, opt=None, n_aug=8):
    from elg_b200 import engine
    N1 = int(xy.shape[1])
    row = dict(case=case, tours=int(rows.shape[0]), N1=N1)
    inst_before = before.reshape(n_aug, -1).min(0)[0].cpu().numpy()
    row["cost_before"] = float(inst_before.mean())
    if opt is not None:
        row["gap_before"] = float(((inst_before - opt) / opt).mean())
    for kernel, per_search in (("2opt", (N1 - 1) * (N1 - 2) // 2), ("ls", N1 * N1)):
        ms, out, length, iters = timed(kernel, xy, rows, rounding)
        assert torch.equal(length, engine.tour_length(xy, out[:, None], rounding=rounding)[:, 0])
        it = iters.cpu().numpy()
        searches = int(it.sum()) + int((it < MAX_IT).sum())
        inst_after = length.reshape(n_aug, -1).min(0)[0].cpu().numpy()
        row.update({kernel + "_ms": ms, kernel + "_moves": int(it.sum()), kernel + "_max_moves": int(it.max()),
                    kernel + "_capped": int((it >= MAX_IT).sum()), kernel + "_us_per_move": 1000 * ms / max(int(it.max()), 1),
                    kernel + "_pair_evals_per_s": searches * per_search / (ms / 1000),
                    kernel + "_cost_after": float(inst_after.mean())})
        if opt is not None:
            row[kernel + "_gap_after"] = float(((inst_after - opt) / opt).mean())
    return row


def random_case(N, n, M, seed):
    from elg_b200 import engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict, synthetic_tsp_batch
    xy, _ = engine.load_problems("tsp", synthetic_tsp_batch(n, N, seed=seed).to(DEV), aug=8)
    h = engine.ModelHandle("tsp", DEFAULT_MODEL_PARAMS["tsp"], synthetic_state_dict("tsp", seed=1234, gain=3.0), DEV)
    start = random.Random(seed).sample(range(N), M)
    tours16, reward, _, _ = engine.rollout(engine.encode(h, xy), M, start)
    rows = tours16[torch.arange(xy.shape[0], device=DEV), reward.argmax(1), :N].long()
    return xy, rows, -reward.max(1)[0]


def tsplib_case(names=None):
    """Every TSPLIB instance through its driver (greedy, x8, rounded unscaled metric) -> list of summaries."""
    import library_parity as lp
    from elg_b200.tsp.test_tsplib import TSPLib_Tester
    with open(os.path.join(LIB, "tsplib_ref.json")) as f:
        ref = json.load(f)
    z = np.load(os.path.join(LIB, "tsplib_inputs.npz"))
    tester = TSPLib_Tester(lp._config("tsp"), model=lp._model("tsp", ref))
    out = []
    for r in ref["instances"]:
        name = r["instance"]
        if names and name not in names:
            continue
        random.seed(ref["seed"])
        opt = float(z[name + "/opt"])
        sols, rewards = tester.test_on_one_ins(name, {}, [z[name + "/coord"], opt])
        xy = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None].to(DEV)
        rows = sols[torch.arange(rewards.shape[0], device=DEV), rewards.argmax(1)]
        out.append(summarize(name, xy, rows, True, -rewards.max(1)[0], opt=opt))
        print(json.dumps(out[-1]), flush=True)
    return out


def markdown(device, power, cases, lib):
    out = ["# TSP local search with 2-opt and Or-opt on the GPU (`elg_tsp_local_search`)", "",
           "Measured on %s, power limit %s, with `tools/tsp_ls_timing.py` (CUDA events around one launch after a "
           "one-move warm-up launch).  Tours are the greedy rollouts of the seeded synthetic checkpoint (gain 3), best POMO "
           "row of every aug-instance.  max_iterations is %d, max_segment %d.  Each case runs the 2-opt + Or-opt search "
           "(`ls`) and 2-opt alone (`elg_two_opt`, `2opt`) on the same tours.  `us/move` is the call time over the largest "
           "per-tour move count (tours are refined side by side, one CTA each).  Pair evaluations count the position pairs "
           "of every search: N1^2 for `ls` (each pair covers up to six variants), (N1-1)(N1-2)/2 for `2opt`.  Cost is the "
           "best over the 8 augmentations, averaged over instances." % (device, power, MAX_IT, MAX_SEGMENT), "",
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
    return "\n".join(out) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_tsp_local_search"))
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
    plan = [(100, 16, 100), (1000, 1, 128)] if args.quick else [(100, 1000, 100), (1000, 1, 128), (4000, 1, 128)]
    cases = []
    for N, n, M in plan:
        xy, rows, before = random_case(N, n, M, seed=N)
        cases.append(summarize("TSP%d x %d" % (N, 8 * n), xy, rows, False, before))
        print(json.dumps(cases[-1]), flush=True)
    lib = tsplib_case(["eil51", "a280"] if args.quick else None)
    md = markdown(device, power, cases, lib)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out + ".md", "w") as f:
        f.write(md)
    with open(args.out + ".json", "w") as f:
        json.dump({"device": device, "power_limit": power, "cases": cases, "tsplib": lib}, f, indent=1)
    print(md)


if __name__ == "__main__":
    main()
