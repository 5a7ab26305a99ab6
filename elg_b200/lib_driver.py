"""Shared machinery of the two library drivers (elg_b200.cvrp.test_vrplib / elg_b200.tsp.test_tsplib), which keep the
reference's class names, config keys, result-file layout and printouts (CVRP/test_vrplib.py:15-151,
TSP/test_tsplib.py:18-168) but are thin shells around the functions here:

    solve_instance(model, env, aug)      one greedy rollout of a loaded instance -> (best cost over aug x POMO, tours, rewards)
    run_set(entries, solve, ...)         the per-instance loop with timing and the record dicts of the result files
    gap_bins(results, edges, ...)        mean gap per size bin, as the reference prints them

Optional 2-opt stage (config params.two_opt_iterations; absent or 0: nothing changes).  load_model records the setting on
the model; solve_instance then refines the best POMO row of every aug-instance in the library metric (rounded unscaled
coordinates) and returns the cost as an InstanceCost carrying the refined result; fill_record adds best_cost_2opt /
gap_2opt / two_opt_seconds / two_opt_iterations to the record; run_set prints one extra line per instance and gap_bins
one per size bin.  two_opt_refine is shared with the test.py drivers.

Optional CVRP local search stage (config params.local_search_iterations; absent or 0: nothing changes), independent of
the 2-opt stage and run on the same rows: solve_instance refines them with engine.cvrp_local_search in the library metric
(with the capacity CVRPEnv.load_vrplib_problem recorded), InstanceCost.local_search carries the result, fill_record adds
best_cost_ls / gap_ls / ls_seconds / ls_iterations, and run_set / gap_bins print their lines after the 2-opt ones.
load_model rejects the key for a TSP model.

Optional TSP local search stage (config params.tsp_local_search_iterations; absent or 0: nothing changes): 2-opt and
Or-opt moves (engine.tsp_local_search), independent of the 2-opt stage and run on the same rows in the library metric;
InstanceCost.tsp_local_search carries the result, fill_record adds best_cost_tsp_ls / gap_tsp_ls / tsp_ls_seconds /
tsp_ls_iterations, and run_set / gap_bins print their lines after the 2-opt ones.  load_model rejects the key for a CVRP
model.
"""
import json
import os
import time

import numpy as np
import torch

from . import engine


def require_cuda(config):
    if not config.get('use_cuda', True):
        raise RuntimeError("elg_b200 has no CPU path: set use_cuda: True")
    device = torch.device('cuda', config['cuda_device_num'])
    torch.cuda.set_device(device)
    return device


def load_model(model_cls, config, device, model=None, needs_local=True):
    """The reference's checkpoint protocol: add_local_policy BEFORE load_state_dict (CVRP/test.py:75-78)."""
    from .cvrp.CVRPModel import CVRPModel
    if not issubclass(model_cls, CVRPModel):
        reject_local_search(config)
    else:
        reject_tsp_local_search(config)
    if model is None:
        model = model_cls(**config['model_params'])
        if needs_local:
            model.decoder.add_local_policy(device)
        model.load_state_dict(torch.load(config['load_checkpoint'], map_location=device)['model_state_dict'])
    model = model.to(device)
    model.eval()
    model.requires_grad_(False)
    model._elg_two_opt_iterations = config.get('params', {}).get('two_opt_iterations') or 0
    model._elg_local_search_iterations = config.get('params', {}).get('local_search_iterations') or 0
    model._elg_tsp_local_search_iterations = config.get('params', {}).get('tsp_local_search_iterations') or 0
    return model


def reject_local_search(config):
    """The TSP drivers: params.local_search_iterations is the CVRP local search, TSP tours have the 2-opt stage."""
    if config.get('params', {}).get('local_search_iterations'):
        raise ValueError("params.local_search_iterations is the capacity-aware CVRP local search; "
                         "refine TSP tours with params.two_opt_iterations")


def reject_tsp_local_search(config):
    """The CVRP drivers: params.tsp_local_search_iterations is the TSP search, CVRP rows have their own local search."""
    if config.get('params', {}).get('tsp_local_search_iterations'):
        raise ValueError("params.tsp_local_search_iterations is the TSP 2-opt + Or-opt local search; "
                         "refine CVRP rows with params.local_search_iterations")


class InstanceCost(float):
    """Best cost of one instance (a plain float to every caller).  `two_opt` / `local_search` / `tsp_local_search` are
    (refined cost, seconds, moves) when the optional stage ran, else None."""
    two_opt = None
    local_search = None
    tsp_local_search = None


# optional refinement stages: (InstanceCost attribute, record key suffix, record key prefix, name in the printouts)
_STAGES = (('two_opt', '2opt', 'two_opt', '2-opt'), ('local_search', 'ls', 'ls', 'local search'),
           ('tsp_local_search', 'tsp_ls', 'tsp_ls', '2-opt + or-opt'))


def _best_rows(solutions, rewards):
    return solutions[torch.arange(rewards.shape[0], device=solutions.device), rewards.argmax(dim=1)]


def two_opt_refine(problem, xy, solutions, rewards, aug_factor, iterations, rounding):
    """2-opt (engine.two_opt, one launch) of the best POMO row of every aug-instance of a greedy rollout.
    xy (aug*n or 1, N1, 2) is the metric the cost is measured in: library runs pass the unscaled coordinates with
    rounding, random instances the scaled ones without.  -> (refined cost per instance, best over its augmentations (n,);
    seconds; moves applied per instance, summed over its augmentations (n,))"""
    rows = _best_rows(solutions, rewards)
    return _timed_refine(lambda: engine.two_opt(problem, xy, rows, max_iterations=iterations, rounding=rounding), aug_factor)


def local_search_refine(xy, demand, capacity, solutions, rewards, aug_factor, iterations, rounding):
    """CVRP local search (engine.cvrp_local_search, one launch) of the best POMO row of every aug-instance of a greedy
    rollout; demand (aug*n, N1) normalised as the environment holds it, capacity the integer capacity; otherwise as
    two_opt_refine."""
    rows = _best_rows(solutions, rewards)
    return _timed_refine(lambda: engine.cvrp_local_search(xy, rows, demand, capacity, max_iterations=iterations,
                                                          rounding=rounding), aug_factor)


def tsp_local_search_refine(xy, solutions, rewards, aug_factor, iterations, rounding):
    """TSP 2-opt + Or-opt local search (engine.tsp_local_search, one launch) of the best POMO row of every aug-instance
    of a greedy rollout; as two_opt_refine."""
    rows = _best_rows(solutions, rewards)
    return _timed_refine(lambda: engine.tsp_local_search(xy, rows, max_iterations=iterations, rounding=rounding),
                         aug_factor)


def _timed_refine(run, aug_factor):
    torch.cuda.synchronize()
    t0 = time.time()
    _, length, iters = run()
    torch.cuda.synchronize()
    seconds = time.time() - t0
    B = length.shape[0]
    cost = length.reshape(aug_factor, B // aug_factor).min(dim=0)[0]
    return cost, seconds, iters.reshape(aug_factor, B // aug_factor).sum(dim=0)


def solve_instance(model, env, rollout, aug_factor, width):
    """env already holds the instance.  Best of POMO, then best of augmentation (CVRP/test_vrplib.py:127-137)."""
    reset_state, _, _ = env.reset()
    model.pre_forward(reset_state)
    with torch.no_grad():
        solutions, _, rewards = rollout(model, env, 'greedy')
    best = -rewards.reshape(aug_factor, 1, width).max(dim=2)[0].max(dim=0)[0].float()
    cost = InstanceCost(best.cpu()[0])
    iterations = getattr(model, '_elg_two_opt_iterations', 0)
    if iterations:
        cvrp = hasattr(env, 'unscaled_depot_node_xy')
        refined, seconds, moves = two_opt_refine('cvrp' if cvrp else 'tsp',
                                                 env.unscaled_depot_node_xy if cvrp else env._unscaled_dev,
                                                 solutions, rewards, aug_factor, iterations, rounding=True)
        cost.two_opt = (float(refined[0]), seconds, int(moves[0]))
    iterations = getattr(model, '_elg_local_search_iterations', 0)
    if iterations:
        if env.capacity is None:
            raise ValueError("the local search stage needs the instance's capacity (CVRPEnv.load_vrplib_problem)")
        refined, seconds, moves = local_search_refine(env.unscaled_depot_node_xy, env.depot_node_demand, env.capacity,
                                                      solutions, rewards, aug_factor, iterations, rounding=True)
        cost.local_search = (float(refined[0]), seconds, int(moves[0]))
    iterations = getattr(model, '_elg_tsp_local_search_iterations', 0)
    if iterations:
        refined, seconds, moves = tsp_local_search_refine(env._unscaled_dev, solutions, rewards, aug_factor, iterations,
                                                          rounding=True)
        cost.tsp_local_search = (float(refined[0]), seconds, int(moves[0]))
    return cost, solutions, rewards


def run_set(entries, solve_one, repeat_times=1, echo_cost=False):
    """entries: iterable of (name, optimal, payload).  solve_one(name, payload, record) fills record['best_cost' / 'scale' / 'gap']."""
    results, total = [], 0.0
    for run_idx in range(repeat_times):
        for name, optimal, payload in entries:
            record = {'run_idx': run_idx}
            t0 = time.time()
            solve_one(name, payload, record)
            torch.cuda.synchronize()
            record['seconds'] = time.time() - t0
            total += record['seconds']
            results.append({'instance': name, 'optimal': optimal, 'record': [record]})
            print("Instance Name {}: gap {:.4f}".format(name, record['gap']))
            if echo_cost:
                print("cost: {}".format(record['best_cost']))
            for _, suffix, _, label in _STAGES:
                if 'gap_' + suffix in record:
                    print("Instance Name {}: gap after {} {:.4f}".format(name, label, record['gap_' + suffix]))
    return results, total


def fill_record(record, best_cost, scale, optimal):
    if record is not None:
        record['best_cost'] = float(best_cost)
        record['scale'] = scale
        record['gap'] = (best_cost - optimal) / optimal
        for attr, suffix, prefix, _ in _STAGES:
            if getattr(best_cost, attr, None):
                cost, seconds, moves = getattr(best_cost, attr)
                record['best_cost_' + suffix] = cost
                record['gap_' + suffix] = (cost - optimal) / optimal
                record[prefix + '_seconds'] = seconds
                record[prefix + '_iterations'] = moves    # moves applied, summed over the augmentations


def gap_bins(results, edges):
    """edges: [(label, lo_exclusive, hi_inclusive)] on the instance scale -> {label: mean gap in %}, plus 'total'.
    When the records carry an optional stage, also prints one line per bin and a total line for it, and adds
    'gap_2opt' / 'gap_ls' / 'gap_tsp_ls': {label: mean gap in %}."""
    out = _bin_means(results, edges, 'gap')
    for _, suffix, _, name in _STAGES:
        key = 'gap_' + suffix
        if results and all(key in r['record'][-1] for r in results):
            out[key] = _bin_means(results, edges, key)
            for label, mean in out[key].items():
                if label != 'total':
                    print("Average gap after {} on subset of {}: {:.2f}%".format(name, label, mean))
            print("Average gap after {} total: {:.2f}%".format(name, out[key]['total']))
    return out


def _bin_means(results, edges, key):
    gap = np.array([r['record'][-1][key] for r in results])
    scale = np.array([int(r['record'][-1]['scale']) for r in results])
    out = {}
    for label, lo, hi in edges:
        sel = (scale > lo) & (scale <= hi)
        if sel.any():
            out[label] = 100 * float(gap[sel].mean())
    out['total'] = 100 * float(gap.mean()) if len(gap) else float('nan')
    return out


def dump_results(results, out_dir, filename):
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, filename), 'w') as f:
            json.dump(results, f)
