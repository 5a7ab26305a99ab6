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
    if model is None:
        model = model_cls(**config['model_params'])
        if needs_local:
            model.decoder.add_local_policy(device)
        model.load_state_dict(torch.load(config['load_checkpoint'], map_location=device)['model_state_dict'])
    model = model.to(device)
    model.eval()
    model.requires_grad_(False)
    model._elg_two_opt_iterations = config.get('params', {}).get('two_opt_iterations') or 0
    return model


class InstanceCost(float):
    """Best cost of one instance (a plain float to every caller).  `two_opt` is (refined cost, seconds, moves) when the
    optional 2-opt stage ran, else None."""
    two_opt = None


def two_opt_refine(problem, xy, solutions, rewards, aug_factor, iterations, rounding):
    """2-opt (engine.two_opt, one launch) of the best POMO row of every aug-instance of a greedy rollout.
    xy (aug*n or 1, N1, 2) is the metric the cost is measured in: library runs pass the unscaled coordinates with
    rounding, random instances the scaled ones without.  -> (refined cost per instance, best over its augmentations (n,);
    seconds; moves applied per instance, summed over its augmentations (n,))"""
    B = rewards.shape[0]
    rows = solutions[torch.arange(B, device=solutions.device), rewards.argmax(dim=1)]
    torch.cuda.synchronize()
    t0 = time.time()
    _, length, iters = engine.two_opt(problem, xy, rows, max_iterations=iterations, rounding=rounding)
    torch.cuda.synchronize()
    seconds = time.time() - t0
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
            if 'gap_2opt' in record:
                print("Instance Name {}: gap after 2-opt {:.4f}".format(name, record['gap_2opt']))
    return results, total


def fill_record(record, best_cost, scale, optimal):
    if record is not None:
        record['best_cost'] = float(best_cost)
        record['scale'] = scale
        record['gap'] = (best_cost - optimal) / optimal
        if getattr(best_cost, 'two_opt', None):
            cost, seconds, moves = best_cost.two_opt
            record['best_cost_2opt'] = cost
            record['gap_2opt'] = (cost - optimal) / optimal
            record['two_opt_seconds'] = seconds
            record['two_opt_iterations'] = moves          # moves applied, summed over the augmentations


def gap_bins(results, edges):
    """edges: [(label, lo_exclusive, hi_inclusive)] on the instance scale -> {label: mean gap in %}, plus 'total'.
    When the records carry the 2-opt stage, also prints one line per bin and 'gap_2opt': {label: mean gap in %}."""
    out = _bin_means(results, edges, 'gap')
    if results and all('gap_2opt' in r['record'][-1] for r in results):
        out['gap_2opt'] = _bin_means(results, edges, 'gap_2opt')
        for label, mean in out['gap_2opt'].items():
            if label != 'total':
                print("Average gap after 2-opt on subset of {}: {:.2f}%".format(label, mean))
        print("Average gap after 2-opt total: {:.2f}%".format(out['gap_2opt']['total']))
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
