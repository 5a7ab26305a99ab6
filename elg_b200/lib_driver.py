"""Shared machinery of the two library drivers (elg_b200.cvrp.test_vrplib / elg_b200.tsp.test_tsplib), which keep the
reference's class names, config keys, result-file layout and printouts (CVRP/test_vrplib.py:15-151,
TSP/test_tsplib.py:18-168) but are thin shells around the functions here:

    solve_instance(model, env, aug)      one greedy rollout of a loaded instance -> (best cost over aug x POMO, tours, rewards)
    run_set(entries, solve, ...)         the per-instance loop with timing and the record dicts of the result files
    gap_bins(results, edges, ...)        mean gap per size bin, as the reference prints them

Optional refinement stages (STAGES; a config key absent or 0: nothing changes): 2-opt (params.two_opt_iterations, both
problems), the capacity-aware CVRP local search (params.local_search_iterations, with the capacity
CVRPEnv.load_vrplib_problem recorded, and its longest Or-opt chain params.local_search_max_segment, 1..3, default 1) and
the TSP 2-opt + Or-opt local search (params.tsp_local_search_iterations).
load_model records the settings on the model and rejects a key the problem does not accept; solve_instance then refines
the best POMO row of every aug-instance with every enabled stage, independently and in the library metric (rounded
unscaled coordinates), and returns the cost as an InstanceCost carrying each stage's result; fill_record adds the
stage's best_cost_ / gap_ / _seconds / _iterations keys to the record, and run_set / gap_bins print one extra line per
instance and per size bin, in the order of STAGES.  refine is shared with the test.py drivers.
"""
import json
import os
import time
from collections import namedtuple

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
    reject('cvrp' if issubclass(model_cls, CVRPModel) else 'tsp', config)
    if model is None:
        model = model_cls(**config['model_params'])
        if needs_local:
            model.decoder.add_local_policy(device)
        model.load_state_dict(torch.load(config['load_checkpoint'], map_location=device)['model_state_dict'])
    model = model.to(device)
    model.eval()
    model.requires_grad_(False)
    model._elg_stage_iterations = {stage.key: config.get('params', {}).get(stage.key) or 0 for stage in STAGES}
    model._elg_local_search_max_segment = config.get('params', {}).get('local_search_max_segment') or 1
    return model


class InstanceCost(float):
    """Best cost of one instance (a plain float to every caller).  `two_opt` / `local_search` / `tsp_local_search` are
    (refined cost, seconds, moves) when the optional stage ran, else None."""
    two_opt = None
    local_search = None
    tsp_local_search = None


def _cvrp_local_search(problem, xy, rows, demand, capacity, iterations, rounding, max_segment):
    if capacity is None:
        raise ValueError("the local search stage needs the instance's capacity (CVRPEnv.load_vrplib_problem)")
    return engine.cvrp_local_search(xy, rows, demand, capacity, max_iterations=iterations, rounding=rounding,
                                    max_segment=max_segment)


# An optional refinement stage: config key (under params), problems that accept it, InstanceCost attribute, record key
# suffix and prefix, name in the printouts, rejection message for the other problem, and the engine call
# run(problem, xy, rows, demand, capacity, iterations, rounding, max_segment) -> (tours, length, moves); max_segment
# (params.local_search_max_segment) only concerns the CVRP local search.
Stage = namedtuple('Stage', 'key problems attr suffix prefix label rejection run')
STAGES = (
    Stage('two_opt_iterations', ('tsp', 'cvrp'), 'two_opt', '2opt', 'two_opt', '2-opt', None,
          lambda problem, xy, rows, demand, capacity, iterations, rounding, max_segment:
          engine.two_opt(problem, xy, rows, max_iterations=iterations, rounding=rounding)),
    Stage('local_search_iterations', ('cvrp',), 'local_search', 'ls', 'ls', 'local search',
          "params.local_search_iterations is the capacity-aware CVRP local search; "
          "refine TSP tours with params.two_opt_iterations", _cvrp_local_search),
    Stage('tsp_local_search_iterations', ('tsp',), 'tsp_local_search', 'tsp_ls', 'tsp_ls', '2-opt + or-opt',
          "params.tsp_local_search_iterations is the TSP 2-opt + Or-opt local search; "
          "refine CVRP rows with params.local_search_iterations",
          lambda problem, xy, rows, demand, capacity, iterations, rounding, max_segment:
          engine.tsp_local_search(xy, rows, max_iterations=iterations, rounding=rounding)),
)


def reject(problem, config):
    """Raises ValueError for a stage key in config['params'] that the problem ('tsp' / 'cvrp') does not accept, and for
    a params.local_search_max_segment that is not 1..3 or has no CVRP local search stage to feed."""
    params = config.get('params', {})
    for stage in STAGES:
        if problem not in stage.problems and params.get(stage.key):
            raise ValueError(stage.rejection)
    max_segment = params.get('local_search_max_segment')
    if max_segment is None:
        return
    if problem != 'cvrp':
        raise ValueError("params.local_search_max_segment is the longest Or-opt chain of the CVRP local search; the TSP "
                         "local search (params.tsp_local_search_iterations) always moves chains of up to 3 nodes")
    if max_segment not in (1, 2, 3):
        raise ValueError("params.local_search_max_segment must be 1, 2 or 3 (got %r)" % (max_segment,))
    if not params.get('local_search_iterations'):
        raise ValueError("params.local_search_max_segment needs the local search stage: set params.local_search_iterations")


def enabled_stages(iterations):
    """{config key: iterations} -> [(stage, iterations)] of the stages with iterations > 0, in the order of STAGES"""
    return [(stage, iterations[stage.key]) for stage in STAGES if iterations.get(stage.key)]


def refine(stage, problem, xy, solutions, rewards, aug_factor, iterations, rounding, demand=None, capacity=None,
           max_segment=1):
    """One stage (one launch) on the best POMO row of every aug-instance of a greedy rollout.  xy (aug*n or 1, N1, 2) is
    the metric the cost is measured in: library runs pass the unscaled coordinates with rounding, random instances the
    scaled ones without; the CVRP local search also takes demand (aug*n, N1), normalised as the environment holds it, the
    integer capacity and its longest Or-opt chain max_segment.  -> (refined cost per instance, best over its augmentations (n,); seconds; moves applied per
    instance, summed over its augmentations (n,))"""
    rows = solutions[torch.arange(rewards.shape[0], device=solutions.device), rewards.argmax(dim=1)]
    torch.cuda.synchronize()
    t0 = time.time()
    _, length, iters = stage.run(problem, xy, rows, demand, capacity, iterations, rounding, max_segment)
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
    cvrp = hasattr(env, 'unscaled_depot_node_xy')
    for stage, iterations in enabled_stages(getattr(model, '_elg_stage_iterations', {})):
        if cvrp:
            refined, seconds, moves = refine(stage, 'cvrp', env.unscaled_depot_node_xy, solutions, rewards, aug_factor,
                                             iterations, True, env.depot_node_demand, env.capacity,
                                             getattr(model, '_elg_local_search_max_segment', 1))
        else:
            refined, seconds, moves = refine(stage, 'tsp', env._unscaled_dev, solutions, rewards, aug_factor, iterations,
                                             True)
        setattr(cost, stage.attr, (float(refined[0]), seconds, int(moves[0])))
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
            for stage in STAGES:
                if 'gap_' + stage.suffix in record:
                    print("Instance Name {}: gap after {} {:.4f}".format(name, stage.label, record['gap_' + stage.suffix]))
    return results, total


def fill_record(record, best_cost, scale, optimal):
    if record is not None:
        record['best_cost'] = float(best_cost)
        record['scale'] = scale
        record['gap'] = (best_cost - optimal) / optimal
        for stage in STAGES:
            if getattr(best_cost, stage.attr, None):
                cost, seconds, moves = getattr(best_cost, stage.attr)
                record['best_cost_' + stage.suffix] = cost
                record['gap_' + stage.suffix] = (cost - optimal) / optimal
                record[stage.prefix + '_seconds'] = seconds
                record[stage.prefix + '_iterations'] = moves    # moves applied, summed over the augmentations


def gap_bins(results, edges):
    """edges: [(label, lo_exclusive, hi_inclusive)] on the instance scale -> {label: mean gap in %}, plus 'total'.
    When the records carry an optional stage, also prints one line per bin and a total line for it, and adds
    'gap_2opt' / 'gap_ls' / 'gap_tsp_ls': {label: mean gap in %}."""
    out = _bin_means(results, edges, 'gap')
    for stage in STAGES:
        key = 'gap_' + stage.suffix
        if results and all(key in r['record'][-1] for r in results):
            out[key] = _bin_means(results, edges, key)
            for label, mean in out[key].items():
                if label != 'total':
                    print("Average gap after {} on subset of {}: {:.2f}%".format(stage.label, label, mean))
            print("Average gap after {} total: {:.2f}%".format(stage.label, out[key]['total']))
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
