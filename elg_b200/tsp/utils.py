"""Drop-in for the reference's TSP/utils.py: rollout (TSP/utils.py:7-26), 2-opt, x8 augmentation, seeding; plus the
2-opt + Or-opt local search tsp_local_search."""
import random

import numpy as np
import torch

from .. import engine
from ..cvrp.utils import _dropin, augment_xy_data_by_8_fold, seed_everything  # noqa: F401  (same functions in both sub-projects)


def rollout(model, env, eval_type='greedy'):
    if getattr(model, "_elg_fused", False) and getattr(env, "_elg_fused", False):
        return _fused_rollout(model, env, eval_type)
    env.reset()
    actions, probs = [], []
    state, reward, done = env.pre_step()
    while not done:
        cur_dist, cur_theta, xy = env.get_local_feature()
        selected, one_step_prob = model.one_step_rollout(state, cur_dist=cur_dist, cur_theta=cur_theta, xy=xy,
                                                         eval_type=eval_type)
        state, reward, done = env.step(selected)
        actions.append(selected)
        probs.append(one_step_prob)
    actions = torch.stack(actions, 1)
    probs = None if eval_type == 'greedy' else torch.stack(probs, 1)
    return torch.transpose(actions, 1, 2), probs, reward


def _fused_rollout(model, env, eval_type):
    env.reset()
    batch = model._batch
    if batch is None or batch.xy.data_ptr() != env.problems.data_ptr():
        raise RuntimeError("model.pre_forward(reset_state) must be called on this env's problems before rollout")
    M = env.pomo_size
    start = random.sample(range(0, M), M)            # TSP/TSPModel.py:31
    batch.tables.unscaled = env._unscaled_dev.data_ptr() if env.tsplib else None
    tours16, reward, logp, n_steps = engine.rollout(batch, M, start, mode=eval_type, seed=model._next_seed())
    solutions = tours16[:, :, :env.problem_size].long()
    env._finish_fused(solutions)
    probs = None if eval_type == 'greedy' else _probs_from_logp(logp, env.problem_size)
    model._last_logp = logp
    return solutions, probs, reward


def batched_two_opt_torch(points, tour, max_iterations=1000, device=None):
    """2-opt local search on closed TSP tours (TSP/utils.py:28-70), on the GPU (elg_two_opt).

    points (N, 2); tour (batch, N+1) closed tours (last node = first node); numpy or torch, and the result comes back in
    the same type and dtype.  Returns (tour, iterations), iterations being the largest number of moves any tour took.
    Position 0 (the start node) never moves.  device=None is the current CUDA device; there is no CPU path.

    The reference tree is not part of this project; the signature is that of the DIFUSCO utility the cited lines are
    understood to be.  One deliberate difference: every tour stops on its own, where the reference's loop couples the
    batch and runs while any tour improves."""
    return _dropin("batched_two_opt_torch", points, tour, device,
                   _closed(lambda xy, t: engine.two_opt("tsp", xy, t, max_iterations=max_iterations)))


def tsp_local_search(points, tour, max_iterations=1000, max_segment=3, device=None):
    """2-opt + Or-opt local search on closed TSP tours, on the GPU (elg_tsp_local_search): best improvement over 2-opt
    and the moves of a segment of 1..max_segment consecutive nodes, forward or reversed, onto another edge; every tour
    stops on its own.  max_segment = 0 is batched_two_opt_torch.

    points (N, 2); tour (batch, N+1) closed tours (last node = first node); numpy or torch, and the result comes back in
    the same type and dtype.  Returns (tour, iterations), iterations being the largest number of moves any tour took.
    Position 0 (the start node) never moves.  device=None is the current CUDA device; there is no CPU path."""
    return _dropin("tsp_local_search", points, tour, device, _closed(
        lambda xy, t: engine.tsp_local_search(xy, t, max_iterations=max_iterations, max_segment=max_segment)))


def _closed(search):
    """search(xy, tours) of the engine -> the same on closed tours (batch, N+1), last node = first node"""
    def closed_search(xy, t):
        if t.dim() != 2 or t.shape[1] < 2 or not bool((t[:, -1] == t[:, 0]).all()):
            raise ValueError("tsp tours must be (batch, N+1) closed tours (last node = first node)")
        refined, length, iters = search(xy, t[:, :-1].contiguous())
        return torch.cat((refined, refined[:, :1]), dim=1), length, iters
    return closed_search


def check_feasible(pi):
    """Every node exactly once (TSP/utils.py:72-78); input (1, multi, problem)."""
    pi = pi.squeeze(0)
    want = torch.arange(pi.size(1), device=pi.device).view(1, -1).expand_as(pi)
    assert (want == pi.data.sort(1)[0]).all(), "Invalid tour"
