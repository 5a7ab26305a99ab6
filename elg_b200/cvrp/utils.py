"""Drop-in for the reference's CVRP/utils.py: rollout, 2-opt, x8 augmentation, feasibility check, seeding; plus the
capacity-aware local search cvrp_local_search.

`rollout(model, env, eval_type)` keeps the reference signature and return convention
(CVRP/utils.py:7-29): (solutions (B, M, T) int64, probs (B, T, M) | None, reward (B, M)).
When both `model` and `env` are elg_b200 objects the whole loop runs as ONE kernel launch
(elg_rollout); otherwise it falls back to the reference's step-by-step protocol so that either
side can be mixed with reference objects.
"""
import random

import numpy as np
import torch

from .. import _lib, engine


def rollout(model, env, eval_type='greedy'):
    if getattr(model, "_elg_fused", False) and getattr(env, "_elg_fused", False):
        return _fused_rollout(model, env, eval_type)
    env.reset()
    actions, probs = [], []
    state, reward, done = env.pre_step()
    while not done:
        cur_dist, cur_theta, xy, norm_demand = env.get_cur_feature()
        selected, one_step_prob = model.one_step_rollout(state, cur_dist, cur_theta, xy, norm_demand=norm_demand,
                                                         eval_type=eval_type)
        state, reward, done = env.step(selected)
        actions.append(selected)
        probs.append(one_step_prob)
    actions = torch.stack(actions, 1)
    probs = None if eval_type == 'greedy' else torch.stack(probs, 1)
    return torch.transpose(actions, 1, 2), probs, reward


def _fused_rollout(model, env, eval_type):
    """Whole rollout in one launch.  In 'sample' mode the per-step probabilities are not materialised;
    `probs` has the reference's (B, T, M) shape and the trajectory log-likelihood as its log-sum (see _probs_from_logp)."""
    env.reset()
    batch = model._batch
    if batch is None or batch.xy.data_ptr() != env.depot_node_xy.data_ptr():
        raise RuntimeError("model.pre_forward(reset_state) must be called on this env's problems before rollout")
    M = env.multi_width
    # POMO start nodes: python RNG on the host exactly as the reference (CVRP/CVRPModel.py:47)
    start = random.sample(range(0, env.problem_size), M)
    batch.tables.unscaled = env.unscaled_depot_node_xy.data_ptr() if env.vrplib else None
    tours16, reward, logp, n_steps = engine.rollout(batch, M, start, mode=eval_type, seed=model._next_seed())
    T = int(n_steps.max().item())
    solutions = tours16[:, :, :T].long()
    env._finish_fused(solutions, reward)
    probs = None if eval_type == 'greedy' else _probs_from_logp(logp, T)
    model._last_logp = logp
    return solutions, probs, reward


def _probs_from_logp(logp, T):
    """(B, M) trajectory log-likelihood -> (B, T, M) tensor with the reference's shape whose `probs.log().sum(dim=1)`
    (CVRP/train.py:115) is that log-likelihood.  The fused rollout does not materialise per-step probabilities; exp(logp) itself
    underflows fp32 (an untrained CVRP100 policy has log-likelihoods around -360), so every step carries the geometric
    mean exp(logp / T) -- an expanded view, no memory.  The exact value is also kept as `model._last_logp`."""
    return torch.exp(logp / T)[:, None, :].expand(-1, T, -1)


def batched_two_opt_torch(points, tour, max_iterations=1000, device=None):
    """2-opt local search on depot-delimited CVRP tours (CVRP/utils.py:31-67), on the GPU (elg_two_opt).

    points (N+1, 2) with the depot at row 0; tour (batch, T) node ids, depot visits as 0 (a rollout row); numpy or torch,
    and the result comes back in the same type and dtype.  Returns (tour, iterations), iterations being the largest number
    of moves any tour took.  device=None is the current CUDA device; there is no CPU path.

    The reference tree is not part of this project; the signature is that of the DIFUSCO utility the cited lines are
    understood to be.  Two deliberate differences: every tour stops on its own (the reference's loop couples the batch
    and runs while any tour improves), and a move only reverses customers of one route, depot edges included, so every
    route keeps its customers and its load.  The TSP function applied to these tours would reverse segments across depot
    visits and could break capacity."""
    return _dropin("batched_two_opt_torch", points, tour, device,
                   lambda xy, t: engine.two_opt("cvrp", xy, t, max_iterations=max_iterations))


def _dropin(name, points, tour, device, search):
    """Shared body of the drop-in searches of both sub-projects (name: the calling function): the CUDA device
    (device=None: the current one), numpy / torch in and out.  search(xy (1, N, 2) fp32, tours int64), both on that
    device, -> (tours, length, iterations) of the engine; returns (tours in the input's type and dtype, the largest move
    count)."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise _lib.ElgError("%s needs a CUDA device (got %s): elg_b200 has no CPU path" % (name, dev))
    t = torch.as_tensor(tour)
    refined, _, iters = search(torch.as_tensor(points).to(dev, torch.float32)[None], t.to(dev, torch.int64))
    n_iter = int(iters.max()) if iters.numel() else 0
    if isinstance(tour, np.ndarray):
        return refined.cpu().numpy().astype(tour.dtype), n_iter
    return refined.to(t.device, t.dtype), n_iter


def cvrp_local_search(points, demand, capacity, tour, max_iterations=1000, device=None, max_segment=1):
    """Capacity-aware CVRP local search on the GPU (elg_cvrp_local_search_ex): 2-opt inside a route, relocate, swap and
    2-opt* between routes, and with max_segment 2 or 3 Or-opt moves of chains of up to that many customers, best
    improvement, every tour stopping on its own.

    points (N+1, 2) with the depot at row 0; demand (N+1,) normalised by the capacity as the environments hold it (depot
    0); capacity the integer vehicle capacity; tour (batch, T) rollout rows (depot visits as 0, every customer once, every
    route within capacity); numpy or torch, and the tour comes back in the same type and dtype, in canonical form (routes
    in order, each preceded by one 0, zero padding to T).  Returns (tour, iterations), iterations being the largest number
    of moves any tour took.  device=None is the current CUDA device; there is no CPU path."""
    return _dropin("cvrp_local_search", points, tour, device, lambda xy, t: engine.cvrp_local_search(
        xy, t, torch.as_tensor(demand).to(xy.device, torch.float32)[None], capacity, max_iterations=max_iterations,
        max_segment=max_segment))


def augment_xy_data_by_8_fold(problems):
    """(batch, problem, 2) -> (8*batch, problem, 2); CVRP/utils.py:69-87."""
    if problems.is_cuda:
        xy, _ = engine.load_problems("tsp", problems, aug=8)
        return xy
    x, y = problems[:, :, [0]], problems[:, :, [1]]
    v = [(x, y), (1 - x, y), (x, 1 - y), (1 - x, 1 - y), (y, x), (1 - y, x), (y, 1 - x), (1 - y, 1 - x)]
    return torch.cat([torch.cat(p, dim=2) for p in v], dim=0)


def check_feasible(pi, demand):
    """Known-answer invariant of the reference (CVRP/utils.py:90-119): input (1, multi, T) tours and
    (1, problem) demands; every customer exactly once and capacity never above 1 + 1e-4."""
    pi = pi.squeeze(0)
    multi = pi.shape[0]
    problem_size = demand.shape[1]
    demand = demand.expand(multi, problem_size)
    sorted_pi = pi.data.sort(1)[0]
    want = torch.arange(1, problem_size + 1, device=pi.device).view(1, -1).expand(multi, problem_size)
    assert (want == sorted_pi[:, -problem_size:]).all() and (sorted_pi[:, :-problem_size] == 0).all(), "Invalid tour"
    d = torch.cat((torch.full_like(demand[:, :1], -1), demand), 1).gather(1, pi)
    used = torch.zeros_like(demand[:, 0])
    for i in range(pi.size(1)):
        used += d[:, i]
        used[used < 0] = 0
        assert (used <= 1 + 1e-4).all(), "Used more than capacity"


def seed_everything(seed=2022):
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)
