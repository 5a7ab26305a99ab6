"""Drop-in for the reference's CVRP/test.py evaluation loop (CVRP/test.py:14-56).

`solve_batch` is one iteration of that loop (load + x8 augmentation, encode, greedy rollout,
best-of-POMO and best-of-augmentation); `test` is the loop itself with the reference's printout.
Run as a script it reads `config.yml` from the current directory like the reference.
"""
import time

import torch

from .CVRPEnv import CVRPEnv
from .CVRPModel import CVRPModel
from .. import lib_driver as drv
from .utils import rollout


def solve_batch(model, env, batch, aug_factor):
    """-> (no_aug_cost (n,), aug_cost (n,), solutions (aug*n, M, T), rewards (aug*n, M))"""
    n = batch['loc'].shape[0]
    env.load_random_problems(batch, aug_factor)
    reset_state, _, _ = env.reset()
    with torch.no_grad():
        model.pre_forward(reset_state)
        solutions, probs, rewards = rollout(model=model, env=env, eval_type='greedy')
    aug_reward = rewards.reshape(aug_factor, n, env.multi_width)
    max_pomo_reward, _ = aug_reward.max(dim=2)          # best of POMO
    no_aug_cost = -max_pomo_reward[0, :].float()
    max_aug_pomo_reward, _ = max_pomo_reward.max(dim=0)  # best of augmentation
    aug_cost = -max_aug_pomo_reward.float()
    return no_aug_cost, aug_cost, solutions, rewards


def test(dataloader, model, env, aug_factor, two_opt_iterations=0, local_search_iterations=0, capacity=None,
         local_search_max_segment=1):
    """two_opt_iterations > 0 (config params.two_opt_iterations) also refines the best POMO row of every aug-instance
    with 2-opt in the reward metric and prints the refined cost after the reference's lines.  local_search_iterations > 0
    (params.local_search_iterations) does the same with the capacity-aware local search, independently of the 2-opt
    stage; it needs the integer vehicle capacity the batches' demands are normalised by, and moves chains of up to
    local_search_max_segment customers (params.local_search_max_segment)."""
    if local_search_iterations and capacity is None:
        raise ValueError("the local search stage needs the capacity the demands are normalised by")
    model.eval()
    model.requires_grad_(False)
    stages = drv.enabled_stages({'two_opt_iterations': two_opt_iterations,
                                 'local_search_iterations': local_search_iterations})
    totals = [[0., 0., 0] for _ in stages]              # cost, seconds, moves per enabled stage
    avg_cost_total, no_avg_cost_total, t = 0., 0., 0
    start = time.time()
    for batch in dataloader:
        no_aug_cost, aug_cost, solutions, rewards = solve_batch(model, env, batch, aug_factor)
        avg_cost_total += aug_cost.mean()
        no_avg_cost_total += no_aug_cost.mean()
        for (stage, iterations), total in zip(stages, totals):
            cost, seconds, moves = drv.refine(stage, "cvrp", env.depot_node_xy, solutions, rewards, aug_factor, iterations,
                                              False, env.depot_node_demand, capacity, local_search_max_segment)
            total[0] += cost.mean()
            total[1] += seconds
            total[2] += int(moves.sum())
        t += 1
    torch.cuda.synchronize()
    end = time.time()
    avg_cost_total /= t
    no_avg_cost_total /= t
    print("Aug cost: {:.4f}".format(avg_cost_total))
    print("no aug Avg cost: {:.4f}, Wall-clock time: {:.2f}s".format(no_avg_cost_total, float(end - start)))
    for (stage, _), (cost, seconds, moves) in zip(stages, totals):
        print("{0} Aug cost: {1:.4f}, {0} time: {2:.2f}s, moves: {3}".format(stage.label, cost / t, seconds, moves))
    return avg_cost_total


def load_model(config, device):
    """Checkpoint loading exactly as the reference (CVRP/test.py:73-79)."""
    model_params = config['model_params']
    model = CVRPModel(**model_params)
    checkpoint = torch.load(config['load_checkpoint'], map_location=device)
    if model_params['ensemble']:
        model.decoder.add_local_policy(device)
    model.load_state_dict(checkpoint['model_state_dict'])
    return model.to(device)


if __name__ == "__main__":
    import pickle
    import yaml
    with open('config.yml', 'r', encoding='utf-8') as f:
        config = yaml.load(f.read(), Loader=yaml.FullLoader)
    drv.reject('cvrp', config)
    device = "cuda:{}".format(config['cuda_device_num'])
    model = load_model(config, device)
    env = CVRPEnv(multi_width=config['params']['multiple_width'], device=device)
    with open(config['test_filename'], 'rb') as f:
        data = pickle.load(f)[:config['params']['test_size']]
    bs = config['params']['test_batch_size']
    batches = [{'depot': torch.FloatTensor([d[0] for d in data[i:i + bs]]),
                'loc': torch.FloatTensor([d[1] for d in data[i:i + bs]]),
                'demand': torch.FloatTensor([d[2] for d in data[i:i + bs]]) / float(data[0][3])}
               for i in range(0, len(data), bs)]
    test(batches, model, env, aug_factor=config['params']['aug_factor'],
         two_opt_iterations=config['params'].get('two_opt_iterations') or 0,
         local_search_iterations=config['params'].get('local_search_iterations') or 0, capacity=data[0][3],
         local_search_max_segment=config['params'].get('local_search_max_segment') or 1)
