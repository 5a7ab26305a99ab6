"""Drop-in for the reference's TSP/test.py evaluation loop (TSP/test.py:14-56).

`solve_batch` is one iteration of that loop (load + x8 augmentation, encode, greedy rollout, best-of-POMO and
best-of-augmentation); `test` is the loop with the reference's printout.  As a script it reads `config.yml` from the
current directory like the reference.
"""
import time

import torch

from .TSPEnv import TSPEnv
from .TSPModel import TSPModel
from .. import lib_driver as drv
from .utils import rollout


def solve_batch(model, env, batch, aug_factor):
    """-> (no_aug_cost (n,), aug_cost (n,), solutions (aug*n, M, N), rewards (aug*n, M))"""
    n = batch.shape[0]
    env.load_random_problems(batch, aug_factor)
    reset_state, _, _ = env.reset()
    with torch.no_grad():
        model.pre_forward(reset_state)
        solutions, probs, rewards = rollout(model=model, env=env, eval_type='greedy')
    aug_reward = rewards.reshape(aug_factor, n, env.pomo_size)
    max_pomo_reward, _ = aug_reward.max(dim=2)          # best of POMO
    no_aug_cost = -max_pomo_reward[0, :].float()
    max_aug_pomo_reward, _ = max_pomo_reward.max(dim=0)  # best of augmentation
    aug_cost = -max_aug_pomo_reward.float()
    return no_aug_cost, aug_cost, solutions, rewards


def test(dataloader, model, env, aug_factor, two_opt_iterations=0, tsp_local_search_iterations=0):
    """two_opt_iterations > 0 (config params.two_opt_iterations) also refines the best POMO row of every aug-instance
    with 2-opt in the reward metric and prints the refined cost after the reference's lines.
    tsp_local_search_iterations > 0 (params.tsp_local_search_iterations) does the same with the 2-opt + Or-opt local
    search, independently of the 2-opt stage."""
    model.eval()
    model.requires_grad_(False)
    avg_cost_total, no_avg_cost_total, t = 0., 0., 0
    two_opt_cost, two_opt_seconds, two_opt_moves = 0., 0., 0
    ls_cost, ls_seconds, ls_moves = 0., 0., 0
    start = time.time()
    for batch in dataloader:
        no_aug_cost, aug_cost, solutions, rewards = solve_batch(model, env, batch, aug_factor)
        avg_cost_total += aug_cost.mean()
        no_avg_cost_total += no_aug_cost.mean()
        if two_opt_iterations:
            cost, seconds, moves = drv.two_opt_refine("tsp", env.problems, solutions, rewards, aug_factor, two_opt_iterations,
                                                      rounding=False)
            two_opt_cost += cost.mean()
            two_opt_seconds += seconds
            two_opt_moves += int(moves.sum())
        if tsp_local_search_iterations:
            cost, seconds, moves = drv.tsp_local_search_refine(env.problems, solutions, rewards, aug_factor,
                                                               tsp_local_search_iterations, rounding=False)
            ls_cost += cost.mean()
            ls_seconds += seconds
            ls_moves += int(moves.sum())
        t += 1
    torch.cuda.synchronize()
    end = time.time()
    avg_cost_total /= t
    no_avg_cost_total /= t
    print("Aug cost: {:.4f}".format(avg_cost_total))
    print("no aug Avg cost: {:.4f}, Wall-clock time: {:.2f}s".format(no_avg_cost_total, float(end - start)))
    if two_opt_iterations:
        print("2-opt Aug cost: {:.4f}, 2-opt time: {:.2f}s, moves: {}".format(two_opt_cost / t, two_opt_seconds, two_opt_moves))
    if tsp_local_search_iterations:
        print("2-opt + or-opt Aug cost: {:.4f}, 2-opt + or-opt time: {:.2f}s, moves: {}".format(ls_cost / t, ls_seconds,
                                                                                                  ls_moves))
    return avg_cost_total


def load_model(config, device):
    """Checkpoint loading exactly as the reference (TSP/test.py:73-80)."""
    model_params = config['model_params']
    model = TSPModel(**model_params)
    if model_params['ensemble']:
        model.decoder.add_local_policy(device)
    checkpoint = torch.load(config['load_checkpoint'], map_location=device)
    model.load_state_dict(checkpoint['model_state_dict'])
    return model.to(device)


if __name__ == "__main__":
    import pickle
    import yaml
    with open('config.yml', 'r', encoding='utf-8') as f:
        config = yaml.load(f.read(), Loader=yaml.FullLoader)
    drv.reject_local_search(config)
    device = "cuda:{}".format(config['cuda_device_num'])
    model = load_model(config, device)
    env = TSPEnv(multi_width=config['params']['multiple_width'], device=device)
    with open(config['test_filename'], 'rb') as f:
        data = pickle.load(f)[:config['params']['test_size']]
    bs = config['params']['test_batch_size']
    batches = [torch.FloatTensor(data[i:i + bs]) for i in range(0, len(data), bs)]
    test(batches, model, env, aug_factor=config['params']['aug_factor'],
         two_opt_iterations=config['params'].get('two_opt_iterations') or 0,
         tsp_local_search_iterations=config['params'].get('tsp_local_search_iterations') or 0)
