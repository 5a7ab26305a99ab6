"""Inputs of the local-search GPU tests (test_gpu_two_opt.py, test_gpu_cvrp_ls.py, test_gpu_tsp_ls.py): greedy rows of the
seeded synthetic model on random instances, and the library drivers run on one TSPLIB / Set-X instance."""
import json
import os
import random

import numpy as np
import torch

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "tests", "golden", "lib")


def cfg(problem, **params):
    """Driver config of the synthetic model with extra params (e.g. two_opt_iterations=100)."""
    from elg_b200.synth import DEFAULT_MODEL_PARAMS
    c = {"name": "ELG", "use_cuda": True, "cuda_device_num": 0, "load_checkpoint": None,
         "params": dict(aug_factor=8, **params), "model_params": dict(DEFAULT_MODEL_PARAMS[problem])}
    if problem == "cvrp":
        c["vrplib_set"] = "X"
    return c


def model(problem, wseed, gain):
    """The CVRPModel / TSPModel of the synthetic weights, local policy added before loading them."""
    from elg_b200.cvrp import CVRPModel
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    from elg_b200.tsp import TSPModel
    m = (CVRPModel if problem == "cvrp" else TSPModel)(**DEFAULT_MODEL_PARAMS[problem])
    m.decoder.add_local_policy(DEV)
    m.load_state_dict(synthetic_state_dict(problem, seed=wseed, gain=gain))
    return m


def greedy_rows(problem, N, n, seed, aug=8, capacity=None):
    """Greedy rollout of n random instances x aug with the synthetic model -> (xy (B, N1, 2), demand | None,
    best POMO row of every aug-instance (B, L) int64), all on the GPU.  capacity: synthetic_cvrp_batch's."""
    from elg_b200 import engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict, synthetic_tsp_batch
    if problem == "cvrp":
        b = synthetic_cvrp_batch(n, N, seed=seed, capacity=capacity)
        xy, dem = engine.load_problems("cvrp", b["loc"].to(DEV), b["depot"].to(DEV), b["demand"].to(DEV), aug=aug)
    else:
        xy, dem = engine.load_problems("tsp", synthetic_tsp_batch(n, N, seed=seed).to(DEV), aug=aug)
    h = engine.ModelHandle(problem, DEFAULT_MODEL_PARAMS[problem], synthetic_state_dict(problem, seed=1234, gain=3.0), DEV)
    tours16, reward, _, n_steps = engine.rollout(engine.encode(h, xy, dem), N, random.Random(seed).sample(range(N), N))
    T = int(n_steps.max()) if problem == "cvrp" else N
    return xy, dem, tours16[torch.arange(xy.shape[0], device=DEV), reward.argmax(1), :T].long()


def _library(kind):
    with open(os.path.join(LIB, kind + "_ref.json")) as f:
        ref = json.load(f)
    return ref, np.load(os.path.join(LIB, kind + "_inputs.npz"))


def _run_setx(name, config, ref, z):
    """The Set-X driver on one instance -> (solutions, rewards, record, capacity, optimal cost)"""
    from elg_b200.cvrp.test_vrplib import VRPLib_Tester
    tester = VRPLib_Tester(config, model=model("cvrp", ref["wseed"], ref["gain"]))
    cap, opt = z[name + "/capopt"]
    inst = {"node_coord": z[name + "/coord"].astype(np.float64), "demand": z[name + "/demand"].astype(np.float64),
            "capacity": float(cap), "depot": np.array([0])}
    random.seed(ref["seed"])
    res = {}
    sols, rewards = tester.test_on_one_ins(name=name, result_dict=res, instance=inst, solution=float(opt))
    return sols, rewards, res, cap, opt


def tsplib_driver(name, params):
    """The TSPLIB driver on one instance with extra config params -> (record, best rows)."""
    from elg_b200.tsp.test_tsplib import TSPLib_Tester
    ref, z = _library("tsplib")
    m = model("tsp", ref["wseed"], ref["gain"])
    random.seed(ref["seed"])
    res = {}
    sols, rewards = TSPLib_Tester(cfg("tsp", **params), model=m).test_on_one_ins(
        name, res, [z[name + "/coord"], float(z[name + "/opt"])])
    return res, sols[torch.arange(rewards.shape[0], device=DEV), rewards.argmax(1)]


def lib_rows(kind, name, two_opt_iterations=None):
    """Greedy rollout of one library instance through its driver -> (unscaled xy (B or 1, N1, 2), best rows (B, L),
    the driver's record, the optimal cost).  two_opt_iterations: params.two_opt_iterations (None: key absent)."""
    from elg_b200 import engine
    params = {} if two_opt_iterations is None else {"two_opt_iterations": two_opt_iterations}
    if kind == "tsplib":
        z = _library("tsplib")[1]
        res, rows = tsplib_driver(name, params)
        xy = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None].to(DEV)           # shared by all augmentations
        return xy, rows, res, float(z[name + "/opt"])
    ref, z = _library("setx")
    sols, rewards, res, _, opt = _run_setx(name, cfg("cvrp", **params), ref, z)
    xy = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None]
    xy = engine.load_problems("cvrp", xy[:, 1:].to(DEV), xy[:, 0].to(DEV),
                              torch.zeros(1, xy.shape[1] - 1, device=DEV), aug=8)[0]         # x8 unscaled, as the driver
    return xy, sols[torch.arange(rewards.shape[0], device=DEV), rewards.argmax(1)], res, float(opt)


def setx_rows(name):
    """Greedy rollout of one Set-X instance through its driver -> (unscaled xy x8 (8, N1, 2), normalised demand (8, N1),
    integer capacity, best rows (8, L))."""
    from elg_b200 import engine
    ref, z = _library("setx")
    sols, rewards, _, cap, _ = _run_setx(name, cfg("cvrp"), ref, z)
    c = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None].to(DEV)
    dem = torch.tensor(z[name + "/demand"], dtype=torch.float32)[None].to(DEV) / float(cap)
    xy, dem = engine.load_problems("cvrp", c[:, 1:], c[:, 0], dem[:, 1:], aug=8)
    return xy, dem, int(cap), sols[torch.arange(8, device=DEV), rewards.argmax(1)]
