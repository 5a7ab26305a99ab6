"""2-opt local search on the GPU (elg_two_opt, engine.two_opt, batched_two_opt_torch, the drivers' opt-in refinement)
against the CPU oracle (tests/two_opt_oracle.py).

Under the rounded library metric every edge is an integer, so gains are exact in fp32 and fp64 alike and the kernel must
make the oracle's moves exactly.  Under the scaled metric the kernel's fp32 gains can order near-ties differently from the
oracle's fp64 gains, so there the invariants are exact and the tours only mostly equal."""
import json
import os
import random

import numpy as np
import pytest
import torch

import two_opt_oracle as TO
from oracle import elg_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "tests", "golden", "lib")


def _model(problem, wseed=1234, gain=3.0):
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    from elg_b200 import engine
    return engine.ModelHandle(problem, DEFAULT_MODEL_PARAMS[problem], synthetic_state_dict(problem, seed=wseed, gain=gain), DEV)


def _greedy_rows(problem, N, n, seed, aug=8):
    """Greedy rollout of n random instances x aug with the synthetic model -> (xy (B, N1, 2), demand | None,
    best POMO row of every aug-instance (B, L) int64), all on the GPU."""
    from elg_b200 import engine
    from elg_b200.synth import synthetic_cvrp_batch, synthetic_tsp_batch
    if problem == "cvrp":
        b = synthetic_cvrp_batch(n, N, seed=seed)
        xy, dem = engine.load_problems("cvrp", b["loc"].to(DEV), b["depot"].to(DEV), b["demand"].to(DEV), aug=aug)
    else:
        xy, dem = engine.load_problems("tsp", synthetic_tsp_batch(n, N, seed=seed).to(DEV), aug=aug)
    batch = engine.encode(_model(problem), xy, dem)
    M = N
    rng = random.Random(seed)
    tours16, reward, _, n_steps = engine.rollout(batch, M, rng.sample(range(N), M))
    T = int(n_steps.max()) if problem == "cvrp" else N
    rows = tours16[torch.arange(xy.shape[0], device=DEV), reward.argmax(1), :T].long()
    return xy, dem, rows


def _lib_rows(kind, name, two_opt_iterations=None):
    """Greedy rollout of one library instance through its driver -> (unscaled xy (B or 1, N1, 2), best rows (B, L),
    the driver's record, the optimal cost).  two_opt_iterations: params.two_opt_iterations (None: key absent)."""
    with open(os.path.join(LIB, kind + "_ref.json")) as f:
        ref = json.load(f)
    z = np.load(os.path.join(LIB, kind + "_inputs.npz"))
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    problem = "cvrp" if kind == "setx" else "tsp"
    cfg = {"name": "ELG", "use_cuda": True, "cuda_device_num": 0, "vrplib_set": "X", "load_checkpoint": None,
           "params": {"aug_factor": 8}, "model_params": dict(DEFAULT_MODEL_PARAMS[problem])}
    if two_opt_iterations is not None:
        cfg["params"]["two_opt_iterations"] = two_opt_iterations
    sd = synthetic_state_dict(problem, seed=ref["wseed"], gain=ref["gain"])
    random.seed(ref["seed"])
    if problem == "cvrp":
        from elg_b200.cvrp import CVRPModel as Model
        from elg_b200.cvrp.test_vrplib import VRPLib_Tester as Tester
    else:
        from elg_b200.tsp import TSPModel as Model
        from elg_b200.tsp.test_tsplib import TSPLib_Tester as Tester
    m = Model(**cfg["model_params"])
    m.decoder.add_local_policy(DEV)
    m.load_state_dict(sd)
    tester = Tester(cfg, model=m)
    res = {}
    if problem == "cvrp":
        cap, opt = z[name + "/capopt"]
        inst = {"node_coord": z[name + "/coord"].astype(np.float64), "demand": z[name + "/demand"].astype(np.float64),
                "capacity": float(cap), "depot": np.array([0])}
        sols, rewards = tester.test_on_one_ins(name=name, result_dict=res, instance=inst, solution=float(opt))
        xy = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None]
        from elg_b200 import engine
        xy = engine.load_problems("cvrp", xy[:, 1:].to(DEV), xy[:, 0].to(DEV),
                                  torch.zeros(1, xy.shape[1] - 1, device=DEV), aug=8)[0]   # x8 unscaled, as the driver
    else:
        opt = float(z[name + "/opt"])
        sols, rewards = tester.test_on_one_ins(name, res, [z[name + "/coord"], opt])
        xy = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None].to(DEV)           # shared by all augmentations
    B = rewards.shape[0]
    return xy, sols[torch.arange(B, device=DEV), rewards.argmax(1)], res, float(opt)


def _oracle(problem, xy, rows, max_iterations, rounding):
    return TO.two_opt(problem, xy.cpu(), rows.cpu(), max_iterations, rounding)


def _min_gain_fp64(problem, xy, t):
    """Smallest admissible gain of one tour, everything in fp64."""
    p = xy.double()
    n = len(t)
    pos = torch.arange(n)
    nxt = (pos + 1) % n
    d = lambda a, b: ((p[a] - p[b]) ** 2).sum(-1).sqrt()
    i, j = pos[:, None], pos[None, :]
    g = d(t[i], t[j]) + d(t[nxt[i]], t[nxt[j]]) - d(t[i], t[nxt[i]]) - d(t[j], t[nxt[j]])
    ok = j >= i + 2
    if problem == "cvrp":
        lastdep = torch.where(t == 0, pos, torch.full_like(pos, -1)).cummax(0)[0]
        ok &= lastdep[j] <= i
    else:
        ok &= ~((i == 0) & (j == n - 1))
    return float(g.masked_fill(~ok, float("inf")).min()) if bool(ok.any()) else float("inf")


def _check_invariants(problem, xy, rows, out, length, iters, max_iterations, demand=None):
    from elg_b200 import engine
    rows, out = rows.cpu(), out.cpu()
    assert torch.equal(length.cpu(), engine.tour_length(xy, out.to(DEV)[:, None])[:, 0].cpu())       # bit for bit
    assert (length.cpu() <= engine.tour_length(xy, rows.to(DEV)[:, None])[:, 0].cpu()).all()
    if problem == "tsp":
        assert torch.equal(out.sort(1)[0], rows.sort(1)[0]) and torch.equal(out[:, 0], rows[:, 0])
    else:
        if demand is not None:
            O.check_feasible_cvrp(out[:, None], demand.cpu())
        assert torch.equal(out == 0, rows == 0)                      # depot visits stay where they are
        for a, b in zip(out, rows):
            cut = (b == 0).nonzero().flatten().tolist() + [len(b)]
            for s, e in zip(cut, cut[1:]):
                assert sorted(a[s + 1:e].tolist()) == sorted(b[s + 1:e].tolist())
    xc = xy.cpu()
    for r in range(len(out)):
        if int(iters[r]) < max_iterations:
            assert _min_gain_fp64(problem, xc[r if xc.shape[0] > 1 else 0], out[r]) >= -1e-5


# ------------------------------------------------------------------------------------------------ 1. exact parity

@pytest.mark.parametrize("kind,name,cap", [("tsplib", "eil51", 300), ("tsplib", "a280", 40), ("tsplib", "rat575", 12),
                                           ("tsplib", "pr1002", 6), ("setx", "X-n101-k25", 300), ("setx", "X-n1001-k43", 40)])
def test_rounded_metric_identical_to_oracle(kind, name, cap):
    from elg_b200 import engine
    problem = "cvrp" if kind == "setx" else "tsp"
    xy, rows, _, _ = _lib_rows(kind, name)
    out, length, iters = engine.two_opt(problem, xy, rows, max_iterations=cap, rounding=True)
    ref_t, ref_len, ref_it = _oracle(problem, xy, rows, cap, True)
    assert torch.equal(iters.cpu().long(), ref_it)
    assert torch.equal(out.cpu(), ref_t)
    assert torch.equal(length.cpu(), ref_len)
    assert int(iters.sum()) > 0


# ------------------------------------------------------------------------------------------------ 2. random instances

@pytest.mark.parametrize("problem", ["tsp", "cvrp"])
def test_random_instances_scaled_metric(problem):
    from elg_b200 import engine
    same, total = 0, 0
    for N in (20, 50, 100, 200, 500):
        xy, dem, rows = _greedy_rows(problem, N, 4, seed=N)
        out, length, iters = engine.two_opt(problem, xy, rows, max_iterations=1000)
        _check_invariants(problem, xy, rows, out, length, iters, 1000, dem)
        k = 32 if N <= 100 else (8 if N == 200 else 3)                       # oracle time grows as N^2 per move
        ref_t, _, _ = _oracle(problem, xy[:k], rows[:k], 1000, False)
        same += int((out[:k].cpu() == ref_t).all(1).sum())
        total += k
    assert same >= 0.9 * total, (same, total)


# ------------------------------------------------------------------------------------------------ 3. edges

@pytest.mark.parametrize("N1", [3, 4, 5])
def test_tiny_tsp(N1):
    from elg_b200 import engine
    g = torch.Generator().manual_seed(N1)
    xy = torch.rand(64, N1, 2, generator=g)
    rows = torch.stack([torch.randperm(N1, generator=g) for _ in range(64)])
    out, length, iters = engine.two_opt("tsp", xy.to(DEV), rows.to(DEV))
    ref_t, ref_len, ref_it = TO.two_opt("tsp", xy, rows, 1000)
    assert torch.equal(out.cpu(), ref_t) and torch.equal(iters.cpu().long(), ref_it) and torch.equal(length.cpu(), ref_len)
    if N1 == 3:
        assert int(iters.sum()) == 0


def test_cvrp_short_routes_padding_and_shared_coordinates():
    from elg_b200 import engine
    g = torch.Generator().manual_seed(3)
    N1 = 11
    xy = torch.rand(1, N1, 2, generator=g)
    rows = []
    for _ in range(40):
        p = (torch.randperm(N1 - 1, generator=g) + 1).tolist()
        rows.append([0, p[0], 0] + p[1:3] + [0] + p[3:4] + [0] + p[4:] + [0])    # routes of 1, 2, 1 and 6 customers
    rows = torch.tensor(rows)
    out, length, iters = engine.two_opt("cvrp", xy.to(DEV), rows.to(DEV))            # Bxy = 1
    ref_t, ref_len, ref_it = TO.two_opt("cvrp", xy, rows, 1000)
    assert torch.equal(out.cpu(), ref_t) and torch.equal(iters.cpu().long(), ref_it) and torch.equal(length.cpu(), ref_len)
    same_xy = engine.two_opt("cvrp", xy.expand(40, -1, -1).to(DEV), rows.to(DEV))      # Bxy = R
    assert all(torch.equal(a, b) for a, b in zip(same_xy, (out, length, iters)))
    inst = torch.zeros(40, dtype=torch.int32, device=DEV)
    by_inst = engine.two_opt("cvrp", torch.cat((torch.rand(1, N1, 2), xy)).to(DEV), rows.to(DEV), inst=inst + 1)
    assert all(torch.equal(a, b) for a, b in zip(by_inst, (out, length, iters)))
    padded = torch.cat((rows, torch.zeros(40, 2 * N1 + 2 - rows.shape[1], dtype=torch.long)), 1)   # t_max > T
    p_out, p_len, p_it = engine.two_opt("cvrp", xy.to(DEV), padded.to(DEV))
    assert torch.equal(p_out[:, :rows.shape[1]], out) and not p_out[:, rows.shape[1]:].any()
    assert torch.equal(p_len, length) and torch.equal(p_it, iters)


def test_many_tours_persistent_loop():
    from elg_b200 import engine
    xy, _, rows = _greedy_rows("tsp", 100, 250, seed=7)                     # 2000 tours, far above the SM count
    out, length, iters = engine.two_opt("tsp", xy, rows)
    _check_invariants("tsp", xy, rows, out, length, iters, 1000)
    parts = [engine.two_opt("tsp", xy[s:s + 100], rows[s:s + 100]) for s in range(0, 2000, 100)]
    assert torch.equal(out, torch.cat([p[0] for p in parts])) and torch.equal(length, torch.cat([p[1] for p in parts]))


@pytest.mark.parametrize("problem", ["tsp", "cvrp"])
def test_largest_instance_against_oracle(problem):
    """N1 = 8192; cvrp rows of the largest length, 2*N1+2, use the most shared memory (about 192 KB)."""
    from elg_b200 import engine
    g = torch.Generator().manual_seed(11)
    N1 = 8192
    xy = torch.rand(1, N1, 2, generator=g)
    if problem == "tsp":
        rows = torch.randperm(N1, generator=g)[None]
        cap = 2
    else:
        p = (torch.randperm(N1 - 1, generator=g) + 1).tolist()
        row = [0]
        for s in range(0, N1 - 1, 20):
            row += p[s:s + 20] + [0]
        rows = torch.tensor(row + [0] * (2 * N1 + 2 - len(row)))[None]
        cap = 30
    out, length, iters = engine.two_opt(problem, xy.to(DEV), rows.to(DEV), max_iterations=cap)
    ref_t, ref_len, ref_it = TO.two_opt(problem, xy, rows, cap)
    assert int(iters[0]) == cap
    assert torch.equal(out.cpu(), ref_t) and torch.equal(length.cpu(), ref_len)


def test_too_many_nodes_fails_loudly():
    from elg_b200 import _lib, engine
    xy = torch.rand(1, 8193, 2, device=DEV)
    with pytest.raises(_lib.ElgError, match="8192"):
        engine.two_opt("tsp", xy, torch.arange(8193, device=DEV)[None])
    with pytest.raises(ValueError):
        engine.two_opt("tsp", xy[:, :10], torch.arange(1, 11, device=DEV)[None])     # node id 10 of 10 nodes


# ------------------------------------------------------------------------------------------------ 4. determinism

@pytest.mark.parametrize("problem", ["tsp", "cvrp"])
def test_deterministic_and_idempotent(problem):
    from elg_b200 import engine
    xy, _, rows = _greedy_rows(problem, 100, 16, seed=5)
    a = engine.two_opt(problem, xy, rows)
    b = engine.two_opt(problem, xy, rows.to(torch.int16))
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert int(a[2].max()) < 1000
    again = engine.two_opt(problem, xy, a[0])
    assert int(again[2].sum()) == 0 and torch.equal(again[0], a[0]) and torch.equal(again[1], a[1])


# ------------------------------------------------------------------------------------------------ 5. drop-in function

@pytest.mark.parametrize("problem", ["tsp", "cvrp"])
def test_batched_two_opt_torch(problem):
    from elg_b200 import engine
    from elg_b200.cvrp import batched_two_opt_torch as cvrp_2opt
    from elg_b200.tsp import batched_two_opt_torch as tsp_2opt
    xy, _, rows = _greedy_rows(problem, 50, 1, seed=9)
    pts, rows = xy[0], rows                                           # augmentation 0 = the instance itself
    want, _, it = engine.two_opt(problem, pts[None], rows, max_iterations=500)
    if problem == "tsp":
        closed = torch.cat((rows, rows[:, :1]), 1)
        want = torch.cat((want, want[:, :1]), 1)
        fn = tsp_2opt
    else:
        closed, fn = rows, cvrp_2opt
    t_np, n_np = fn(pts.cpu().numpy(), closed.cpu().numpy().astype(np.int32), max_iterations=500)
    assert isinstance(t_np, np.ndarray) and t_np.dtype == np.int32 and n_np == int(it.max())
    assert np.array_equal(t_np, want.cpu().numpy())
    t_pt, n_pt = fn(pts, closed, max_iterations=500, device=DEV)
    assert torch.is_tensor(t_pt) and t_pt.device == closed.device and torch.equal(t_pt, want) and n_pt == n_np
    t_cpu, _ = fn(pts.cpu(), closed.cpu(), max_iterations=500)        # torch on the host in, host out
    assert t_cpu.device.type == "cpu" and torch.equal(t_cpu, want.cpu())


# ------------------------------------------------------------------------------------------------ 6. drivers

def test_library_drivers_refine_with_2opt():
    for kind, name in (("tsplib", "eil51"), ("tsplib", "berlin52"), ("setx", "X-n101-k25")):
        problem = "cvrp" if kind == "setx" else "tsp"
        xy, rows, res_off, opt = _lib_rows(kind, name)
        assert not any("2opt" in k or "two_opt" in k for k in res_off)        # key absent: no new fields
        _, rows_on, res, _ = _lib_rows(kind, name, 200)
        assert torch.equal(rows_on, rows) and res["best_cost"] == res_off["best_cost"]
        _, ref_len, ref_it = _oracle(problem, xy, rows, 200, True)
        assert res["best_cost_2opt"] == float(ref_len.min()) <= res["best_cost"]
        assert res["gap_2opt"] == (res["best_cost_2opt"] - opt) / opt
        assert res["two_opt_iterations"] == int(ref_it.sum()) > 0 and res["two_opt_seconds"] > 0


def test_tsplib_driver_prints_and_records(tmp_path, capsys):
    import pickle
    from elg_b200.synth import DEFAULT_MODEL_PARAMS
    from elg_b200.tsp.test_tsplib import TSPLib_Tester
    z = np.load(os.path.join(LIB, "tsplib_inputs.npz"))
    d = tmp_path / "TSPLib"
    d.mkdir()
    for name in ("eil51", "st70"):
        with open(d / (name + ".pkl"), "wb") as f:
            pickle.dump([z[name + "/coord"], float(z[name + "/opt"])], f)
    for iters in (0, 100):
        cfg = {"name": "ELG", "use_cuda": True, "cuda_device_num": 0, "tsplib_path": str(d), "load_checkpoint": None,
               "params": {"aug_factor": 8, "two_opt_iterations": iters}, "model_params": dict(DEFAULT_MODEL_PARAMS["tsp"])}
        from elg_b200.tsp import TSPModel
        m = TSPModel(**cfg["model_params"])
        m.decoder.add_local_policy(DEV)
        from elg_b200.synth import synthetic_state_dict
        m.load_state_dict(synthetic_state_dict("tsp", seed=3, gain=3.0))
        random.seed(1)
        results = TSPLib_Tester(cfg, model=m).test_on_tsplib(out_dir=str(tmp_path / ("out%d" % iters)))
        out = capsys.readouterr().out
        recs = [r["record"][0] for r in results]
        if iters:
            assert out.count("gap after 2-opt") == 2 + 1 + 1 and all(r["best_cost_2opt"] <= r["best_cost"] for r in recs)
        else:
            assert "2-opt" not in out and not any(k in r for r in recs for k in ("best_cost_2opt", "gap_2opt",
                                                                                   "two_opt_seconds", "two_opt_iterations"))


@pytest.mark.parametrize("kind", ["cvrp", "tsp"])
def test_test_py_with_2opt(kind, capsys):
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict, synthetic_tsp_batch
    if kind == "cvrp":
        from elg_b200.cvrp import CVRPEnv as Env, CVRPModel as Model
        from elg_b200.cvrp.test import test
        batch = {k: v.to(DEV) for k, v in synthetic_cvrp_batch(4, 20, seed=8).items()}
    else:
        from elg_b200.tsp import TSPEnv as Env, TSPModel as Model
        from elg_b200.tsp.test import test
        batch = synthetic_tsp_batch(4, 20, seed=8).to(DEV)
    model = Model(**DEFAULT_MODEL_PARAMS[kind])
    model.decoder.add_local_policy(DEV)
    model.load_state_dict(synthetic_state_dict(kind, seed=21, gain=3.0))
    model = model.to(DEV)
    env = Env(20, DEV)
    random.seed(5)
    avg = test([batch], model, env, 8)
    plain = capsys.readouterr().out
    assert "2-opt" not in plain
    random.seed(5)
    avg2 = test([batch], model, env, 8, two_opt_iterations=100)
    out = capsys.readouterr().out
    assert out.startswith(plain.split("Wall-clock")[0]) and float(avg2) == float(avg)
    line = [l for l in out.splitlines() if l.startswith("2-opt Aug cost: ")]
    assert len(line) == 1 and float(line[0].split()[3].rstrip(",")) <= float(avg) + 1e-6
