"""Capacity-aware CVRP local search on the GPU (elg_cvrp_local_search, engine.cvrp_local_search, cvrp_local_search, the
drivers' opt-in stage) against the CPU oracle (tests/cvrp_ls_oracle.py).

Under the rounded library metric every edge is an integer, so gains are exact in fp32 and fp64 alike and the kernel must
make the oracle's moves exactly.  Under the scaled metric the kernel's fp32 gains can order near-ties differently from
the oracle's fp64 gains, so there only the invariants are exact."""
import json
import os
import random

import numpy as np
import pytest
import torch

import cvrp_ls_oracle as LS

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "tests", "golden", "lib")


def _cfg(ls_iterations=None):
    from elg_b200.synth import DEFAULT_MODEL_PARAMS
    cfg = {"name": "ELG", "use_cuda": True, "cuda_device_num": 0, "vrplib_set": "X", "load_checkpoint": None,
           "params": {"aug_factor": 8}, "model_params": dict(DEFAULT_MODEL_PARAMS["cvrp"])}
    if ls_iterations is not None:
        cfg["params"]["local_search_iterations"] = ls_iterations
    return cfg


def _model(wseed, gain):
    from elg_b200.cvrp import CVRPModel
    from elg_b200.synth import synthetic_state_dict
    m = CVRPModel(**_cfg()["model_params"])
    m.decoder.add_local_policy(DEV)
    m.load_state_dict(synthetic_state_dict("cvrp", seed=wseed, gain=gain))
    return m


def _setx_rows(name):
    """Greedy rollout of one Set-X instance through its driver -> (unscaled xy x8 (8, N1, 2), normalised demand (8, N1),
    integer capacity, best rows (8, L))."""
    from elg_b200 import engine
    from elg_b200.cvrp.test_vrplib import VRPLib_Tester
    with open(os.path.join(LIB, "setx_ref.json")) as f:
        ref = json.load(f)
    z = np.load(os.path.join(LIB, "setx_inputs.npz"))
    tester = VRPLib_Tester(_cfg(), model=_model(ref["wseed"], ref["gain"]))
    cap, opt = z[name + "/capopt"]
    inst = {"node_coord": z[name + "/coord"].astype(np.float64), "demand": z[name + "/demand"].astype(np.float64),
            "capacity": float(cap), "depot": np.array([0])}
    random.seed(ref["seed"])
    sols, rewards = tester.test_on_one_ins(name=name, result_dict={}, instance=inst, solution=float(opt))
    c = torch.tensor(z[name + "/coord"], dtype=torch.float32)[None].to(DEV)
    dem = torch.tensor(z[name + "/demand"], dtype=torch.float32)[None].to(DEV) / float(cap)
    xy, dem = engine.load_problems("cvrp", c[:, 1:], c[:, 0], dem[:, 1:], aug=8)
    return xy, dem, int(cap), sols[torch.arange(8, device=DEV), rewards.argmax(1)]


def _greedy_rows(N, n, seed):
    """Greedy rollout of n random CVRP instances x 8 -> (xy, normalised demand, integer capacity, best rows)."""
    from elg_b200 import engine
    from elg_b200.synth import synthetic_cvrp_batch
    cap = {100: 50, 1000: 250}[N]
    b = synthetic_cvrp_batch(n, N, seed=seed, capacity=float(cap))
    xy, dem = engine.load_problems("cvrp", b["loc"].to(DEV), b["depot"].to(DEV), b["demand"].to(DEV), aug=8)
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    h = engine.ModelHandle("cvrp", DEFAULT_MODEL_PARAMS["cvrp"], synthetic_state_dict("cvrp", seed=1234, gain=3.0), DEV)
    tours16, reward, _, n_steps = engine.rollout(engine.encode(h, xy, dem), N, random.Random(seed).sample(range(N), N))
    rows = tours16[torch.arange(xy.shape[0], device=DEV), reward.argmax(1), :int(n_steps.max())].long()
    return xy, dem, cap, rows


def _oracle(xy, dem, cap, rows, max_iterations, rounding):
    units = torch.round(dem.double().cpu() * cap).long()
    return LS.cvrp_local_search(xy.cpu(), rows.cpu(), units, cap, max_iterations, rounding)


def _check_invariants(xy, dem, rows, out, length, rounding=False):
    from elg_b200 import engine
    from elg_b200.cvrp import check_feasible
    rows, out = rows.cpu(), out.cpu()
    assert torch.equal(length.cpu(), engine.tour_length(xy, out.to(DEV)[:, None], rounding)[:, 0].cpu())   # bit for bit
    before = engine.tour_length(xy, rows.to(DEV)[:, None], rounding)[:, 0].cpu()
    assert (length.cpu() <= before).all()
    for r in range(len(out)):
        row = out[r].tolist()
        assert LS.canonical(row, len(row)) == row
        assert len(LS.routes_of(row)) <= len(LS.routes_of(rows[r].tolist()))
        check_feasible(out[r][None, None].to(DEV), dem[r if dem.shape[0] > 1 else 0][None, 1:])


# ------------------------------------------------------------------------------------------------ 1. exact parity

@pytest.mark.parametrize("name,rows_used,cap", [("X-n101-k25", 8, 1000), ("X-n200-k36", 8, 1000),
                                                ("X-n298-k31", 3, 1000), ("X-n1001-k43", 2, 6)])
def test_rounded_metric_identical_to_oracle(name, rows_used, cap):
    from elg_b200 import engine
    xy, dem, capacity, rows = _setx_rows(name)
    xy, dem, rows = xy[:rows_used], dem[:rows_used], rows[:rows_used]
    out, length, iters = engine.cvrp_local_search(xy, rows, dem, capacity, max_iterations=cap, rounding=True)
    ref_t, ref_len, ref_it = _oracle(xy, dem, capacity, rows, cap, True)
    assert torch.equal(iters.cpu().long(), ref_it)
    assert torch.equal(out.cpu(), ref_t)
    assert torch.equal(length.cpu(), ref_len)
    assert int(iters.min()) > 0
    if cap < 1000:
        assert int(iters.min()) == cap


def test_small_random_rows_identical_to_oracle():
    """Integer coordinates and the rounded metric: doubled depot visits, one-customer routes, tight capacities."""
    from elg_b200 import engine
    g = torch.Generator().manual_seed(5)
    N1, R, cap = 13, 64, 10
    xy = torch.floor(torch.rand(R, N1, 2, generator=g) * 30)
    units = torch.randint(1, 5, (R, N1), generator=g)
    units[:, 0] = 0
    rows = []
    for r in range(R):
        row, load = [0], 0
        for v in (torch.randperm(N1 - 1, generator=g) + 1).tolist():
            if load + int(units[r, v]) > cap or float(torch.rand(1, generator=g)) < 0.3:
                row += [0] * (1 + int(len(row) < 10 and float(torch.rand(1, generator=g)) < 0.3))   # L = 2*N1+2 holds
                load = 0
            row.append(v)
            load += int(units[r, v])
        rows.append(row + [0] * (2 * N1 + 2 - len(row)))
    rows = torch.tensor(rows)
    out, length, iters = engine.cvrp_local_search(xy.to(DEV), rows.to(DEV), (units.float() / cap).to(DEV), cap,
                                                  rounding=True)
    ref_t, ref_len, ref_it = LS.cvrp_local_search(xy, rows, units, cap, 1000, True)
    assert torch.equal(out.cpu(), ref_t) and torch.equal(iters.cpu().long(), ref_it) and torch.equal(length.cpu(), ref_len)
    assert int(iters.sum()) > 0


# ------------------------------------------------------------------------------------------------ 2. random instances

@pytest.mark.parametrize("N,n", [(100, 4), (1000, 1)])
def test_random_instances_scaled_metric(N, n):
    from elg_b200 import engine
    xy, dem, cap, rows = _greedy_rows(N, n, seed=N)
    out, length, iters = engine.cvrp_local_search(xy, rows, dem, cap, max_iterations=1000)
    _check_invariants(xy, dem, rows, out, length)
    assert int(iters.min()) > 0
    two = engine.two_opt("cvrp", xy, rows, max_iterations=1000)[1]
    assert float(length.mean()) < float(two.mean())          # moves between routes beat 2-opt inside them


# ------------------------------------------------------------------------------------------------ 3. edges

def test_largest_rows_one_customer_per_route():
    """N1 = 8192 and L = 2*N1+2 with one customer per route: the shared-memory worst case (224 KB)."""
    from elg_b200 import engine
    g = torch.Generator().manual_seed(11)
    N1 = 8192
    xy = torch.rand(1, N1, 2, generator=g)
    units = torch.randint(1, 10, (1, N1), generator=g)
    units[:, 0] = 0
    row = [0]
    for v in (torch.randperm(N1 - 1, generator=g) + 1).tolist():
        row += [v, 0]
    rows = torch.tensor(row + [0] * (2 * N1 + 2 - len(row)))[None]
    dem = (units.float() / 100).to(DEV)
    out, length, iters = engine.cvrp_local_search(xy.to(DEV), rows.to(DEV), dem, 100, max_iterations=2)
    assert int(iters[0]) == 2
    _check_invariants(xy.to(DEV), dem, rows, out, length)
    assert len(LS.routes_of(out[0].tolist())) == N1 - 3          # every improving move here merges two routes


def test_one_customer_and_local_optimum():
    from elg_b200 import engine
    xy = torch.tensor([[[0.0, 0.0], [3.0, 4.0]]], device=DEV)
    rows = torch.tensor([[0, 0, 1, 0, 0, 0]], device=DEV)
    out, length, iters = engine.cvrp_local_search(xy, rows, torch.tensor([[0.0, 0.5]], device=DEV), 2)
    assert out.tolist() == [[0, 1, 0, 0, 0, 0]] and int(iters[0]) == 0 and float(length[0]) == 10.0
    xy, dem, cap, rows = _greedy_rows(100, 2, seed=3)
    a = engine.cvrp_local_search(xy, rows, dem, cap)
    again = engine.cvrp_local_search(xy, a[0], dem, cap)
    assert int(again[2].sum()) == 0 and torch.equal(again[0], a[0]) and torch.equal(again[1], a[1])


def test_inst_mapping_shared_instance_and_determinism():
    from elg_b200 import engine
    xy, dem, cap, rows = _greedy_rows(100, 2, seed=4)          # 16 rows over 16 aug-instances
    a = engine.cvrp_local_search(xy, rows, dem, cap)
    b = engine.cvrp_local_search(xy, rows.to(torch.int16), dem, cap)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    inst = torch.arange(16, device=DEV).flip(0)
    by_inst = engine.cvrp_local_search(xy.flip(0), rows, dem.flip(0), cap, inst=inst)
    assert all(torch.equal(x, y) for x, y in zip(a, by_inst))
    one = engine.cvrp_local_search(xy[:1], rows[:1].expand(5, -1), dem[:1], cap)        # Bxy = 1
    assert all(torch.equal(x, y[:1].expand_as(x)) for x, y in zip(one, a))


def test_too_many_nodes_fails_loudly():
    from elg_b200 import _lib, engine
    xy = torch.rand(1, 8193, 2, device=DEV)
    dem = torch.zeros(1, 8193, device=DEV)
    row = torch.cat((torch.zeros(1, dtype=torch.long), torch.arange(1, 8193)))[None].to(DEV)
    with pytest.raises(_lib.ElgError, match="8192"):
        engine.cvrp_local_search(xy, row, dem, 10)


# ------------------------------------------------------------------------------------------------ 4. drop-in function

def test_cvrp_local_search_drop_in():
    from elg_b200 import engine
    from elg_b200.cvrp import cvrp_local_search
    xy, dem, cap, rows = _greedy_rows(100, 1, seed=9)
    pts, d, rows = xy[0], dem[0], rows[:1]
    want, _, it = engine.cvrp_local_search(pts[None], rows, d[None], cap, max_iterations=500)
    t_np, n_np = cvrp_local_search(pts.cpu().numpy(), d.cpu().numpy(), cap, rows.cpu().numpy().astype(np.int32),
                                   max_iterations=500)
    assert isinstance(t_np, np.ndarray) and t_np.dtype == np.int32 and n_np == int(it.max()) > 0
    assert np.array_equal(t_np, want.cpu().numpy())
    t_pt, n_pt = cvrp_local_search(pts, d, cap, rows, max_iterations=500, device=DEV)
    assert torch.is_tensor(t_pt) and t_pt.device == rows.device and torch.equal(t_pt, want) and n_pt == n_np
    t_cpu, _ = cvrp_local_search(pts.cpu(), d.cpu(), cap, rows.cpu(), max_iterations=500)
    assert t_cpu.device.type == "cpu" and torch.equal(t_cpu, want.cpu())
    with pytest.raises(ValueError):
        cvrp_local_search(pts, d + 0.003, cap, rows)                             # not whole units
    with pytest.raises(ValueError):
        cvrp_local_search(pts, d, cap, torch.zeros_like(rows))                     # no customer visited
    with pytest.raises(ValueError):
        cvrp_local_search(pts, d * 2, cap // 2, rows)                              # same units, half the capacity


# ------------------------------------------------------------------------------------------------ 5. drivers

def test_vrplib_driver_with_the_stage(tmp_path, capsys):
    from elg_b200.cvrp.test_vrplib import VRPLib_Tester
    out = {}
    for iters in (None, 300):
        cfg = _cfg(iters)
        cfg["vrplib_path"] = os.path.join(ROOT, "tests", "golden", "vrplib")
        random.seed(1)
        results = VRPLib_Tester(cfg, model=_model(3, 3.0)).test_on_vrplib(out_dir=str(tmp_path / str(iters)))
        out[iters] = (capsys.readouterr().out, [r["record"][0] for r in results[:-1]])
    plain, recs = out[None]
    assert "local search" not in plain and not any(k.endswith("_ls") or k.startswith("ls_") for r in recs for k in r)
    text, recs_on = out[300]
    assert [r["best_cost"] for r in recs_on] == [r["best_cost"] for r in recs]
    for r in recs_on:
        assert r["gap_ls"] <= r["gap"] and r["best_cost_ls"] <= r["best_cost"] and r["ls_iterations"] > 0
        assert r["ls_seconds"] > 0
    lines = text.splitlines()
    assert sum(l.startswith("Instance Name ") and "gap after local search" in l for l in lines) == 2
    assert sum(l.startswith("Average gap after local search on subset of ") for l in lines) == \
        sum(l.startswith("Average gap on subset of ") for l in lines) >= 1
    assert sum(l.startswith("Average gap after local search total: ") for l in lines) == 1
    assert [l for l in lines if "local search" not in l][:4] == plain.splitlines()[:4]


def test_test_py_with_the_stage(capsys):
    from elg_b200.cvrp import CVRPEnv
    from elg_b200.cvrp.test import test
    from elg_b200.synth import synthetic_cvrp_batch
    batch = {k: v.to(DEV) for k, v in synthetic_cvrp_batch(4, 20, seed=8, capacity=30.).items()}
    model = _model(21, 3.0).to(DEV)
    env = CVRPEnv(20, DEV)
    random.seed(5)
    avg = test([batch], model, env, 8)
    plain = capsys.readouterr().out
    random.seed(5)
    avg2 = test([batch], model, env, 8, local_search_iterations=100, capacity=30)
    out = capsys.readouterr().out
    assert "local search" not in plain and out.startswith(plain.split("Wall-clock")[0]) and float(avg2) == float(avg)
    line = [l for l in out.splitlines() if l.startswith("local search Aug cost: ")]
    assert len(line) == 1 and float(line[0].split()[4].rstrip(",")) <= float(avg) + 1e-6
