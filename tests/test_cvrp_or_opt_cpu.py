"""Or-opt moves of the CVRP local search (elg_cvrp_local_search_ex, max_segment 2 and 3) without a GPU: the oracle's
segment moves (tests/cvrp_or_opt_oracle.py, types 4..7) against an enumeration of every segment relocation on the list of
routes, the default max_segment = 1, the argument checks of the C entry point and the engine, and the drivers' key
params.local_search_max_segment."""
import ctypes as C
from collections import Counter
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from elg_b200 import _lib, engine
import cvrp_ls_oracle
import cvrp_or_opt_oracle as LS


def _random_case(seed, N1=12, cap=7):
    """A row of N1 nodes with tight capacities: one-customer routes, doubled depot visits, demands 1..3."""
    g = torch.Generator().manual_seed(seed)
    xy = torch.rand(1, N1, 2, generator=g)
    dem = torch.randint(1, 4, (N1,), generator=g)
    dem[0] = 0
    row, load = [0], 0
    for v in (torch.randperm(N1 - 1, generator=g) + 1).tolist():
        if load + int(dem[v]) > cap or float(torch.rand(1, generator=g)) < 0.25:
            row.append(0)
            load = 0
            if float(torch.rand(1, generator=g)) < 0.3:
                row.append(0)                                    # a doubled depot visit: not canonical
        row.append(v)
        load += int(dem[v])
    L = 2 * N1 + 2
    return xy, dem.numpy(), torch.tensor([row + [0] * (L - len(row))]), cap


def _segment_neighbours(row, dem, cap, max_segment):
    """Every relocation of a chain of 2..max_segment customers of one route, forward or reversed, into any gap of any
    route (the own route after taking the chain out), built on the list of routes.  -> (feasible new rows, number of
    infeasible ones).  The chain put back into its own gap (unchanged, or reversed in place) is left out."""
    L = len(row)
    routes = LS.routes_of(row)
    load = [sum(int(dem[v]) for v in r) for r in routes]
    out, infeasible = [], 0
    for k, route in enumerate(routes):
        for s in range(2, max_segment + 1):
            for c in range(len(route) - s + 1):
                seg = route[c:c + s]
                for m in range(len(routes)):
                    rest = route[:c] + route[c + s:] if m == k else routes[m]
                    for gap in range(len(rest) + 1):
                        if m == k and gap == c:
                            continue
                        for chain in (seg, seg[::-1]):
                            new = [list(r) for r in routes]
                            new[k] = route[:c] + route[c + s:]
                            new[m] = new[m][:gap] + chain + new[m][gap:]
                            if m != k and load[m] + sum(int(dem[v]) for v in seg) > cap:
                                infeasible += 1
                            else:
                                out.append(LS.row_of(new, L))
    return out, infeasible


def _length(D, r):
    return sum(D[r[p], r[(p + 1) % len(r)]] for p in range(len(r)))


@pytest.mark.parametrize("max_segment", [2, 3])
def test_segment_moves_are_exactly_every_segment_relocation(max_segment):
    checked, infeasible_total, emptied = 0, 0, 0
    for seed in range(16):
        xy, dem, rows, cap = _random_case(seed)
        D = LS.edge_matrix(xy[0], False)
        row = LS.canonical(rows[0].tolist(), rows.shape[1])
        base = _length(D, row)
        g = LS.move_gains(D, dem, cap, row, max_segment)
        assert g.shape[0] == 2 + 2 * max_segment
        reached = []
        for t, i, j in zip(*np.nonzero(np.isfinite(g[4:]))):
            new = LS.apply_move(row, len(row), int(t) + 4, int(i), int(j))
            assert abs(g[t + 4, i, j] - (_length(D, new) - base)) < 1e-9
            emptied += len(LS.routes_of(new)) < len(LS.routes_of(row))
            reached.append(tuple(new))
        want, infeasible = _segment_neighbours(row, dem, cap, max_segment)
        assert Counter(reached) == Counter(tuple(r) for r in want)
        checked += len(reached)
        infeasible_total += infeasible
    assert checked > 500 and infeasible_total > 500 and emptied > 20


def test_segment_load_and_key_order():
    """A two-customer route and a route with spare load 2: the pair moves into it only if the pair's load fits; the
    search records segment moves and ties keep relocate (type 1) ahead of the segment types."""
    xy = torch.tensor([[0, 0], [10, 0], [11, 0], [30, 1], [31, 1]], dtype=torch.float32)
    row = [0, 1, 2, 0, 3, 4, 0, 0, 0, 0, 0, 0]
    D = LS.edge_matrix(xy, True)
    for cap, fits in ((4, True), (3, False)):
        g = LS.move_gains(D, np.array([0, 1, 1, 1, 1]), cap, row, 3)
        assert np.isfinite(g[4, 4, 2]) == fits and np.isfinite(g[5, 4, 2]) == fits     # 3 4 after customer 2
        assert (g[6:] == np.inf).all()                                                 # no chain of 3
    out, length, iters, moves = LS.cvrp_local_search(xy[None], torch.tensor([row]), torch.tensor([[0, 1, 1, 1, 1]]), 4,
                                                     10, rounding=True, record_moves=True, max_segment=2)
    assert len(LS.routes_of(out[0].tolist())) == 1 and moves[0][0][0] in (3, 4, 5)


def test_default_is_the_four_move_search():
    """max_segment = 1 evaluates types 0..3 only and gives the results of the four-move oracle (cvrp_ls_oracle)."""
    for seed in range(6):
        xy, dem, rows, cap = _random_case(50 + seed)
        row = LS.canonical(rows[0].tolist(), rows.shape[1])
        D = LS.edge_matrix(xy[0], True)
        assert np.array_equal(LS.move_gains(D, dem, cap, row), LS.move_gains(D, dem, cap, row, 1))
        assert LS.move_gains(D, dem, cap, row).shape[0] == 4
        xy = torch.floor(xy * 20)
        a = LS.cvrp_local_search(xy, rows, torch.tensor(dem)[None], cap, 1000, rounding=True, record_moves=True)
        b = LS.cvrp_local_search(xy, rows, torch.tensor(dem)[None], cap, 1000, rounding=True, record_moves=True,
                                 max_segment=1)
        assert all(torch.equal(x, y) for x, y in zip(a[:3], b[:3])) and a[3] == b[3]
        four = cvrp_ls_oracle.cvrp_local_search(xy, rows, torch.tensor(dem)[None], cap, 1000, rounding=True,
                                                record_moves=True)
        assert all(torch.equal(x, y) for x, y in zip(a[:3], four[:3])) and a[3] == four[3]
        assert np.array_equal(LS.move_gains(D, dem, cap, row), cvrp_ls_oracle.move_gains(D, dem, cap, row))
        assert all(m[0] < 4 for m in a[3][0])
        c = LS.cvrp_local_search(xy, rows, torch.tensor(dem)[None], cap, 1000, rounding=True, max_segment=3)
        assert c[0].shape == a[0].shape


def test_converged_or_opt_output_has_no_improving_segment_move():
    found = 0
    for seed in range(8):
        xy, dem, rows, cap = _random_case(200 + seed)
        out, length, iters, moves = LS.cvrp_local_search(xy, rows, torch.tensor(dem)[None], cap, 1000,
                                                         record_moves=True, max_segment=3)
        row = out[0].tolist()
        D = LS.edge_matrix(xy[0], False)
        assert LS.move_gains(D, dem, cap, row, 3).min() >= -1e-6
        assert all(sum(int(dem[v]) for v in r) <= cap for r in LS.routes_of(row))
        assert sorted(v for r in LS.routes_of(row) for v in r) == list(range(1, xy.shape[1]))
        found += sum(m[0] >= 4 for m in moves[0])
    assert found > 0


# --------------------------------------------------------------------------------------------- argument checks

def test_binding_and_argument_checks():
    lib = _lib.lib
    assert "elg_cvrp_local_search_ex" in _lib.SYMBOLS and _lib.ABI_VERSION == 4
    f = lib.elg_cvrp_local_search_ex
    null = C.c_void_p(0)
    p = C.c_void_p(16)                       # never dereferenced: every call below fails its argument checks
    assert f(p, 1, 10, p, 10, null, p, 1, 22, 0, 0, 10, p, p, null) == -1                 # max_segment 0
    assert f(p, 1, 10, p, 10, null, p, 1, 22, 4, 0, 10, p, p, null) == -1                 # max_segment 4
    assert b"max_segment" in lib.elg_last_error()
    assert f(p, 1, 8193, p, 10, null, p, 1, 100, 3, 0, 10, p, p, null) == -2              # ELG_EUNSUPPORTED
    assert b"8192" in lib.elg_last_error()
    assert f(p, 1, 10, p, 10, null, p, 1, 23, 2, 0, 10, p, p, null) == -1                 # L > 2*N1+2
    assert f(p, 1, 10, p, 0, null, p, 1, 22, 2, 0, 10, p, p, null) == -1                  # capacity 0
    assert f(p, 1, 10, null, 10, null, p, 1, 22, 2, 0, 10, p, p, null) == -1              # NULL demand


def test_engine_rejects_bad_max_segment_before_the_device_checks():
    xy = torch.rand(1, 6, 2)
    dem = torch.tensor([[0, 1, 2, 3, 1, 2]]) / 5.
    rows = torch.tensor([[0, 1, 2, 0, 3, 4, 0, 5, 0, 0]])
    for bad in (0, 4, 1.5, None):
        with pytest.raises(ValueError, match="max_segment"):
            engine.cvrp_local_search(xy, rows, dem, 5, max_segment=bad)
    with pytest.raises(_lib.ElgError):
        engine.cvrp_local_search(xy, rows, dem, 5, max_segment=3)                   # CPU tensors


# --------------------------------------------------------------------------------------------- drivers

def _cfg(**params):
    return {"use_cuda": True, "cuda_device_num": 0, "params": dict(aug_factor=8, **params)}


def test_drivers_accept_and_reject_the_key():
    from elg_b200 import lib_driver as drv
    from elg_b200.cvrp import CVRPModel
    from elg_b200.synth import DEFAULT_MODEL_PARAMS
    from elg_b200.tsp import TSPModel
    for seg in (1, 2, 3):
        drv.reject("cvrp", _cfg(local_search_iterations=10, local_search_max_segment=seg))
    drv.reject("cvrp", _cfg(local_search_iterations=10))
    drv.reject("tsp", _cfg(tsp_local_search_iterations=10))
    for bad in (0, 4, -1):
        with pytest.raises(ValueError, match="1, 2 or 3"):
            drv.reject("cvrp", _cfg(local_search_iterations=10, local_search_max_segment=bad))
    with pytest.raises(ValueError, match="params.local_search_iterations"):
        drv.reject("cvrp", _cfg(local_search_max_segment=2))
    with pytest.raises(ValueError, match="params.local_search_iterations"):
        drv.reject("cvrp", _cfg(local_search_iterations=0, local_search_max_segment=2))
    with pytest.raises(ValueError, match="tsp_local_search_iterations"):
        drv.load_model(TSPModel, _cfg(tsp_local_search_iterations=10, local_search_max_segment=3), "cpu")
    with pytest.raises(ValueError, match="1, 2 or 3"):
        drv.load_model(CVRPModel, _cfg(local_search_iterations=10, local_search_max_segment=5), "cpu")
    m = CVRPModel(**DEFAULT_MODEL_PARAMS["cvrp"])
    m = drv.load_model(CVRPModel, _cfg(local_search_iterations=10, local_search_max_segment=3), "cpu", model=m)
    assert m._elg_local_search_max_segment == 3 and m._elg_stage_iterations["local_search_iterations"] == 10
    m = drv.load_model(CVRPModel, _cfg(local_search_iterations=10), "cpu", model=m)
    assert m._elg_local_search_max_segment == 1


def test_the_key_reaches_the_engine_call(monkeypatch):
    """solve_instance (the library driver) and refine (test.py) pass the setting to engine.cvrp_local_search; the other
    stages do not take it."""
    from elg_b200 import lib_driver as drv
    calls = []

    def fake(xy, rows, demand, capacity, **kw):
        calls.append(kw)
        return rows, torch.full((rows.shape[0],), 7.0), torch.ones(rows.shape[0], dtype=torch.int32)
    monkeypatch.setattr(drv.engine, "cvrp_local_search", fake)
    monkeypatch.setattr(drv.engine, "two_opt", lambda *a, **kw: calls.append(("two_opt", kw)) or fake(a[1], a[2], 0, 0))
    monkeypatch.setattr(drv.torch.cuda, "synchronize", lambda: None)
    sols = torch.tensor([[[0, 1, 2, 0, 3, 0]] * 3] * 8)
    rewards = -torch.arange(24, dtype=torch.float32).reshape(8, 3)
    env = SimpleNamespace(reset=lambda: (None, None, None), unscaled_depot_node_xy=torch.rand(8, 4, 2),
                          depot_node_demand=torch.zeros(8, 4), capacity=10)
    model = SimpleNamespace(pre_forward=lambda s: None, _elg_local_search_max_segment=3,
                            _elg_stage_iterations={"two_opt_iterations": 5, "local_search_iterations": 20})
    cost, _, _ = drv.solve_instance(model, env, lambda m, e, kind: (sols, None, rewards), 8, 3)
    assert cost.local_search == (7.0, cost.local_search[1], 8)
    assert calls[0][0] == "two_opt" and "max_segment" not in calls[0][1]
    assert calls[-1] == {"max_iterations": 20, "rounding": True, "max_segment": 3}
    stage = next(s for s in drv.STAGES if s.key == "local_search_iterations")
    drv.refine(stage, "cvrp", env.unscaled_depot_node_xy, sols, rewards, 8, 30, False, env.depot_node_demand, 10, 2)
    assert calls[-1] == {"max_iterations": 30, "rounding": False, "max_segment": 2}
    drv.refine(stage, "cvrp", env.unscaled_depot_node_xy, sols, rewards, 8, 30, False, env.depot_node_demand, 10)
    assert calls[-1]["max_segment"] == 1
