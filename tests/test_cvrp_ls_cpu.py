"""Capacity-aware CVRP local search without a GPU: the oracle (tests/cvrp_ls_oracle.py) on hand-made cases and against a
brute-force restatement of the contract, the argument checks of elg_cvrp_local_search / engine.cvrp_local_search /
cvrp_local_search, and the drivers' optional stage."""
import ctypes as C
import json
import math

import numpy as np
import pytest
import torch

from elg_b200 import _lib, engine
import cvrp_ls_oracle as LS


def _run(xy, row, dem, cap, iters, rounding=True):
    return LS.cvrp_local_search(torch.tensor(xy, dtype=torch.float32)[None], torch.tensor([row]),
                                torch.tensor([dem]), cap, iters, rounding=rounding, record_moves=True)


# --------------------------------------------------------------------------------------------- hand-made cases

def test_relocate_empties_a_route_and_ties_go_to_the_lowest_key():
    """Customer 3 sits between 1 and 2.  Moving it into route 1 between them, moving it to the end of route 1, and the
    2-opt* that appends route 2 to route 1 all gain exactly -22; the relocate onto edge (1, 2) has the lowest key."""
    xy = [[0, 0], [10, 0], [12, 0], [11, 0]]
    row = [0, 1, 2, 0, 3, 0, 0, 0]
    D = LS.edge_matrix(torch.tensor(xy, dtype=torch.float32), True)
    g = LS.move_gains(D, np.array([0, 1, 1, 1]), 10, row)
    assert g[1, 4, 1] == g[1, 4, 2] == g[3, 2, 3] == -22 == g.min()
    tours, length, iters, moves = _run(xy, row, [0, 1, 1, 1], 10, 1)
    assert moves[0][0] == (1, 4, 1, -22.0)
    assert tours[0].tolist() == [0, 1, 3, 2, 0, 0, 0, 0] and len(LS.routes_of(tours[0])) == 1
    assert float(length[0]) == 24.0


def test_two_opt_star_merges_two_routes():
    xy = [[0, 0], [10, 0], [20, 0], [30, 0], [40, 0]]
    row = [0, 1, 2, 0, 3, 4, 0, 0, 0, 0]
    tours, length, iters, moves = _run(xy, row, [0, 1, 1, 1, 1], 4, 10)
    assert moves[0][0] == (3, 2, 3, -40.0)                      # A + B: the tail of B (all of it) moves behind A
    assert tours[0].tolist() == [0, 1, 2, 3, 4, 0, 0, 0, 0, 0] and float(length[0]) == 80.0
    tours, _, _, moves = _run(xy, row, [0, 1, 1, 1, 1], 3, 10)   # capacity 3: no merge
    assert len(LS.routes_of(tours[0])) == 2 and all(m[0] != 3 or m[3] > -40 for m in moves[0])


def test_swap_and_relocate_blocked_by_capacity():
    """Routes (w1, e2) and (e1, w2) each cross between a west and an east pair.  Swapping e2 and w2, or moving e2 into
    the other route, would help; with capacity 3 the west route (load 4) and the overfull other route are infeasible."""
    xy = [[0, 0], [-10, 1], [-10, -1], [10, 1], [10, -1]]
    dem = np.array([0, 2, 2, 1, 1])
    row = [0, 1, 4, 0, 3, 2, 0, 0]
    D = LS.edge_matrix(torch.tensor(xy, dtype=torch.float32), True)
    loose, tight = LS.move_gains(D, dem, 4, row), LS.move_gains(D, dem, 3, row)
    assert loose[2, 2, 5] < -1e-6 and tight[2, 2, 5] == math.inf
    assert (loose[1, 2, 3:5] < -1e-6).all() and (tight[1, 2, 3:6] == math.inf).all()
    assert _run(xy, row, dem.tolist(), 4, 1)[3][0][0][0] == 2          # the swap is the best move when allowed
    tours, _, _, _ = _run(xy, row, dem.tolist(), 3, 100)
    assert all(sum(dem[v] for v in r) <= 3 for r in LS.routes_of(tours[0]))


def test_zero_iterations_returns_the_canonical_input():
    xy = torch.rand(1, 6, 2, generator=torch.Generator().manual_seed(0))
    row = torch.tensor([[0, 1, 0, 0, 2, 3, 0, 4, 5, 0, 0, 0, 0, 0]])
    tours, length, iters = LS.cvrp_local_search(xy, row, torch.tensor([[0, 1, 1, 1, 1, 1]]), 3, 0)
    assert tours[0].tolist() == [0, 1, 0, 2, 3, 0, 4, 5, 0, 0, 0, 0, 0, 0] and int(iters[0]) == 0
    from oracle import elg_oracle as O
    assert float(length[0]) == float(O.tour_length(xy, tours[None])[0, 0])


# --------------------------------------------------------------------------------------------- brute force

def _random_case(seed, N1=13, cap=10):
    g = torch.Generator().manual_seed(seed)
    xy = torch.rand(1, N1, 2, generator=g)
    dem = torch.randint(1, 5, (N1,), generator=g)
    dem[0] = 0
    row, load = [0], 0
    for v in (torch.randperm(N1 - 1, generator=g) + 1).tolist():
        if load + int(dem[v]) > cap or float(torch.rand(1, generator=g)) < 0.2:
            row.append(0)
            load = 0
            if float(torch.rand(1, generator=g)) < 0.3:
                row.append(0)                                    # a doubled depot visit: not canonical
        row.append(v)
        load += int(dem[v])
    L = 2 * N1 + 2
    return xy, dem, torch.tensor([row + [0] * (L - len(row))]), cap


def _locate(row, p):
    """(route index, offset) of a position of a canonical row: offset 0 is the route's depot visit."""
    k = row[:p + 1].count(0) - 1
    return k, p - max(q for q in range(p + 1) if row[q] == 0)


def _brute_moves(row, dem, cap):
    """Every move of the contract, in key order, as (type, i, j, new canonical row), built on the list of routes and
    kept only if every new route is within capacity."""
    L = len(row)
    P = max(p for p in range(L) if row[p] != 0) + 1
    routes = LS.routes_of(row)
    out = []

    def emit(t, i, j, new_routes):
        if all(sum(int(dem[v]) for v in r) <= cap for r in new_routes):
            out.append((t, i, j, LS.row_of(new_routes, L)))

    for t in range(4):
        for i in range(P):
            ki, oi = _locate(row, i)
            for j in range(P):
                kj, oj = _locate(row, j)
                rs = [list(r) for r in routes]
                if t == 0 and j >= i + 2 and ki == kj:
                    rs[ki][oi:oj] = rs[ki][oi:oj][::-1]
                    emit(t, i, j, rs)
                elif t == 1 and oi > 0 and j not in (i - 1, i):
                    u = rs[ki].pop(oi - 1)
                    rs[kj].insert(oj - 1 if (kj == ki and oj > oi) else oj, u)
                    emit(t, i, j, rs)
                elif t == 2 and i < j and ki != kj and oi > 0 and oj > 0:
                    rs[ki][oi - 1], rs[kj][oj - 1] = rs[kj][oj - 1], rs[ki][oi - 1]
                    emit(t, i, j, rs)
                elif t == 3 and i < j and ki != kj:
                    a, b = rs[ki], rs[kj]
                    rs[ki], rs[kj] = a[:oi] + b[oj:], b[:oj] + a[oi:]
                    emit(t, i, j, rs)
    return out


def _brute_gains(D, row, dem, cap):
    def length(r):
        return sum(D[r[p], r[(p + 1) % len(r)]] for p in range(len(r)))
    base = length(row)
    return [(t, i, j, length(new) - base) for t, i, j, new in _brute_moves(row, dem, cap)]


@pytest.mark.parametrize("rounding", [False, True])
def test_oracle_first_move_matches_brute_force(rounding):
    improving = 0
    for seed in range(12):
        xy, dem, rows, cap = _random_case(seed)
        if rounding:
            xy = torch.floor(xy * 20)
        D = LS.edge_matrix(xy[0], rounding)
        row = LS.canonical(rows[0].tolist(), rows.shape[1])
        gains = _brute_gains(D, row, dem.numpy(), cap)
        best = min(g for _, _, _, g in gains)
        _, _, iters, moves = LS.cvrp_local_search(xy, rows, dem[None], cap, 1, rounding=rounding, record_moves=True)
        if best < -1e-6:
            improving += 1
            t, i, j, g = moves[0][0]
            if rounding:                                          # integer gains: the argmin is exact
                first = next(m for m in gains if m[3] == best)
                assert (t, i, j) == first[:3] and g == best
            else:                                                 # equal gains may differ in the last fp64 bits
                near = [m for m in gains if m[3] <= best + 1e-9]
                assert abs(g - best) < 1e-9 and (t, i, j) == near[0][:3]
        else:
            assert int(iters[0]) == 0
    assert improving >= 10


def test_converged_oracle_output_is_a_local_optimum():
    for seed in range(10):
        xy, dem, rows, cap = _random_case(100 + seed)
        tours, length, iters = LS.cvrp_local_search(xy, rows, dem[None], cap, 1000)
        assert int(iters[0]) > 0
        row = tours[0].tolist()
        assert LS.canonical(row, len(row)) == row
        D = LS.edge_matrix(xy[0], False)
        assert min(g for _, _, _, g in _brute_gains(D, row, dem.numpy(), cap)) >= -1e-6
        assert sorted(v for r in LS.routes_of(row) for v in r) == list(range(1, xy.shape[1]))
        assert all(sum(int(dem[v]) for v in r) <= cap for r in LS.routes_of(row))
        assert len(LS.routes_of(row)) <= len(LS.routes_of(rows[0].tolist()))
        start = LS.closed_length(xy[0], LS.canonical(rows[0].tolist(), rows.shape[1]), False)
        assert float(length[0]) < float(start)


# --------------------------------------------------------------------------------------------- argument checks

def test_binding_and_argument_checks():
    lib = _lib.lib
    assert "elg_cvrp_local_search" in _lib.SYMBOLS and _lib.ABI_VERSION == 4
    f = lib.elg_cvrp_local_search
    null = C.c_void_p(0)
    p = C.c_void_p(16)                       # never dereferenced: every call below fails its argument checks
    assert f(p, 1, 8193, p, 10, null, p, 1, 100, 0, 10, p, p, null) == -2                 # ELG_EUNSUPPORTED
    assert b"8192" in lib.elg_last_error()
    assert f(p, 1, 10, p, 10, null, p, 1, 23, 0, 10, p, p, null) == -1                    # L > 2*N1+2
    assert f(p, 1, 10, p, 0, null, p, 1, 22, 0, 10, p, p, null) == -1                     # capacity 0
    assert f(p, 1, 10, p, 10, null, p, 1, 22, 0, -1, p, p, null) == -1                    # max_iterations < 0
    assert f(p, 1, 10, null, 10, null, p, 1, 22, 0, 10, p, p, null) == -1                 # NULL demand
    assert f(null, 1, 10, p, 10, null, p, 1, 22, 0, 10, p, p, null) == -1                 # NULL xy
    assert f(p, 3, 10, p, 10, null, p, 2, 22, 0, 10, p, p, null) == -1                    # Bxy neither 1 nor R
    assert f(p, 1, 0, p, 10, null, p, 1, 22, 0, 10, p, p, null) == -1                     # N1 = 0


def _valid():
    xy = torch.rand(1, 6, 2)
    dem = torch.tensor([[0, 1, 2, 3, 1, 2]]) / 5.
    return xy, torch.tensor([[0, 1, 2, 0, 3, 4, 0, 5, 0, 0]]), dem


def test_engine_rejects_bad_input():
    xy, rows, dem = _valid()
    with pytest.raises(_lib.ElgError):
        engine.cvrp_local_search(xy, rows, dem, 5)                                      # CPU tensors
    with pytest.raises(ValueError, match="integral"):
        engine.cvrp_local_search(xy, rows, dem + 0.01, 5)
    with pytest.raises(ValueError, match="exactly once"):
        engine.cvrp_local_search(xy, torch.tensor([[0, 1, 2, 0, 3, 3, 0, 5, 0, 0]]), dem, 5)
    with pytest.raises(ValueError, match="exactly once"):
        engine.cvrp_local_search(xy, torch.tensor([[0, 1, 2, 0, 3, 0, 0, 5, 0, 0]]), dem, 5)   # 4 missing
    with pytest.raises(ValueError, match="depot"):
        engine.cvrp_local_search(xy, torch.tensor([[1, 2, 0, 3, 4, 0, 5, 0, 0, 0]]), dem, 5)
    with pytest.raises(ValueError, match="capacity"):
        engine.cvrp_local_search(xy, torch.tensor([[0, 1, 2, 3, 4, 0, 5, 0, 0, 0]]), dem, 5)   # load 7 > 5
    with pytest.raises(ValueError, match="capacity"):
        engine.cvrp_local_search(xy, rows, dem, 0)
    from elg_b200.cvrp import cvrp_local_search
    with pytest.raises(_lib.ElgError):
        cvrp_local_search(xy[0].numpy(), dem[0].numpy(), 5, rows.numpy(), device="cpu")


# --------------------------------------------------------------------------------------------- drivers

def test_library_driver_records_carry_the_local_search_stage(capsys):
    from elg_b200 import lib_driver as drv
    plain, both, ls_only = {}, {}, {}
    drv.fill_record(plain, drv.InstanceCost(110.0), 100, 100.0)
    cost = drv.InstanceCost(110.0)
    cost.two_opt = (104.0, 0.5, 7)
    cost.local_search = (102.0, 0.25, 9)
    drv.fill_record(both, cost, 100, 100.0)
    cost = drv.InstanceCost(110.0)
    cost.local_search = (103.0, 0.25, 5)
    drv.fill_record(ls_only, cost, 300, 100.0)
    assert set(plain) == {"best_cost", "scale", "gap"}
    assert list(both) == ["best_cost", "scale", "gap", "best_cost_2opt", "gap_2opt", "two_opt_seconds",
                          "two_opt_iterations", "best_cost_ls", "gap_ls", "ls_seconds", "ls_iterations"]
    assert both["best_cost_ls"] == 102.0 and abs(both["gap_ls"] - 0.02) < 1e-12
    assert both["ls_seconds"] == 0.25 and both["ls_iterations"] == 9
    assert set(ls_only) == {"best_cost", "scale", "gap", "best_cost_ls", "gap_ls", "ls_seconds", "ls_iterations"}
    json.dumps(both)
    edges = [("<200", 0, 200), ("200-500", 200, 500)]
    bins = drv.gap_bins([{"record": [plain]}], edges)
    assert "gap_ls" not in bins and capsys.readouterr().out == ""
    bins = drv.gap_bins([{"record": [ls_only]}], edges)
    assert "gap_2opt" not in bins and abs(bins["gap_ls"]["200-500"] - 3.0) < 1e-9
    assert capsys.readouterr().out.splitlines() == ["Average gap after local search on subset of 200-500: 3.00%",
                                                    "Average gap after local search total: 3.00%"]
    drv.gap_bins([{"record": [both]}], edges)
    assert capsys.readouterr().out.splitlines() == ["Average gap after 2-opt on subset of <200: 4.00%",
                                                    "Average gap after 2-opt total: 4.00%",
                                                    "Average gap after local search on subset of <200: 2.00%",
                                                    "Average gap after local search total: 2.00%"]


def test_stage_needs_cvrp_and_a_capacity():
    from elg_b200 import lib_driver as drv
    from elg_b200.cvrp.test import test as cvrp_test
    from elg_b200.tsp import TSPModel
    cfg = {"use_cuda": True, "cuda_device_num": 0, "params": {"aug_factor": 8, "local_search_iterations": 10}}
    with pytest.raises(ValueError, match="two_opt_iterations"):
        drv.load_model(TSPModel, cfg, "cpu")                    # what TSPLib_Tester calls
    drv.reject_local_search({"params": {"local_search_iterations": 0}})
    with pytest.raises(ValueError, match="capacity"):
        cvrp_test([], None, None, 8, local_search_iterations=10)
