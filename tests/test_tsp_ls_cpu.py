"""TSP local search with 2-opt and Or-opt moves without a GPU: the oracle (tests/tsp_ls_oracle.py) on hand-made tours and
against a brute force over explicit neighbour permutations, the argument checks of elg_tsp_local_search /
engine.tsp_local_search / tsp.tsp_local_search, and the drivers' optional stage."""
import ctypes as C
import json

import pytest
import torch

from elg_b200 import _lib, engine
import tsp_ls_oracle as LS
import two_opt_oracle as TO


def _run(xy, tour, iters, max_segment=3):
    return LS.tsp_local_search(torch.tensor(xy, dtype=torch.float32)[None], torch.tensor([tour]), iters,
                               max_segment=max_segment, rounding=True, record_moves=True)


def _edges(xy, rounding=True):
    e = TO._seglen(xy[:, None, :] - xy[None, :, :])
    return (torch.round(e) if rounding else e).double()


def _length(D, t):
    return sum(float(D[t[k], t[(k + 1) % len(t)]]) for k in range(len(t)))


def _neighbours(n, max_segment=3):
    """Every admissible move (v, i, j) of the contract in key order, with the new tour as a permutation of positions."""
    for v, (s, rev) in enumerate(LS.VARIANTS):
        if s > max_segment:
            continue
        for i in range(n):
            for j in range(n):
                if v == 0:
                    if j >= i + 2 and not (i == 0 and j == n - 1):
                        yield v, i, j, list(range(i + 1)) + list(range(j, i, -1)) + list(range(j + 1, n))
                    continue
                last = i + s - 1
                if i < 1 or last > n - 1 or i - 1 <= j <= last:
                    continue
                seg = list(range(i, last + 1))[::-1 if rev else 1]
                if j > last:
                    yield v, i, j, list(range(i)) + list(range(last + 1, j + 1)) + seg + list(range(j + 1, n))
                else:
                    yield v, i, j, list(range(j + 1)) + seg + list(range(j + 1, i)) + list(range(last + 1, n))


def _brute(D, t, max_segment=3):
    """[(v, i, j, gain, new tour)] over every neighbour, gains as differences of fp64 closed lengths."""
    base = _length(D, t)
    out = []
    for v, i, j, perm in _neighbours(len(t), max_segment):
        new = [t[p] for p in perm]
        out.append((v, i, j, _length(D, new) - base, new))
    return out


# --------------------------------------------------------------------------------------------- hand-made tours

def test_relocation_improves_a_two_opt_optimal_tour():
    xy = [[2, 4], [7, 6], [9, 6], [5, 7], [8, 9], [2, 9]]
    tour = [0, 5, 3, 4, 2, 1]
    p = torch.tensor(xy, dtype=torch.float32)
    assert LS.best_move(p, tour, 0, rounding=True)[0] == 1.0            # no 2-opt move improves
    assert TO.two_opt("tsp", p[None], torch.tensor([tour]), 10, rounding=True)[2].item() == 0
    tours, length, iters, moves = _run(xy, tour, 1)
    assert moves[0] == [(1, 2, 5, -1.0)]                                # node 3 onto the edge (t_5, t_0) = (1, 0)
    assert tours[0].tolist() == [0, 5, 4, 2, 1, 3]
    assert float(length[0]) == _length(_edges(p), tours[0].tolist()) == _length(_edges(p), tour) - 1


def test_reversed_two_and_three_node_segments():
    xy = [[9, 4], [8, 3], [3, 1], [1, 9], [2, 8], [9, 6], [3, 3]]
    tour = [5, 1, 3, 0, 2, 4, 6]
    _, _, _, moves = _run(xy, tour, 1)
    assert moves[0] == [(3, 3, 6, -18.0)]                               # (0, 2) reversed onto (6, 5)
    assert LS.apply_move(tour, 3, 3, 6) == [5, 1, 3, 4, 6, 2, 0]
    assert _run(xy, tour, 1, max_segment=1)[3][0][0][0] <= 1            # not evaluated with max_segment = 1
    xy = [[3, 4], [5, 0], [9, 2], [2, 8], [0, 3], [0, 0], [4, 7]]
    tour = [3, 6, 4, 5, 1, 0, 2]
    _, _, _, moves = _run(xy, tour, 1)
    assert moves[0] == [(5, 2, 6, -7.0)]                                # (4, 5, 1) reversed onto (2, 3)
    assert LS.apply_move(tour, 5, 2, 6) == [3, 6, 0, 2, 1, 5, 4]


def test_segment_at_the_end_and_insertion_before_position_zero():
    xy = [[6, 9], [0, 8], [7, 7], [3, 2], [7, 7], [2, 7], [3, 3]]
    tour = [5, 0, 3, 2, 1, 4, 6]
    _, _, _, moves = _run(xy, tour, 1)
    assert moves[0] == [(2, 5, 1, -14.0)]                               # segment 5..6 = (4, 6), t_i+s wraps to t_0
    assert LS.apply_move(tour, 2, 5, 1) == [5, 0, 4, 6, 3, 2, 1]
    xy = [[3, 3], [1, 7], [2, 8], [9, 3], [0, 2], [2, 8], [5, 9], [9, 0]]
    tour = [7, 0, 4, 3, 1, 5, 2, 6]
    _, _, _, moves = _run(xy, tour, 1)
    assert moves[0] == [(1, 3, 7, -13.0)]                               # node 3 onto the closing edge (6, 7)
    assert LS.apply_move(tour, 1, 3, 7) == [7, 0, 4, 1, 5, 2, 6, 3]


def test_equal_gains_go_to_the_lowest_key_and_two_opt_comes_first():
    """Swapping t_2 and t_3 is both the 2-opt move (1, 3) and the relocation of t_2 onto (t_3, t_4): v = 0 wins."""
    xy = [[6, 4], [3, 6], [4, 2], [9, 4], [8, 6], [7, 3]]
    tour = [1, 4, 5, 3, 0, 2]
    D = _edges(torch.tensor(xy, dtype=torch.float32))
    gains = {(v, i, j): g for v, i, j, g, _ in _brute(D, tour)}
    best = min(gains.values())
    assert gains[(0, 1, 3)] == gains[(1, 2, 3)] == best == -3.0
    tied = sorted(k for k, g in gains.items() if g == best)
    assert tied[0] == (0, 1, 3) and len(tied) > 1
    assert _run(xy, tour, 1)[3][0] == [(0, 1, 3, -3.0)]


def test_zero_iterations():
    xy = torch.rand(2, 9, 2, generator=torch.Generator().manual_seed(0))
    rows = torch.stack([torch.randperm(9), torch.randperm(9)])
    tours, length, iters = LS.tsp_local_search(xy, rows, 0)
    assert torch.equal(tours, rows) and not iters.any()
    assert torch.equal(length, TO.two_opt("tsp", xy, rows, 0)[1])                 # elg_tour_length's summation order


@pytest.mark.parametrize("rounding", [False, True])
def test_max_segment_zero_is_the_two_opt_oracle(rounding):
    g = torch.Generator().manual_seed(4)
    xy = torch.rand(6, 30, 2, generator=g) * (100 if rounding else 1)
    rows = torch.cat((torch.stack([torch.randperm(30, generator=g) for _ in range(6)]), torch.zeros(6, 3).long()), 1)
    a = LS.tsp_local_search(xy, rows, 1000, max_segment=0, rounding=rounding)
    b = TO.two_opt("tsp", xy, rows, 1000, rounding=rounding)
    assert all(torch.equal(x, y) for x, y in zip(a, b)) and int(a[2].min()) > 0


# --------------------------------------------------------------------------------------------- brute force

@pytest.mark.parametrize("rounding", [False, True])
def test_oracle_first_move_matches_brute_force(rounding):
    improving = 0
    for seed in range(40):
        g = torch.Generator().manual_seed(seed)
        n = 3 + seed % 7                                                # N1 = 3..9
        xy = torch.rand(n, 2, generator=g)
        if rounding:
            xy = torch.floor(xy * 20)
        tour = torch.randperm(n, generator=g).tolist()
        D = _edges(xy, rounding)
        moves = _brute(D, tour)
        for v, i, j, _, new in moves:                                   # list surgery = the explicit permutation
            assert LS.apply_move(tour, v, i, j) == new
        gain, v, i, j = LS.best_move(xy, tour, 3, rounding=rounding)
        if not moves:
            assert gain == float("inf")
            continue
        best = min(m[3] for m in moves)
        if rounding:                                                    # integer gains: the argmin is exact
            assert (v, i, j) == next(m[:3] for m in moves if m[3] == best) and gain == best
        else:                                                           # equal gains may differ in the last fp64 bits
            assert abs(gain - best) < 1e-9 and (v, i, j) == next(m[:3] for m in moves if m[3] <= best + 1e-9)
        improving += best < -1e-6
    assert improving >= 25


def test_converged_oracle_output_is_a_local_optimum():
    for seed in range(10):
        g = torch.Generator().manual_seed(100 + seed)
        xy = torch.rand(1, 9, 2, generator=g)
        rows = torch.randperm(9, generator=g)[None]
        tours, length, iters = LS.tsp_local_search(xy, rows, 1000)
        t = tours[0].tolist()
        assert sorted(t) == list(range(9)) and t[0] == rows[0, 0]
        assert min(m[3] for m in _brute(_edges(xy[0], False), t)) >= -1e-6
        assert LS.best_move(xy[0], t, 3, exact=True)[0] >= -1e-5
        assert int(iters[0]) == 0 or float(length[0]) < float(LS.closed_length(xy[0], rows[0], False))


# --------------------------------------------------------------------------------------------- argument checks

def test_binding_and_argument_checks():
    lib = _lib.lib
    assert "elg_tsp_local_search" in _lib.SYMBOLS and _lib.ABI_VERSION == 4
    f = lib.elg_tsp_local_search
    null = C.c_void_p(0)
    p = C.c_void_p(16)                       # never dereferenced: every call below fails its argument checks
    assert f(p, 1, 8193, null, p, 1, 8193, 3, 0, 10, p, p, null) == -2                  # ELG_EUNSUPPORTED
    assert b"8192" in lib.elg_last_error()
    assert f(p, 1, 10, null, p, 1, 9, 3, 0, 10, p, p, null) == -1                       # L < N1
    assert f(p, 1, 10, null, p, 1, 10, 4, 0, 10, p, p, null) == -1                      # max_segment 4
    assert b"max_segment" in lib.elg_last_error()
    assert f(p, 1, 10, null, p, 1, 10, -1, 0, 10, p, p, null) == -1                     # max_segment -1
    assert f(p, 1, 10, null, p, 1, 10, 3, 0, -1, p, p, null) == -1                      # max_iterations < 0
    assert f(null, 1, 10, null, p, 1, 10, 3, 0, 10, p, p, null) == -1                   # NULL xy
    assert f(p, 3, 10, null, p, 2, 10, 3, 0, 10, p, p, null) == -1                      # Bxy neither 1 nor R
    assert f(p, 1, 0, null, p, 1, 10, 3, 0, 10, p, p, null) == -1                       # N1 = 0


def test_engine_rejects_bad_input():
    xy = torch.rand(1, 6, 2)
    rows = torch.tensor([[0, 3, 1, 5, 2, 4]])
    with pytest.raises(_lib.ElgError):
        engine.tsp_local_search(xy, rows)                                                   # CPU tensors
    with pytest.raises(ValueError, match="max_segment"):
        engine.tsp_local_search(xy, rows, max_segment=4)
    with pytest.raises(ValueError, match="max_segment"):
        engine.tsp_local_search(xy, rows, max_segment=-1)
    with pytest.raises(ValueError, match="max_iterations"):
        engine.tsp_local_search(xy, rows, max_iterations=-1)
    with pytest.raises(ValueError, match="permutation"):
        engine.tsp_local_search(xy, torch.tensor([[0, 3, 1, 5, 2, 2]]))
    with pytest.raises(ValueError, match=r"\[0, 6\)"):
        engine.tsp_local_search(xy, torch.tensor([[0, 3, 1, 5, 2, 6]]))
    with pytest.raises(ValueError):
        engine.tsp_local_search(xy, rows[:, :5])                                            # L < N1
    with pytest.raises(ValueError):
        engine.tsp_local_search(xy[0], rows)                                                # xy not (Bxy, N1, 2)
    with pytest.raises(ValueError, match="inst"):
        engine.tsp_local_search(xy, rows, inst=torch.tensor([1]))
    with pytest.raises(ValueError, match="inst"):
        engine.tsp_local_search(xy.expand(3, -1, -1), rows.expand(2, -1))                   # Bxy neither 1 nor R
    from elg_b200.tsp import tsp_local_search
    with pytest.raises(_lib.ElgError, match="tsp_local_search"):
        tsp_local_search(xy[0].numpy(), torch.cat((rows, rows[:, :1]), 1).numpy(), device="cpu")


# --------------------------------------------------------------------------------------------- drivers

def _records():
    from elg_b200 import lib_driver as drv
    plain, both, ls_only = {}, {}, {}
    drv.fill_record(plain, drv.InstanceCost(110.0), 100, 100.0)
    cost = drv.InstanceCost(110.0)
    cost.two_opt = (104.0, 0.5, 7)
    cost.tsp_local_search = (102.0, 0.25, 9)
    drv.fill_record(both, cost, 100, 100.0)
    cost = drv.InstanceCost(110.0)
    cost.tsp_local_search = (103.0, 0.25, 5)
    drv.fill_record(ls_only, cost, 300, 100.0)
    return plain, both, ls_only


def test_library_driver_records_carry_the_tsp_local_search_stage(capsys):
    from elg_b200 import lib_driver as drv
    plain, both, ls_only = _records()
    assert set(plain) == {"best_cost", "scale", "gap"}
    assert list(both) == ["best_cost", "scale", "gap", "best_cost_2opt", "gap_2opt", "two_opt_seconds",
                          "two_opt_iterations", "best_cost_tsp_ls", "gap_tsp_ls", "tsp_ls_seconds", "tsp_ls_iterations"]
    assert both["best_cost_tsp_ls"] == 102.0 and abs(both["gap_tsp_ls"] - 0.02) < 1e-12
    assert both["tsp_ls_seconds"] == 0.25 and both["tsp_ls_iterations"] == 9
    assert set(ls_only) == {"best_cost", "scale", "gap", "best_cost_tsp_ls", "gap_tsp_ls", "tsp_ls_seconds",
                            "tsp_ls_iterations"}
    json.dumps(both)
    edges = [("<200", 0, 200), ("200-500", 200, 500)]
    bins = drv.gap_bins([{"record": [plain]}], edges)
    assert "gap_tsp_ls" not in bins and capsys.readouterr().out == ""
    bins = drv.gap_bins([{"record": [ls_only]}], edges)
    assert "gap_2opt" not in bins and abs(bins["gap_tsp_ls"]["200-500"] - 3.0) < 1e-9
    assert capsys.readouterr().out.splitlines() == ["Average gap after 2-opt + or-opt on subset of 200-500: 3.00%",
                                                    "Average gap after 2-opt + or-opt total: 3.00%"]
    drv.gap_bins([{"record": [both]}], edges)
    assert capsys.readouterr().out.splitlines() == ["Average gap after 2-opt on subset of <200: 4.00%",
                                                    "Average gap after 2-opt total: 4.00%",
                                                    "Average gap after 2-opt + or-opt on subset of <200: 2.00%",
                                                    "Average gap after 2-opt + or-opt total: 2.00%"]


def test_run_set_prints_the_stage_after_two_opt(monkeypatch, capsys):
    from elg_b200 import lib_driver as drv
    monkeypatch.setattr(drv.torch.cuda, "synchronize", lambda: None)
    plain, both, _ = _records()

    def solve(rec):
        return lambda name, payload, record: record.update(rec)
    drv.run_set([("a", 100.0, None)], solve(plain))
    assert capsys.readouterr().out.splitlines() == ["Instance Name a: gap 0.1000"]
    drv.run_set([("b", 100.0, None)], solve(both))
    assert capsys.readouterr().out.splitlines() == ["Instance Name b: gap 0.1000", "Instance Name b: gap after 2-opt 0.0400",
                                                    "Instance Name b: gap after 2-opt + or-opt 0.0200"]


def test_cvrp_models_reject_the_key():
    from elg_b200 import lib_driver as drv
    from elg_b200.cvrp import CVRPModel
    from elg_b200.tsp import TSPModel
    cfg = {"use_cuda": True, "cuda_device_num": 0, "params": {"aug_factor": 8, "tsp_local_search_iterations": 10}}
    with pytest.raises(ValueError, match="local_search_iterations"):
        drv.load_model(CVRPModel, cfg, "cpu")                   # what VRPLib_Tester calls
    with pytest.raises(ValueError, match="params.local_search_iterations"):
        drv.reject_tsp_local_search(cfg)                        # cvrp/test.py
    drv.reject_tsp_local_search({"params": {"tsp_local_search_iterations": 0}})
    drv.reject_tsp_local_search({"params": {}})
    cfg["params"]["local_search_iterations"] = 10               # the TSP rejection of the CVRP key is unchanged
    with pytest.raises(ValueError, match="two_opt_iterations"):
        drv.load_model(TSPModel, cfg, "cpu")
