"""2-opt local search without a GPU: the oracle (tests/two_opt_oracle.py) on hand-made cases and against a brute-force
restatement of the contract, and the argument checks of elg_two_opt / engine.two_opt / batched_two_opt_torch."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from elg_b200 import _lib, engine
import two_opt_oracle as TO
from oracle import elg_oracle as O


def test_crossed_square_is_untangled_in_one_move():
    xy = torch.tensor([[[0., 0.], [1., 1.], [1., 0.], [0., 1.]]])
    tours, length, iters, moves = TO.two_opt("tsp", xy, torch.tensor([[0, 1, 2, 3]]), 100, record_moves=True)
    assert tours.tolist() == [[0, 2, 1, 3]] and int(iters[0]) == 1
    assert moves[0][0][:2] == (0, 2) and abs(moves[0][0][2] - (2 - 2 * math.sqrt(2))) < 1e-6
    assert float(length[0]) == 4.0


def test_convex_polygon_in_order_is_left_alone():
    a = torch.arange(12, dtype=torch.float32) * (2 * math.pi / 12)
    xy = torch.stack((torch.cos(a), torch.sin(a)), -1)[None]
    t = torch.arange(12)[None]
    tours, length, iters = TO.two_opt("tsp", xy, t, 100)
    assert int(iters[0]) == 0 and torch.equal(tours, t)
    assert abs(float(length[0]) - 24 * math.sin(math.pi / 12)) < 1e-5


def test_zero_iterations_returns_the_input():
    g = torch.Generator().manual_seed(0)
    xy = torch.rand(1, 30, 2, generator=g)
    t = torch.randperm(30, generator=g)[None]
    tours, _, iters = TO.two_opt("tsp", xy, t, 0)
    assert torch.equal(tours, t) and int(iters[0]) == 0


def _brute_first_move(kind, xy, t, rounding):
    """Every admissible pair in (i, j) order, fp32 edges, fp64 gains; -> (i, j, gain) of the lowest-index minimum, count."""
    n = len(t)
    p = xy[0]

    def d(a, b):
        e = float(((p[a] - p[b]) ** 2).sum().sqrt())
        return float(round(e)) if rounding else e      # python round: half to even, as torch.round / rintf
    best, arg, count = math.inf, None, 0
    for i in range(n):
        for j in range(i + 2, n):
            if kind == "tsp" and i == 0 and j == n - 1:
                continue
            if kind == "cvrp" and any(int(t[k]) == 0 for k in range(i + 1, j + 1)):
                continue
            j1 = (j + 1) % n
            g = d(t[i], t[j]) + d(t[i + 1], t[j1]) - d(t[i], t[i + 1]) - d(t[j], t[j1])
            if g < best:
                best, arg, count = g, (i, j), 1
            elif g == best:
                count += 1
    return arg, best, count


def test_ties_go_to_the_lowest_pair():
    """Small integer coordinates with rounded edges: many exactly equal gains."""
    seen_tie = False
    for seed in range(40):
        g = torch.Generator().manual_seed(seed)
        xy = torch.randint(0, 6, (1, 9, 2), generator=g).float()
        t = torch.randperm(9, generator=g)
        (i, j), best, count = _brute_first_move("tsp", xy, t, True)
        _, _, iters, moves = TO.two_opt("tsp", xy, t[None], 1, rounding=True, record_moves=True)
        if best < -1e-6:
            assert moves[0][0][:2] == (i, j) and moves[0][0][2] == best
            seen_tie |= count > 1
        else:
            assert int(iters[0]) == 0
    assert seen_tie


def test_crossing_inside_a_cvrp_route_is_removed():
    xy = torch.tensor([[[0., 0.], [0., 1.], [1., 0.], [1., 1.]]])
    t = torch.tensor([[0, 1, 2, 3, 0, 0, 0]])                 # one route, crossed, then padding
    tours, length, iters = TO.two_opt("cvrp", xy, t, 100)
    assert int(iters[0]) == 1 and float(length[0]) == 4.0
    assert tours[0, 4:].tolist() == [0, 0, 0] and sorted(tours[0, 1:4].tolist()) == [1, 2, 3]


def _routes(row):
    out, cur = [], []
    for v in row.tolist():
        if v == 0:
            if cur:
                out.append(cur)
            cur = []
        else:
            cur.append(v)
    return out + ([cur] if cur else [])


def test_moves_never_cross_cvrp_routes():
    """Random routes: reversing across a depot visit would shorten these tours, the CVRP search never does it."""
    for seed in range(6):
        g = torch.Generator().manual_seed(seed)
        N = 24
        xy = torch.rand(1, N + 1, 2, generator=g)
        perm = (torch.randperm(N, generator=g) + 1).tolist()
        row, k = [0], 0
        while k < N:
            s = int(torch.randint(1, 6, (1,), generator=g))
            row += perm[k:k + s] + [0]
            k += s
        t = torch.tensor(row + [0] * 3)[None]
        _, cross_best, _ = _brute_first_move("tsp", xy, t[0], False)
        assert cross_best < -1e-6                                # an unconstrained move would help
        tours, length, iters = TO.two_opt("cvrp", xy, t, 1000)
        assert [sorted(r) for r in _routes(tours[0])] == [sorted(r) for r in _routes(t[0])]
        assert (tours[0] == 0).nonzero().flatten().tolist() == (t[0] == 0).nonzero().flatten().tolist()
        assert float(length[0]) <= float(O.tour_length(xy, t[None])[0, 0])
        _, best, _ = _brute_first_move("cvrp", xy, tours[0], False)
        assert best >= -1e-6                                     # converged under the route constraint
        dem = torch.full((1, N + 1), 1.0 / 6); dem[0, 0] = 0
        O.check_feasible_cvrp(tours[None], dem)


@pytest.mark.parametrize("kind", ["tsp", "cvrp"])
def test_oracle_first_move_matches_brute_force(kind):
    for seed in range(10):
        g = torch.Generator().manual_seed(100 + seed)
        N1 = 12
        xy = torch.rand(1, N1, 2, generator=g)
        if kind == "tsp":
            t = torch.randperm(N1, generator=g)
        else:
            p = (torch.randperm(N1 - 1, generator=g) + 1).tolist()
            t = torch.tensor([0] + p[:4] + [0] + p[4:9] + [0] + p[9:] + [0, 0])
        arg, best, _ = _brute_first_move(kind, xy, t, False)
        _, _, iters, moves = TO.two_opt(kind, xy, t[None], 1, record_moves=True)
        if best < -1e-6:
            assert moves[0][0][:2] == arg and abs(moves[0][0][2] - best) < 1e-12
        else:
            assert int(iters[0]) == 0


def test_binding_and_argument_checks():
    lib = _lib.lib
    assert "elg_two_opt" in _lib.SYMBOLS and _lib.ABI_VERSION == 4
    null = C.c_void_p(0)
    p = C.c_void_p(16)                       # never dereferenced: every call below fails its argument checks
    assert lib.elg_two_opt(0, p, 1, 8193, null, p, 1, 8193, 0, 10, p, p, null) == -2      # ELG_EUNSUPPORTED
    assert b"8192" in lib.elg_last_error()
    assert lib.elg_two_opt(1, p, 1, 10, null, p, 1, 23, 0, 10, p, p, null) == -1          # cvrp L > 2*N1+2
    assert lib.elg_two_opt(0, p, 1, 10, null, p, 1, 9, 0, 10, p, p, null) == -1           # tsp L < N1
    assert lib.elg_two_opt(0, p, 1, 10, null, p, 1, 10, 0, -1, p, p, null) == -1          # max_iterations < 0
    assert lib.elg_two_opt(0, null, 1, 10, null, p, 1, 10, 0, 10, p, p, null) == -1       # NULL xy
    assert lib.elg_two_opt(0, p, 3, 10, null, p, 2, 10, 0, 10, p, p, null) == -1          # Bxy neither 1 nor R
    assert lib.elg_two_opt(2, p, 1, 10, null, p, 1, 10, 0, 10, p, p, null) == -1          # unknown problem


def test_engine_and_drop_in_reject_the_cpu():
    xy = torch.rand(1, 10, 2)
    with pytest.raises(_lib.ElgError):
        engine.two_opt("tsp", xy, torch.arange(10)[None])
    with pytest.raises(ValueError, match="inst"):                                    # Bxy neither 1 nor R, before the
        engine.two_opt("tsp", xy.expand(3, -1, -1), torch.arange(10).expand(2, -1))  # device check
    from elg_b200.cvrp import batched_two_opt_torch as cvrp_2opt
    from elg_b200.tsp import batched_two_opt_torch as tsp_2opt
    with pytest.raises(_lib.ElgError):
        tsp_2opt(np.random.rand(10, 2), np.append(np.arange(10), 0)[None], device="cpu")
    with pytest.raises(_lib.ElgError):
        cvrp_2opt(np.random.rand(10, 2), np.array([[0, 1, 2, 0, 3, 0]]), device="cpu")


def test_library_driver_records_carry_the_2opt_stage(capsys):
    """Host side of the drivers' optional 2-opt stage (elg_b200/lib_driver.py): record fields, per-bin lines; nothing new
    without it."""
    import json
    from elg_b200 import lib_driver as drv
    plain, refined = {}, {}
    drv.fill_record(plain, drv.InstanceCost(110.0), 100, 100.0)
    cost = drv.InstanceCost(110.0)
    cost.two_opt = (104.0, 0.5, 7)
    drv.fill_record(refined, cost, 100, 100.0)
    assert set(plain) == {"best_cost", "scale", "gap"} and json.dumps(plain) == json.dumps(
        {"best_cost": 110.0, "scale": 100, "gap": 0.1})
    assert refined["best_cost"] == 110.0 and abs(refined["gap_2opt"] - 0.04) < 1e-12
    assert refined["best_cost_2opt"] == 104.0 and refined["two_opt_seconds"] == 0.5 and refined["two_opt_iterations"] == 7
    edges = [("<200", 0, 200), ("200-500", 200, 500)]
    bins = drv.gap_bins([{"record": [plain]}], edges)
    assert "gap_2opt" not in bins and capsys.readouterr().out == ""
    bins = drv.gap_bins([{"record": [refined]}], edges)
    assert abs(bins["gap_2opt"]["<200"] - 4.0) < 1e-9 and abs(bins["<200"] - 10.0) < 1e-9
    assert capsys.readouterr().out.splitlines() == ["Average gap after 2-opt on subset of <200: 4.00%",
                                                    "Average gap after 2-opt total: 4.00%"]
