"""Or-opt moves of the CVRP local search on the GPU (elg_cvrp_local_search_ex with max_segment 2 and 3, engine and drop-in
max_segment, the drivers' params.local_search_max_segment) against the CPU oracle (tests/cvrp_or_opt_oracle.py).

Under the rounded library metric every edge is an integer, so the kernel must make the oracle's moves exactly.  Under
the scaled metric only the invariants are exact.  max_segment = 1 must be elg_cvrp_local_search bit for bit."""
import ctypes as C
import os
import random

import pytest
import torch

import cvrp_or_opt_oracle as LS
from local_search_helpers import DEV, ROOT, cfg, greedy_rows, model, setx_rows

pytestmark = pytest.mark.gpu


def _greedy_rows(N, n, seed):
    cap = {100: 50, 1000: 250}[N]
    xy, dem, rows = greedy_rows("cvrp", N, n, seed, capacity=float(cap))
    return xy, dem, cap, rows


def _units(dem, cap):
    return torch.round(dem.double().cpu() * cap).long()


def _check_invariants(xy, dem, rows, out, length, rounding=False):
    from elg_b200 import engine
    from elg_b200.cvrp import check_feasible
    rows, out = rows.cpu(), out.cpu()
    assert torch.equal(length.cpu(), engine.tour_length(xy, out.to(DEV)[:, None], rounding)[:, 0].cpu())   # bit for bit
    assert (length.cpu() <= engine.tour_length(xy, rows.to(DEV)[:, None], rounding)[:, 0].cpu()).all()
    for r in range(len(out)):
        row = out[r].tolist()
        assert LS.canonical(row, len(row)) == row
        assert len(LS.routes_of(row)) <= len(LS.routes_of(rows[r].tolist()))
        check_feasible(out[r][None, None].to(DEV), dem[r if dem.shape[0] > 1 else 0][None, 1:])


def _parent_call(xy, rows, dem, cap, max_iterations, rounding):
    """elg_cvrp_local_search, the four-move entry point, called directly"""
    from elg_b200._lib import check, lib
    R, L = rows.shape
    t16 = rows.to(torch.int16).contiguous()
    xy = xy.contiguous().float()
    units = torch.round(dem.double() * cap).to(torch.int32).contiguous()
    length = torch.empty(R, dtype=torch.float32, device=DEV)
    iters = torch.empty(R, dtype=torch.int32, device=DEV)
    p = lambda t: C.c_void_p(t.data_ptr())
    check(lib.elg_cvrp_local_search(p(xy), int(xy.shape[0]), int(xy.shape[1]), p(units), cap, C.c_void_p(0), p(t16), R,
                                    L, int(rounding), max_iterations, p(iters), p(length),
                                    C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return t16.long(), length, iters


# ------------------------------------------------------------------------------------------------ 1. exact parity

_seen = {2: set(), 3: set()}


@pytest.mark.parametrize("max_segment", [2, 3])
@pytest.mark.parametrize("name,rows_used,cap", [("X-n101-k25", 8, 1000), ("X-n200-k36", 8, 1000),
                                                ("X-n298-k31", 3, 1000), ("X-n1001-k43", 2, 6)])
def test_rounded_metric_identical_to_oracle(name, rows_used, cap, max_segment):
    from elg_b200 import engine
    xy, dem, capacity, rows = setx_rows(name)
    xy, dem, rows = xy[:rows_used], dem[:rows_used], rows[:rows_used]
    out, length, iters = engine.cvrp_local_search(xy, rows, dem, capacity, max_iterations=cap, rounding=True,
                                                  max_segment=max_segment)
    ref_t, ref_len, ref_it, moves = LS.cvrp_local_search(xy.cpu(), rows.cpu(), _units(dem, capacity), capacity, cap,
                                                         True, record_moves=True, max_segment=max_segment)
    assert torch.equal(iters.cpu().long(), ref_it)
    assert torch.equal(out.cpu(), ref_t)
    assert torch.equal(length.cpu(), ref_len)
    assert int(iters.min()) > 0
    if cap < 1000:
        assert int(iters.min()) == cap
    _seen[max_segment].update(m[0] for row in moves for m in row)


def test_parity_cases_made_segment_moves():
    """The parity runs above applied moves of every new type (runs after them in file order)."""
    if not _seen[3]:
        pytest.skip("the parity cases did not run in this session")
    assert {4, 5} <= _seen[2] and max(_seen[2]) == 5
    assert {4, 5, 6, 7} <= _seen[3]


@pytest.mark.parametrize("max_segment", [2, 3])
def test_small_random_rows_identical_to_oracle(max_segment):
    """Integer coordinates and the rounded metric: doubled depot visits, one-customer routes, tight capacities."""
    from elg_b200 import engine
    g = torch.Generator().manual_seed(7)
    N1, R, cap = 12, 64, 8
    xy = torch.floor(torch.rand(R, N1, 2, generator=g) * 30)
    units = torch.randint(1, 4, (R, N1), generator=g)
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
                                                  rounding=True, max_segment=max_segment)
    ref_t, ref_len, ref_it, moves = LS.cvrp_local_search(xy, rows, units, cap, 1000, True, record_moves=True,
                                                         max_segment=max_segment)
    assert torch.equal(out.cpu(), ref_t) and torch.equal(iters.cpu().long(), ref_it) and torch.equal(length.cpu(), ref_len)
    assert any(m[0] >= 4 for row in moves for m in row)


# ------------------------------------------------------------------------------------------------ 2. max_segment = 1

def test_max_segment_one_is_the_four_move_search():
    from elg_b200 import engine
    xy, dem, cap, rows = _greedy_rows(100, 4, seed=21)
    for rounding in (False, True):
        a = engine.cvrp_local_search(xy, rows, dem, cap, rounding=rounding, max_segment=1)
        b = _parent_call(xy, rows, dem, cap, 1000, rounding)
        assert all(torch.equal(x, y) for x, y in zip(a, b)) and int(a[2].sum()) > 0
    for name in ("X-n101-k25", "X-n200-k36"):
        xy, dem, cap, rows = setx_rows(name)
        a = engine.cvrp_local_search(xy, rows, dem, cap, rounding=True)
        b = _parent_call(xy, rows, dem, cap, 1000, True)
        assert all(torch.equal(x, y) for x, y in zip(a, b)) and int(a[2].sum()) > 0


# ------------------------------------------------------------------------------------------------ 3. invariants

@pytest.mark.parametrize("N,n", [(100, 4), (1000, 1)])
def test_random_instances_scaled_metric(N, n):
    from elg_b200 import engine
    xy, dem, cap, rows = _greedy_rows(N, n, seed=N + 1)
    for max_segment in (2, 3):
        out, length, iters = engine.cvrp_local_search(xy, rows, dem, cap, max_segment=max_segment)
        _check_invariants(xy, dem, rows, out, length)
        assert int(iters.min()) > 0
        again = engine.cvrp_local_search(xy, rows, dem, cap, max_segment=max_segment)
        assert all(torch.equal(x, y) for x, y in zip((out, length, iters), again))          # deterministic


def test_inst_mapping_and_shared_instance():
    from elg_b200 import engine
    xy, dem, cap, rows = _greedy_rows(100, 2, seed=4)          # 16 rows over 16 aug-instances
    a = engine.cvrp_local_search(xy, rows, dem, cap, max_segment=3)
    b = engine.cvrp_local_search(xy, rows.to(torch.int16), dem, cap, max_segment=3)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    inst = torch.arange(16, device=DEV).flip(0)
    by_inst = engine.cvrp_local_search(xy.flip(0), rows, dem.flip(0), cap, inst=inst, max_segment=3)
    assert all(torch.equal(x, y) for x, y in zip(a, by_inst))
    one = engine.cvrp_local_search(xy[:1], rows[:1].expand(5, -1), dem[:1], cap, max_segment=3)     # Bxy = 1
    assert all(torch.equal(x, y[:1].expand_as(x)) for x, y in zip(one, a))


# ------------------------------------------------------------------------------------------------ 4. the largest rows

def test_largest_rows_best_move_has_a_key_above_int32():
    """N1 = 8192, L = 2*N1+2: 8170 one-customer routes (customers at the depot's coordinates, so moving them gains
    nothing) and a last route of 21 customers on a quarter circle of radius 1000 around the depot, visited in angular
    order 0..20 except that points 5, 6, 7 come last as 7 6 5.  The best move puts them back reversed between points 4
    and 8: type 7, i = 16359, j = 16345, key 7*L^2 + i*L + j = 2147581891 > 2^31-1, gain -1133 under the rounded metric.
    With max_segment = 2 the best move is a 2-opt of gain -436 (both checked with the oracle on a reduced row)."""
    import math
    from elg_b200 import engine
    N1, L = 8192, 2 * 8192 + 2
    arc = [(round(1000 * math.cos(k * math.pi / 40)), round(1000 * math.sin(k * math.pi / 40))) for k in range(21)]
    order = [k for k in range(21) if k not in (5, 6, 7)] + [7, 6, 5]
    K = N1 - 1 - len(order)
    xy = torch.zeros(1, N1, 2)
    xy[0, K + 1:] = torch.tensor([arc[k] for k in order], dtype=torch.float32)
    row = [0]
    for v in range(1, K + 1):
        row += [v, 0]
    row += list(range(K + 1, N1))
    P = len(row)
    assert K == 8170 and P == 16362 and 7 * L * L + 16359 * L + 16345 > 2 ** 31 - 1
    rows = torch.tensor(row + [0] * (L - P))[None]
    dem = torch.full((1, N1), 0.01)
    dem[0, 0] = 0
    want = row[:16346] + row[16359:][::-1] + row[16346:16359] + [0] * (L - P)
    before = float(engine.tour_length(xy.to(DEV), rows.to(DEV)[:, None], rounding=True)[0, 0])
    for max_segment, gain in ((3, 1133), (2, 436)):
        out, length, iters = engine.cvrp_local_search(xy.to(DEV), rows.to(DEV), dem.to(DEV), 100, max_iterations=1,
                                                      rounding=True, max_segment=max_segment)
        assert int(iters[0]) == 1 and float(length[0]) == before - gain
        assert (out[0].tolist() == want) == (max_segment == 3)
        _check_invariants(xy.to(DEV), dem.to(DEV), rows, out, length, rounding=True)


# ------------------------------------------------------------------------------------------------ 5. drop-in, drivers

def test_drop_in_passes_max_segment():
    from elg_b200 import engine
    from elg_b200.cvrp import cvrp_local_search
    xy, dem, cap, rows = _greedy_rows(100, 1, seed=9)
    pts, d, rows = xy[0], dem[0], rows[:1]
    for max_segment in (1, 3):
        want, _, it = engine.cvrp_local_search(pts[None], rows, d[None], cap, max_iterations=500, max_segment=max_segment)
        t, n = cvrp_local_search(pts, d, cap, rows, max_iterations=500, device=DEV, max_segment=max_segment)
        assert torch.equal(t, want) and n == int(it.max()) > 0
    with pytest.raises(ValueError, match="max_segment"):
        cvrp_local_search(pts, d, cap, rows, max_segment=0)


def test_vrplib_driver_with_max_segment(tmp_path, monkeypatch, capsys):
    """test_vrplib with local_search_max_segment 3: the usual records, best_cost_ls the best over the augmentations of
    engine.cvrp_local_search(..., max_segment=3, rounding=True) on the rows the stage refined."""
    from elg_b200 import engine, lib_driver as drv
    from elg_b200.cvrp.test_vrplib import VRPLib_Tester
    real, calls = engine.cvrp_local_search, []

    def recording(xy, rows, demand, capacity, **kw):
        calls.append((xy.clone(), rows.clone(), demand.clone(), capacity, kw))
        return real(xy, rows, demand, capacity, **kw)
    monkeypatch.setattr(drv.engine, "cvrp_local_search", recording)
    config = cfg("cvrp", local_search_iterations=300, local_search_max_segment=3)
    config["vrplib_path"] = os.path.join(ROOT, "tests", "golden", "vrplib")
    random.seed(1)
    results = VRPLib_Tester(config, model=model("cvrp", 3, 3.0)).test_on_vrplib(out_dir=str(tmp_path))
    recs = [r["record"][0] for r in results[:-1]]
    assert len(recs) == len(calls) == 2
    lines = capsys.readouterr().out.splitlines()
    assert sum(l.startswith("Instance Name ") and "gap after local search" in l for l in lines) == 2
    for rec, (xy, rows, demand, capacity, kw) in zip(recs, calls):
        assert set(rec) >= {"best_cost", "gap", "best_cost_ls", "gap_ls", "ls_seconds", "ls_iterations"}
        assert kw == {"max_iterations": 300, "rounding": True, "max_segment": 3}
        _, length, iters = real(xy, rows, demand, capacity, max_iterations=300, rounding=True, max_segment=3)
        assert rec["best_cost_ls"] == float(length.min()) and rec["ls_iterations"] == int(iters.sum())
        assert rec["best_cost_ls"] <= rec["best_cost"]
