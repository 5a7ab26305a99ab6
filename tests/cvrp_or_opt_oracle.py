"""CPU oracle of the CVRP local search with Or-opt moves (elg_cvrp_local_search_ex; tests only).  It extends
tests/cvrp_ls_oracle.py, which states types 0..3 and stays the reference of elg_cvrp_local_search, with the segment
moves of max_segment 2 and 3: types 2s / 2s+1 move the s customers at positions i..i+s-1 (all of one route) forward /
reversed onto the edge (t_j, t_j+1), j outside i-1..i+s-1.  Gains are fp64 sums of the fp32 edges, loads are integer;
a move is applied by list surgery on the routes, so a route emptied by it disappears."""
import numpy as np
import torch

from cvrp_ls_oracle import _structure, apply_move as _apply_four, canonical, closed_length, edge_matrix, \
    move_gains as _gains_four, routes_of, row_of

__all__ = ["apply_move", "canonical", "closed_length", "cvrp_local_search", "edge_matrix", "move_gains", "routes_of",
           "row_of"]


def move_gains(D, dem, cap, row, max_segment=1):
    """Gains (2 + 2*max_segment, P, P) fp64 of every move on a canonical row, +inf where a move is not admissible or not
    feasible: types 0..3 of cvrp_ls_oracle, then for s = 2..max_segment the segment of s customers forward and reversed
    (types 2s, 2s+1).  D (N1, N1) fp64 edge lengths (fp32 values), dem (N1,) int demands."""
    g4 = _gains_four(D, dem, cap, row)
    if max_segment == 1:
        return g4
    P, rs = _structure(row)
    t = np.asarray(row[:P], dtype=np.int64)
    tt = np.append(t, [0, 0, 0])                          # node at each position, 0 past the last customer
    tn = np.append(t[1:], 0)
    tp = np.insert(t[:-1], 0, 0)
    load = np.zeros(P, dtype=np.int64)                    # route total by route start
    run = 0
    for p in range(P):
        run = 0 if t[p] == 0 else run + dem[t[p]]
        load[rs[p]] = max(load[rs[p]], run)
    I, J = np.arange(P)[:, None], np.arange(P)[None, :]
    a, v, vn = tp[I], t[J], tn[J]
    ri, rj = rs[I], rs[J]
    g = np.full((2 + 2 * max_segment, P, P), np.inf)
    g[:4] = g4
    for s in range(2, max_segment + 1):
        first, last, after = tt[I], tt[I + s - 1], tt[I + s]
        cust = np.all([tt[I + k] != 0 for k in range(s)], axis=0)
        sload = sum(dem[tt[I + k]] for k in range(s))
        ok = cust & ((J < I - 1) | (J > I + s - 1)) & ((rj == ri) | (load[rj] + sload <= cap))
        removed = D[a, after] - D[a, first] - D[last, after]
        g[2 * s] = np.where(ok, removed + D[v, first] - D[v, vn] + D[last, vn], np.inf)
        g[2 * s + 1] = np.where(ok, removed + D[v, last] - D[v, vn] + D[first, vn], np.inf)
    return g


def apply_move(row, L, move_type, i, j):
    """The move (type, i, j) of the contract on a canonical row -> the new canonical row."""
    if move_type < 4:
        return _apply_four(row, L, move_type, i, j)
    row = list(row)
    _, rs = _structure(row)
    s = move_type // 2
    routes = routes_of(row)
    ka, kb = row[:i + 1].count(0) - 1, row[:j + 1].count(0) - 1
    ca, cb = i - int(rs[i]) - 1, j - int(rs[j])           # list index of t_i; list index the segment goes before
    seg = routes[ka][ca:ca + s]
    del routes[ka][ca:ca + s]
    if kb == ka and cb > ca:
        cb -= s
    routes[kb][cb:cb] = seg if move_type % 2 == 0 else seg[::-1]
    return row_of(routes, L)


def cvrp_local_search(xy, rows, demand, capacity, max_iterations, rounding=False, record_moves=False, max_segment=1):
    """Best-improvement CVRP local search, the contract of elg_cvrp_local_search_ex (include/elg_b200.h), with the
    arguments and results of cvrp_ls_oracle.cvrp_local_search plus max_segment: smallest gain first, ties to the lowest
    (type, i, j), applied only if below -1e-6, at most max_iterations moves per row."""
    xy = torch.as_tensor(xy).float()
    demand = np.asarray(torch.as_tensor(demand).long())
    rows = torch.as_tensor(rows).long()
    R, L = rows.shape
    out = torch.zeros(R, L, dtype=torch.int64)
    length = torch.zeros(R, dtype=torch.float32)
    iters = torch.zeros(R, dtype=torch.int64)
    moves = [[] for _ in range(R)]
    cache = {}
    for r in range(R):
        b = r if xy.shape[0] > 1 else 0
        if b not in cache:
            cache[b] = edge_matrix(xy[b], rounding)
        D, dem = cache[b], demand[r if demand.shape[0] > 1 else 0]
        row = canonical(rows[r].tolist(), L)
        while int(iters[r]) < max_iterations:
            g = move_gains(D, dem, capacity, row, max_segment)
            k = int(np.argmin(g))
            best = float(g.reshape(-1)[k])
            if not best < -1e-6:
                break
            P = g.shape[1]
            mt, i, j = k // (P * P), k // P % P, k % P
            row = apply_move(row, L, mt, i, j)
            iters[r] += 1
            if record_moves:
                moves[r].append((mt, i, j, best))
        out[r] = torch.tensor(row)
        length[r] = closed_length(xy[b], row, rounding)
    return (out, length, iters, moves) if record_moves else (out, length, iters)
