"""CPU oracle of the capacity-aware CVRP local search (elg_cvrp_local_search; tests only): a restatement of its contract
with fp32 edges computed as the kernels' seglen, fp64 gains, integer loads and canonical compaction.

Each iteration builds the gains of every move of the four types as (P, P) arrays over the used positions of the
canonical row, takes the first minimum in (type, i, j) order and applies the move to the list of routes."""
import numpy as np
import torch

from two_opt_oracle import _seglen


def canonical(row, L):
    """Routes of a row in their order, each preceded by one 0, no empty route, zero padding to L."""
    out = [0]
    for v in row:
        v = int(v)
        if v != 0 or out[-1] != 0:
            out.append(v)
    return out + [0] * (L - len(out))


def routes_of(row):
    """Customer lists of a row's non-empty routes."""
    out, cur = [], []
    for v in row:
        v = int(v)
        if v == 0:
            if cur:
                out.append(cur)
            cur = []
        else:
            cur.append(v)
    return out + ([cur] if cur else [])


def row_of(routes, L):
    """Canonical row of a list of routes (empty ones dropped)."""
    out = [0]
    for r in routes:
        if r:
            out += r + [0]
    return out[:-1] + [0] * (L - len(out) + 1)


def _structure(row):
    """-> used positions P, route start rs[p] of every used position, load prefix pref[p] (route total at the depot)."""
    t = np.asarray(row)
    nz = np.nonzero(t)[0]
    P = int(nz[-1]) + 1 if len(nz) else 1
    rs = np.zeros(P, dtype=np.int64)
    start = 0
    for p in range(P):
        if t[p] == 0:
            start = p
        rs[p] = start
    return P, rs


def apply_move(row, L, move_type, i, j):
    """The move (type, i, j) of the contract on a canonical row -> the new canonical row."""
    row = list(row)
    P, rs = _structure(row)
    if move_type == 0:
        row[i + 1:j + 1] = row[i + 1:j + 1][::-1]
    elif move_type == 1:
        u = row[i]
        new = row[:i] + row[i + 1:]
        new.insert(j + 1 if j < i else j, u)
        row = new
    elif move_type == 2:
        row[i], row[j] = row[j], row[i]
    else:
        routes = routes_of(row)
        ka, kb = row[:i + 1].count(0) - 1, row[:j + 1].count(0) - 1     # every route is preceded by one 0
        A, B = routes[ka], routes[kb]
        ca, cb = i - int(rs[i]), j - int(rs[j])
        routes[ka], routes[kb] = A[:ca] + B[cb:], B[:cb] + A[ca:]
        return row_of(routes, L)
    return canonical(row, L)


def closed_length(xy, row, rounding):
    """fp32 closed length summed sequentially from the edge leaving position 0, as elg_tour_length sums it."""
    t = torch.as_tensor(row)
    e = _seglen(xy[t] - xy[torch.roll(t, -1)])
    if rounding:
        e = torch.round(e)
    s = torch.zeros((), dtype=torch.float32)
    for q in range(len(e)):
        s = s + e[q]
    return s


def move_gains(D, dem, cap, row):
    """Gains (4, P, P) fp64 of every move on a canonical row, +inf where a move is not admissible or not feasible.
    D (N1, N1) fp64 edge lengths (fp32 values), dem (N1,) int demands."""
    P, rs = _structure(row)
    t = np.asarray(row[:P], dtype=np.int64)
    tn = np.append(t[1:], 0)                              # node after each position (0 after the last customer)
    tp = np.insert(t[:-1], 0, 0)                          # node before each position (unused at position 0)
    pref = np.zeros(P, dtype=np.int64)
    for p in range(1, P):
        pref[p] = 0 if t[p] == 0 else pref[p - 1] + dem[t[p]]
    load = np.zeros(P, dtype=np.int64)                    # route total by route start
    for p in range(P):
        load[rs[p]] = max(load[rs[p]], pref[p])
    I, J = np.arange(P)[:, None], np.arange(P)[None, :]
    u, a, b = t[I], tp[I], tn[I]
    v, vn, vp = t[J], tn[J], tp[J]
    ri, rj = rs[I], rs[J]
    du, dv = dem[u], dem[v]
    pa, pb = np.where(u != 0, pref[I], 0), np.where(v != 0, pref[J], 0)
    la, lb = load[ri], load[rj]
    other = (J > I) & (ri != rj)
    g = np.full((4, P, P), np.inf)
    ok0 = (J >= I + 2) & (rj <= I)
    g[0] = np.where(ok0, D[u, v] + D[b, vn] - D[u, b] - D[v, vn], np.inf)
    ok1 = (u != 0) & (J != I - 1) & (J != I) & ((rj == ri) | (lb + du <= cap))
    g[1] = np.where(ok1, D[a, b] - D[a, u] - D[u, b] + D[v, u] + D[u, vn] - D[v, vn], np.inf)
    ok2 = other & (u != 0) & (v != 0) & (la - du + dv <= cap) & (lb - dv + du <= cap)
    g[2] = np.where(ok2, D[a, v] + D[v, b] + D[vp, u] + D[u, vn] - D[a, u] - D[u, b] - D[vp, v] - D[v, vn], np.inf)
    ok3 = other & (pa + lb - pb <= cap) & (pb + la - pa <= cap)
    g[3] = np.where(ok3, D[u, vn] + D[v, b] - D[u, b] - D[v, vn], np.inf)
    return g


def edge_matrix(xy, rounding):
    e = _seglen(xy[:, None, :] - xy[None, :, :])
    return (torch.round(e) if rounding else e).double().numpy()


def cvrp_local_search(xy, rows, demand, capacity, max_iterations, rounding=False, record_moves=False):
    """Best-improvement CVRP local search, the contract of elg_cvrp_local_search (include/elg_b200.h).

    xy (R or 1, N1, 2) coordinates of each row's instance; rows (R, L) int64 rollout rows; demand (R or 1, N1) integer
    demands (demand[., 0] = 0); capacity an integer.  Smallest gain first, ties to the lowest type*L^2 + i*L + j; applied
    only if below -1e-6; at most max_iterations moves per row.  Returns (canonical rows (R, L) int64, length (R,) fp32,
    iterations (R,) int64), plus per row the list of applied moves (type, i, j, gain) if record_moves."""
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
            g = move_gains(D, dem, capacity, row)
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
