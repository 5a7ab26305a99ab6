"""CPU oracle of the TSP local search with 2-opt and Or-opt moves (elg_tsp_local_search; tests only): a restatement of
its contract with fp32 edges computed as the kernels' seglen and fp64 gains.

Each iteration builds the gains of every variant as (6, rows, N1) arrays over blocks of positions i, takes the first
minimum in (v, i, j) order and applies the move to the tour as a list: a 2-opt move reverses a slice, an Or-opt move
takes the segment out and inserts it after the node t_j."""
import math

import torch

from two_opt_oracle import _seglen

# (segment length s, reversed) of the variants v = 0..5; s = 0 is the 2-opt move
VARIANTS = ((0, False), (1, False), (2, False), (2, True), (3, False), (3, True))


def _dist(rounding, exact):
    if exact:
        return lambda a, b: ((a.double() - b.double()) ** 2).sum(-1).sqrt()

    def d(a, b):
        e = _seglen(a - b)
        return (torch.round(e) if rounding else e).double()
    return d


def best_move(p, tour, max_segment, rounding=False, exact=False):
    """Smallest-gain admissible move of one tour -> (gain, v, i, j), first in key order v*N1^2 + i*N1 + j among equal
    gains; (inf, -1, -1, -1) if no move is admissible.  p (N1, 2) coordinates, tour the N1 node ids.  Edges are fp32
    seglen (rint if rounding) and gains fp64; exact: fp64 edges instead, for checking local optimality."""
    d = _dist(rounding, exact)
    t = torch.as_tensor(tour).long()
    n = len(t)
    pt = p[t].float()                                   # coordinates by position
    nxt = torch.roll(torch.arange(n), -1)
    e = d(pt, pt[nxt])                                  # e_p = d(t_p, t_p+1)
    J = torch.arange(n)[None, :]
    best = (math.inf, -1, -1, -1)
    blk = max(1, 1_000_000 // n)
    for i0 in range(0, n, blk):
        I = torch.arange(i0, min(n, i0 + blk))[:, None]
        # near[k][i, j] = d(t_j, t_i+k); the same quantity at j+1 is d(t_i+k, t_j+1)
        near = [d(pt[None, :], pt[torch.clamp(I + k, max=n - 1)]) for k in range(3)]
        g = torch.full((6, I.shape[0], n), math.inf, dtype=torch.float64)
        ok = (J >= I + 2) & ~((I == 0) & (J == n - 1))
        g[0] = torch.where(ok, (near[0] - e[I]) + (near[1][:, nxt] - e[J]), math.inf)
        for v in range(1, 6):
            s, rev = VARIANTS[v]
            if s > max_segment:
                continue
            last = I + s - 1
            ok = (I >= 1) & (last <= n - 1) & ((J < I - 1) | (J > last))
            lc = torch.clamp(last, max=n - 1)
            rem = (d(pt[I - 1], pt[(lc + 1) % n]) - e[I - 1]) - e[lc]          # t_i-1 joined to t_i+s
            ka, kb = (s - 1, 0) if rev else (0, s - 1)                          # a = t_i+ka, b = t_i+kb
            g[v] = torch.where(ok, rem + ((near[ka] - e[J]) + near[kb][:, nxt]), math.inf)
        k = int(g.argmin())
        m = float(g.reshape(-1)[k])
        v, i, j = k // (I.shape[0] * n), i0 + k // n % I.shape[0], k % n
        if m < best[0] or (m == best[0] and (v, i, j) < best[1:]):
            best = (m, v, i, j)
    return best


def apply_move(tour, v, i, j):
    """The move (v, i, j) of the contract on a tour given as a list of node ids -> the new list."""
    t = list(tour)
    if v == 0:
        t[i + 1:j + 1] = t[i + 1:j + 1][::-1]
        return t
    s, rev = VARIANTS[v]
    seg = t[i:i + s]
    anchor = t[j]
    rest = t[:i] + t[i + s:]
    k = rest.index(anchor)
    return rest[:k + 1] + (seg[::-1] if rev else seg) + rest[k + 1:]


def closed_length(p, tour, rounding):
    """fp32 closed length summed sequentially from the edge leaving position 0, as elg_tour_length sums it."""
    t = torch.as_tensor(tour).long()
    e = _seglen(p[t] - p[torch.roll(t, -1)])
    if rounding:
        e = torch.round(e)
    s = torch.zeros((), dtype=torch.float32)
    for q in range(len(e)):
        s = s + e[q]
    return s


def tsp_local_search(xy, tours, max_iterations, max_segment=3, rounding=False, record_moves=False):
    """Best-improvement 2-opt + Or-opt, the contract of elg_tsp_local_search (include/elg_b200.h).

    xy (R or 1, N1, 2) coordinates of each tour's instance; tours (R, L) int64 with a permutation in positions 0..N1-1
    (the rest is left alone).  Smallest gain first, ties to the lowest key; applied only if below -1e-6; at most
    max_iterations moves per tour.  Returns (tours (R, L), length (R,) fp32, iterations (R,) int64), plus per tour the
    list of applied moves (v, i, j, gain) if record_moves."""
    xy = torch.as_tensor(xy).float()
    tours = torch.as_tensor(tours).long().clone()
    R = tours.shape[0]
    N1 = xy.shape[1]
    length = torch.zeros(R, dtype=torch.float32)
    iters = torch.zeros(R, dtype=torch.int64)
    moves = [[] for _ in range(R)]
    for r in range(R):
        p = xy[r if xy.shape[0] > 1 else 0]
        t = tours[r, :N1].tolist()
        while int(iters[r]) < max_iterations:
            g, v, i, j = best_move(p, t, max_segment, rounding)
            if not g < -1e-6:
                break
            t = apply_move(t, v, i, j)
            iters[r] += 1
            if record_moves:
                moves[r].append((v, i, j, g))
        tours[r, :N1] = torch.tensor(t)
        length[r] = closed_length(p, t, rounding)
    return (tours, length, iters, moves) if record_moves else (tours, length, iters)
