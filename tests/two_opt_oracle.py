"""CPU oracle of the 2-opt local search (elg_two_opt; tests only): a vectorised restatement of its contract, with
fp32 edges computed as the kernels' seglen and fp64 gains.

It is the counterpart of the reference's batched_two_opt_torch (TSP/utils.py:28-70, CVRP/utils.py:31-67) with the
semantics of elg_two_opt: each tour stops on its own and CVRP moves stay inside one route."""
import math

import torch


def _seglen(d):
    """((a-b)**2).sum(-1).sqrt() with a correctly rounded fp32 sqrt, as the kernels' seglen (__fsqrt_rn).  torch's
    vectorised fp32 sqrt on the CPU is off by one ulp now and then; the fp64 sqrt of an fp32 value rounded to fp32 is
    exact."""
    return (d ** 2).sum(-1).double().sqrt().float()


def two_opt(kind, xy, tours, max_iterations, rounding=False, record_moves=False):
    """Best-improvement 2-opt, the contract of elg_two_opt (include/elg_b200.h).

    xy (R or 1, N1, 2) coordinates of each tour's instance; tours (R, L) int64 (tsp: positions 0..N1-1 are the tour,
    the rest is left alone; cvrp: a rollout row with depot visits and zero padding).  A move reverses positions
    i+1..j (i < j, j+1 wraps to 0) with gain d(t_i,t_j) + d(t_i+1,t_j+1) - d(t_i,t_i+1) - d(t_j,t_j+1): edges in fp32
    as the kernels' seglen computes them (then rint if rounding), gains in fp64.  Admissible: j >= i+2; tsp not
    (0, N1-1); cvrp only if positions i+1..j are all customers.  Smallest gain first, ties to the lowest i*L + j; applied
    only if below -1e-6; at most max_iterations moves per tour.
    Returns (tours (R, L), length (R,) fp32 summed sequentially like elg_tour_length, iterations (R,) int64), plus
    per tour the list of applied moves (i, j, gain) if record_moves."""
    xy = xy.float()
    tours = tours.clone().long()
    R, L = tours.shape
    N1 = xy.shape[1]
    n = L if kind == "cvrp" else N1
    pos = torch.arange(n)
    nxt = (pos + 1) % n
    iters = torch.zeros(R, dtype=torch.int64)
    moves = [[] for _ in range(R)]

    for r in range(R):
        p = xy[r if xy.shape[0] > 1 else 0]
        t = tours[r, :n]

        def seg(a, b):
            e = _seglen(p[a] - p[b])
            return torch.round(e) if rounding else e

        if kind == "cvrp":
            lastdep = torch.where(t == 0, pos, torch.full_like(pos, -1)).cummax(0)[0]
            dmax = int((pos - lastdep).max()) if n else 0
        else:
            lastdep, dmax = None, n - 1
        blk = max(1, 4_000_000 // max(n, 1)) if kind == "tsp" else max(64, dmax)   # cvrp: narrow column windows
        while int(iters[r]) < max_iterations:
            edge = seg(t, t[nxt]).double()
            best, bi, bj = math.inf, -1, -1
            for i0 in range(0, n, blk):
                i = pos[i0:i0 + blk, None]
                j = pos[None, i0:min(n, i0 + blk + dmax + 1)]       # columns beyond i + dmax are never admissible
                gain = seg(t[i], t[j]).double() + seg(t[nxt[i]], t[nxt[j]]).double() - edge[i] - edge[j]
                ok = j >= i + 2
                if kind == "cvrp":
                    ok = ok & (lastdep[j] <= i)
                else:
                    ok = ok & ~((i == 0) & (j == n - 1))
                gain = gain.masked_fill(~ok, math.inf)
                k = int(gain.argmin())
                g = float(gain.reshape(-1)[k])
                if g < best:
                    best, bi, bj = g, i0 + k // gain.shape[1], i0 + k % gain.shape[1]
            if not best < -1e-6:
                break
            t[bi + 1:bj + 1] = t[bi + 1:bj + 1].flip(0)
            iters[r] += 1
            if record_moves:
                moves[r].append((bi, bj, best))

    pts = xy.expand(R, -1, -1).gather(1, tours[:, :n, None].expand(-1, -1, 2))
    edges = _seglen(pts - pts[:, nxt])
    if rounding:
        edges = torch.round(edges)
    length = torch.zeros(R, dtype=torch.float32)
    for q in range(n):                                  # sequential fp32 sum, the order of elg_tour_length
        length = length + edges[:, q]
    return (tours, length, iters, moves) if record_moves else (tours, length, iters)
