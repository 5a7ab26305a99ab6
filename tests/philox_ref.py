"""CPU restatement of the library's random streams (Philox4x32-10, rollout_common.cuh), in numpy.

- `sample_uniform`: the uniform behind every sampled decision of `elg_rollout` / `elg_decode_step` (mode = sample).
  Counter (grow lo, grow hi, step lo, step hi), grow = b * M + m the global row; key (seed lo, seed hi); the first
  output word x is mapped to ((x >> 8) + 0.5f) * 2^-24 in fp32, so u lies in [2^-25, 1] and 2^24 - 1 rounds to 1.0.
  The kernel selects the first node j, in node-index order, with u * total <= cdf[j] and p[j] > 0.
- `generate`: `generate_kernel` (generate.cu) instance by instance, for the uniform, cluster and mixed kinds.
"""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
PHILOX_M0, PHILOX_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
PHILOX_W0, PHILOX_W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
U_TOP = np.float32(1.0)                      # the largest uniform: x >> 8 == 2^24 - 1
U_BOTTOM = np.float32(2.0 ** -25)            # the smallest: x >> 8 == 0


def philox4x32_10(ctr, key):
    """ctr: four uint32 words, key: two (scalars or broadcastable arrays) -> four uint64 arrays holding uint32 values."""
    c = [np.asarray(x, dtype=np.uint64) & M32 for x in ctr]
    k = [np.asarray(x, dtype=np.uint64) & M32 for x in key]
    for _ in range(10):
        p0, p1 = PHILOX_M0 * c[0], PHILOX_M1 * c[2]          # < 2^64: exact in uint64
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k[0], p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k[1], p0 & M32]
        k = [(k[0] + PHILOX_W0) & M32, (k[1] + PHILOX_W1) & M32]
    return c


def _lo_hi(v):
    v = np.asarray(v, dtype=np.uint64)
    return v & M32, v >> np.uint64(32)


def uniform_from_word(x):
    """The sampler's fp32 mapping ((x >> 8) + 0.5f) * (1 / 2^24), with the kernel's roundings."""
    k = (np.asarray(x, dtype=np.uint64) >> np.uint64(8)).astype(np.float32)
    return (k + np.float32(0.5)) * np.float32(1.0 / 16777216.0)


def sample_uniform(seed, grow, step):
    """Uniform of the sampled decision of global row grow (= b * M + m) at `step` (the fused rollout's tour position t,
    or elg_decode_step's step argument).  Arguments broadcast; returns fp32."""
    g_lo, g_hi = _lo_hi(grow)
    s_lo, s_hi = _lo_hi(step)
    k_lo, k_hi = _lo_hi(seed)
    return uniform_from_word(philox4x32_10((g_lo, g_hi, s_lo, s_hi), (k_lo, k_hi))[0])


# ------------------------------------------------------------------------------------------------ generators
def generator_stream(seed, b, stream, i):
    """Four uint32 words rnd(stream, i) of instance b: counter (i, b, stream, 0x9e3779b9), key (seed lo, seed hi)."""
    k_lo, k_hi = _lo_hi(seed)
    return philox4x32_10((i, b, stream, 0x9E3779B9), (k_lo, k_hi))


def u01(x):
    """(x >> 8) * 2^-24 in fp32: exact, in [0, 1)."""
    return (np.asarray(x, dtype=np.uint64) >> np.uint64(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)


def _gauss(r, stdv):
    """fp64 of stdv * rad * (cos ang, sin ang) with the kernel's fp32 inputs rad = sqrt(-2 log(1 - u_z)),
    ang = 2 pi u_w (the fp32 product, as the kernel rounds it)."""
    uz, uw = u01(r[2]), u01(r[3])
    rad = np.sqrt(-2.0 * np.log((np.float32(1.0) - uz).astype(np.float64)))
    ang = (np.float32(6.283185307179586) * uw).astype(np.float64)
    s = float(np.float32(stdv))
    return s * rad * np.cos(ang), s * rad * np.sin(ang)


def generate(problem, kind, n, N, n_cluster, lower, upper, stdv, capacity, seed):
    """generate_kernel for instances b = 0 .. n-1.  Returns a dict of numpy arrays:
    node (n, N, 2) and depot (n, 2) | None in fp64: exact where the kernel is exact, and for Gaussian points the fp64
    value before the clamp to [0, 1]; gauss (n, N) / depot_gauss (n,): which points went through logf / sinf / cosf;
    demand (n, N) fp32 | None; depot_idx (n,): cvrp cluster, the depot's index among the P = N + 1 points, else -1;
    mutated (n, N) bool: mixed, the redrawn half.

    The cluster centres lower + (upper - lower) u are rounded as a product and a sum; nvcc may contract them into one
    FMA, which moves a centre by at most one ulp (< 6e-8), far inside the bar Gaussian points are compared at."""
    cvrp = problem == "cvrp"
    nc = 1 if kind == 0 else n_cluster
    P = N + 1 if (cvrp and kind == 1) else N
    lo, hi = np.float32(lower), np.float32(upper)
    span = hi - lo
    out = dict(depot=np.zeros((n, 2)) if cvrp else None, depot_gauss=np.zeros(n, bool), node=np.zeros((n, N, 2)),
               gauss=np.zeros((n, N), bool), demand=np.zeros((n, N), np.float32) if cvrp else None,
               depot_idx=np.full(n, -1), mutated=np.zeros((n, N), bool))
    for b in range(n):
        r = generator_stream(seed, b, 1, np.arange(nc))
        cu = np.stack((u01(r[0]), u01(r[1])), axis=1)
        mul = (span * cu).astype(np.float32) + lo
        depot_idx = int(u01(generator_stream(seed, b, 2, 0)[0]) * np.float32(N + 1))
        perm = np.arange(N)
        if kind == 2:
            for i in range(N // 2):
                j = i + int(u01(generator_stream(seed, b, 3, i)[0]) * np.float32(N - i))
                j = min(j, N - 1)
                perm[i], perm[j] = perm[j], perm[i]
        r = generator_stream(seed, b, 4, np.arange(P))
        pts = np.stack((u01(r[0]), u01(r[1])), axis=1).astype(np.float64)
        gauss = np.zeros(P, bool)
        if kind == 1:
            g = P // nc
            c = np.minimum(np.arange(P) // max(g, 1), nc - 1)
            dx, dy = _gauss(r, stdv)
            pts = np.stack((mul[c, 0] + dx, mul[c, 1] + dy), axis=1)
            gauss[:] = True
        if kind == 2:
            half, g = N // 2, N // nc // 2
            i = np.arange(half)
            c = np.minimum(i // max(g, 1), nc - 1)
            dx, dy = _gauss(generator_stream(seed, b, 5, i), stdv)
            idx = perm[:half]
            pts[idx] = np.stack((mul[c, 0] + dx, mul[c, 1] + dy), axis=1)
            gauss[idx] = True
            out["mutated"][b, idx] = True
        if cvrp and kind == 1:
            out["depot_idx"][b] = depot_idx
            keep = np.arange(P) != depot_idx
            out["depot"][b], out["depot_gauss"][b] = pts[depot_idx], True
            out["node"][b], out["gauss"][b] = pts[keep], gauss[keep]
        else:
            out["node"][b], out["gauss"][b] = pts[:N], gauss[:N]
            if cvrp:
                r6 = generator_stream(seed, b, 6, 0)
                out["depot"][b] = (u01(r6[0]), u01(r6[1]))
        if cvrp:
            q = 1 + np.minimum((u01(generator_stream(seed, b, 7, np.arange(N))[0]) * np.float32(9.0)).astype(np.int64), 8)
            out["demand"][b] = q.astype(np.float32) / np.float32(capacity)
    return out
