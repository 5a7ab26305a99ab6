"""GPU: device data generators against the distributions of the reference's generate_vrp_data / generate_tsp_data
(CVRP/generate_data.py:9-92, TSP/generate_data.py:9-57): ranges, clamps, demand alphabet, cluster geometry, the
mutated half of `mixed`, determinism per seed; and instance by instance against the CPU restatement of the kernel."""
import numpy as np
import pytest
import torch

import philox_ref

pytestmark = pytest.mark.gpu
DIST = {"data_type": "uniform", "n_cluster": 3, "n_cluster_mix": 1, "lower": 0.2, "upper": 0.8, "std": 0.07}


def test_uniform_cvrp():
    from elg_b200.generate_data import CAPACITIES, generate_vrp_data
    d = generate_vrp_data(512, 100, DIST, seed=1)
    assert d["loc"].shape == (512, 100, 2) and d["depot"].shape == (512, 1, 2) and d["demand"].shape == (512, 100)
    for t in (d["loc"], d["depot"]):
        assert float(t.min()) >= 0.0 and float(t.max()) < 1.0
    assert abs(float(d["loc"].mean()) - 0.5) < 5e-3 and abs(float(d["loc"].var()) - 1 / 12) < 3e-3
    q = d["demand"] * CAPACITIES[100]
    assert torch.equal(q, q.round()) and float(q.min()) == 1 and float(q.max()) == 9
    counts = torch.bincount(q.long().flatten(), minlength=10)[1:].float()
    assert float((counts / counts.sum() - 1 / 9).abs().max()) < 0.01
    d2 = generate_vrp_data(512, 100, DIST, seed=1)
    assert torch.equal(d["loc"], d2["loc"]) and torch.equal(d["demand"], d2["demand"])
    assert not torch.equal(d["loc"], generate_vrp_data(512, 100, DIST, seed=2)["loc"])
    with pytest.raises(KeyError):
        generate_vrp_data(4, 37, DIST, seed=1)


@pytest.mark.parametrize("problem", ["cvrp", "tsp"])
def test_cluster(problem):
    from elg_b200.generate_data import generate_tsp_data, generate_vrp_data
    dist = dict(DIST, data_type="cluster")
    N = 100
    if problem == "cvrp":
        d = generate_vrp_data(256, N, dist, seed=3)
        pts = torch.cat((d["loc"], d["depot"]), dim=1)          # the depot was one of the N + 1 clustered points
    else:
        pts = generate_tsp_data(256, N, dist, seed=3)
    assert float(pts.min()) >= 0.0 and float(pts.max()) <= 1.0
    # every point lies within 6 std of one of at most 3 centres inside [lower, upper]^2: per-instance k-means-free
    # check through the group structure (tsp keeps the generation order: 3 consecutive groups of 33, 33, 34)
    if problem == "tsp":
        g = [pts[:, :33], pts[:, 33:66], pts[:, 66:]]
        for grp in g:
            c = grp.mean(dim=1, keepdim=True)
            assert float(c.min()) > 0.2 - 0.05 and float(c.max()) < 0.8 + 0.05
            sd = (grp - c).pow(2).mean(dim=(1, 2)).sqrt()
            assert abs(float(sd.mean()) - 0.07) < 0.01
    # clustered data is far more concentrated than uniform data
    assert float(pts.var(dim=1).mean()) < 0.06


def test_mixed_tsp_half_mutated():
    from elg_b200.generate_data import generate_tsp_data
    dist = dict(DIST, data_type="mixed")
    pts = generate_tsp_data(256, 100, dist, seed=5)
    assert pts.shape == (256, 100, 2) and float(pts.min()) >= 0.0 and float(pts.max()) <= 1.0
    # one cluster of 50 points with std 0.07 around a centre in [0.2, 0.8]^2: the 50 points nearest to the densest spot
    med = pts.median(dim=1, keepdim=True)[0]
    d = (pts - med).norm(dim=2)
    near = (d < 0.25).float().sum(dim=1)
    assert float(near.mean()) > 50          # the cluster (50) plus the uniform points that happen to fall inside
    assert float(near.mean()) < 75


# ---------------------------------------------------------------------------------------- instance by instance
# generate_kernel restated on the CPU (philox_ref.generate): the same Philox4x32-10 counters.  Uniform coordinates,
# depots and demands are exact (integer -> float, products by 2^-24, truncation, IEEE division), so they must agree bit
# for bit, as must the depot index of cvrp `cluster` and the points `mixed` leaves alone.  Gaussian points go through
# logf / sinf / cosf and possibly a contracted FMA: within 1e-6, and exactly 0 or 1 where the fp64 value lies outside
# [0, 1] (the clamp).
GAUSS_ATOL = 1e-6


def _check_points(got, ref, gauss, what):
    got = got.detach().cpu().double().numpy()
    gauss = np.broadcast_to(gauss[..., None], ref.shape) if ref.ndim == gauss.ndim + 1 else gauss
    exact = ~gauss
    assert np.array_equal(got[exact], ref[exact]), (what, int((got[exact] != ref[exact]).sum()))
    if gauss.any():
        err = np.abs(got[gauss] - np.clip(ref[gauss], 0.0, 1.0))
        assert float(err.max()) < GAUSS_ATOL, (what, float(err.max()))
        lo, hi = gauss & (ref < -GAUSS_ATOL), gauss & (ref > 1 + GAUSS_ATOL)
        assert np.all(got[lo] == 0.0) and np.all(got[hi] == 1.0), what
        return int(lo.sum() + hi.sum())
    return 0


def _generate(problem, kind, n, N, nc, lower, upper, std, seed):
    from elg_b200.generate_data import CAPACITIES, generate_tsp_data, generate_vrp_data
    dist = {"data_type": ["uniform", "cluster", "mixed"][kind], "n_cluster": nc, "n_cluster_mix": nc, "lower": lower,
            "upper": upper, "std": std}
    cap = CAPACITIES[N] if problem == "cvrp" else 1.0
    ref = philox_ref.generate(problem, kind, n, N, nc, lower, upper, std, cap, seed)
    if problem == "cvrp":
        d = generate_vrp_data(n, N, dist, seed=seed)
        return ref, d["loc"], d["depot"][:, 0], d["demand"]
    return ref, generate_tsp_data(n, N, dist, seed=seed), None, None


@pytest.mark.parametrize("N", [10, 20, 50, 100, 200, 500, 1000])
def test_uniform_cvrp_bit_for_bit(N):
    ref, loc, depot, demand = _generate("cvrp", 0, 3, N, 1, 0.2, 0.8, 0.07, seed=11 + N)
    _check_points(loc, ref["node"], ref["gauss"], "loc")
    _check_points(depot, ref["depot"], ref["depot_gauss"], "depot")
    assert np.array_equal(demand.cpu().numpy(), ref["demand"])


def test_uniform_tsp_bit_for_bit_with_a_seed_above_2_32():
    for seed in (3, 2 ** 32 + 3, 2 ** 63 + 12345):
        ref, loc, _, _ = _generate("tsp", 0, 5, 37, 1, 0.2, 0.8, 0.07, seed=seed)
        _check_points(loc, ref["node"], ref["gauss"], seed)
    a = _generate("tsp", 0, 2, 37, 1, 0.2, 0.8, 0.07, seed=3)[1]
    b = _generate("tsp", 0, 2, 37, 1, 0.2, 0.8, 0.07, seed=2 ** 32 + 3)[1]
    assert not torch.equal(a, b)                 # the key's high word reaches the stream


# (problem, N, n_cluster, std): N not divisible by n_cluster, N + 1 < n_cluster, one cluster, the largest count; a wide
# std so that some points are clamped
CLUSTER_CASES = [("tsp", 50, 3, 0.07), ("tsp", 37, 16, 0.07), ("tsp", 10, 16, 0.07), ("tsp", 41, 1, 0.3),
                 ("cvrp", 50, 3, 0.07), ("cvrp", 10, 16, 0.3), ("cvrp", 20, 1, 0.07), ("cvrp", 100, 16, 0.3)]


@pytest.mark.parametrize("problem,N,nc,std", CLUSTER_CASES)
def test_cluster_instance_by_instance(problem, N, nc, std):
    ref, loc, depot, demand = _generate(problem, 1, 4, N, nc, 0.2, 0.8, std, seed=2 ** 33 + N + nc)
    clamped = _check_points(loc, ref["node"], ref["gauss"], "loc")
    if problem == "cvrp":
        # the depot is the point at depot_idx of the N + 1 drawn together; the rest keep their order (a wrong index
        # shifts the nodes and fails the comparison above)
        assert len(set(ref["depot_idx"].tolist())) > 1 or N == 10
        clamped += _check_points(depot, ref["depot"], ref["depot_gauss"], "depot")
        assert np.array_equal(demand.cpu().numpy(), ref["demand"])
    if std > 0.1:
        assert clamped > 0


@pytest.mark.parametrize("problem,N,nc", [("tsp", 21, 1), ("tsp", 100, 3), ("tsp", 9, 16), ("cvrp", 20, 1), ("cvrp", 50, 4)])
def test_mixed_instance_by_instance(problem, N, nc):
    ref, loc, depot, demand = _generate(problem, 2, 4, N, nc, 0.2, 0.8, 0.07, seed=77 + N)
    assert (ref["mutated"].sum(1) == N // 2).all()
    _check_points(loc, ref["node"], ref["gauss"], "loc")    # unmutated points bit for bit: the right half was redrawn
    if problem == "cvrp":
        _check_points(depot, ref["depot"], ref["depot_gauss"], "depot")
        assert np.array_equal(demand.cpu().numpy(), ref["demand"])


def test_generator_argument_checks():
    import ctypes as C
    from elg_b200 import _lib
    from elg_b200.generate_data import generate_tsp_data
    with pytest.raises(_lib.ElgError, match="n_cluster"):
        generate_tsp_data(2, 20, dict(DIST, data_type="cluster", n_cluster=17), seed=1)
    with pytest.raises(_lib.ElgError, match="n_cluster"):
        generate_tsp_data(2, 20, dict(DIST, data_type="mixed", n_cluster_mix=0), seed=1)
    with pytest.raises(_lib.ElgError, match="too large"):
        generate_tsp_data(1, 17100, DIST, seed=1)            # (3 N + 2) floats of shared memory > 200 KB
    generate_tsp_data(1, 17000, DIST, seed=1)                # just inside
    node = torch.empty((1, 20, 2), device="cuda:0")
    rc = _lib.lib.elg_generate_problems(_lib.ELG_TSP, 3, 1, 20, 1, 0.2, 0.8, 0.07, 1.0, 1, None, C.c_void_p(node.data_ptr()),
                                        None, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc != 0 and b"data kind" in _lib.lib.elg_last_error()
