"""Sampled decisions of the fp32-pipe decode kernel replayed one by one against the fp64 oracle.

A sampled decision of row m of aug-instance b draws u = sample_uniform(seed, b * M + m, step) (philox_ref.py) and takes
the first node j, in node-index order, with p[j] > 0 and u <= F[j], F the CDF of softmax(logits).  The fused rollout
uses the tour position t as the step (cvrp: t = 0 depot and t = 1 start node are forced, policies from t = 2; tsp:
policies from t = 1); elg_decode_step uses the caller's step.  Every check below teacher-forces the oracle on the
kernel's own choices and asserts, at every policy step of every unfinished row, F64[j - 1] - delta <= u <= F64[j] + delta
with delta two of the parity suite's logit bars mapped into CDF space (|dF| <= 2 max |dlogit|).  A draw with a wrong
counter, a wrong row index or a CDF scanned in another order lands outside that window for most decisions.

Instances are synthetic random points, so there are no distance ties.  Sampling is implemented up to N1 = 128, on the
resident and on the streaming template of rollout_kernel; every instantiation is identified through torch.profiler.
"""
import numpy as np
import pytest
import torch

from philox_ref import U_BOTTOM, U_TOP, sample_uniform
from test_gpu_model_config import assert_kernel, expected_kernel, launched_kernels, maxe, RESIDENT_MAX_N1
from helpers import Golden
from oracle import elg_oracle as O

DEV = "cuda:0"
LOGP_REL = 5e-3               # test_gpu_train's bar on the rollout's log-likelihood
AMBIGUOUS_MAX = 0.05          # share of decisions allowed within delta of an interval end


def delta(clip):
    return 4e-3 * clip / 50.0


# ---------------------------------------------------------------------------------------------------- the check
def check_draws(p64, sel, u, live, clip, where=""):
    """p64 (R, N1) fp64 probabilities, sel (R,) the kernel's nodes, u (R,) the uniforms, live (R,) rows that decided.
    Asserts the inverse-CDF window on every live row; returns (live rows within delta of an interval end, live rows)."""
    d = delta(clip)
    pj = p64.gather(1, sel[:, None]).squeeze(1)
    Fj = p64.cumsum(1).gather(1, sel[:, None]).squeeze(1)
    Fprev = Fj - pj
    u = torch.as_tensor(np.asarray(u, dtype=np.float64))
    bad = live & ~((pj > 0) & (Fprev - d <= u) & (u <= Fj + d))
    if bad.any():
        r = int(bad.nonzero()[0, 0])
        raise AssertionError("%s: row %d drew node %d with u=%.9f outside [F(j-1), F(j)] = [%.9f, %.9f] (p=%.3g), %d of %d rows"
                             % (where, r, int(sel[r]), float(u[r]), float(Fprev[r]), float(Fj[r]), float(pj[r]),
                                int(bad.sum()), int(live.sum())))
    near = live & (((u - Fprev) < d) | ((Fj - u) < d))
    return int(near.sum()), int(live.sum())


def replay_rollout(W, prob, M, perm, tours, seed, clip):
    """Teacher-force the fp64 oracle on the kernel's tours (B, M, T): check every sampled decision, return
    (logp64 (B, M): the sum of log p64 over the policy steps of unfinished rows, decisions within delta, decisions,
    per-step record {t: (p64 (B, M, N1), masked)} of the states)."""
    B, _, T = tours.shape
    cache = O.decoder_cache(W, O.encode(W, prob))
    grow = np.arange(B * M, dtype=np.uint64)
    logp = torch.zeros(B, M, dtype=torch.float64)
    near = total = 0
    rec = {}
    cvrp = W.kind == "cvrp"
    st = O.cvrp_reset(prob, M) if cvrp else O.tsp_reset(prob, M)
    for t in range(T):
        sel = tours[:, :, t]
        forced = t < (2 if cvrp else 1)
        if forced:
            want = torch.zeros_like(sel) if (cvrp and t == 0) else perm[None, :].expand(B, M)
            assert torch.equal(sel, want), t
            if not cvrp:
                O.set_first(W, cache, sel)
        else:
            live = ~st.finished if cvrp else torch.ones(B, M, dtype=torch.bool)
            masked = st.masked.clone()
            logits = O.decode_logits(W, prob, cache, st.cur, masked, st.load if cvrp else None)
            p64 = torch.softmax(logits, dim=2)
            rec[t] = (p64, masked)
            u = sample_uniform(seed, grow, t).reshape(B * M)
            n, c = check_draws(p64.reshape(B * M, -1), sel.reshape(-1), u, live.reshape(-1), clip, "t=%d" % t)
            near, total = near + n, total + c
            if cvrp:
                assert bool((sel[~live] == 0).all()), "a finished row left the depot at t=%d" % t
            lp = p64.gather(2, sel[:, :, None]).squeeze(2).log()
            logp += torch.where(live, lp, torch.zeros_like(lp))
        if cvrp:
            O.cvrp_env_step(prob, st, sel)
        else:
            O.tsp_env_step(prob, st, sel)
    if cvrp:
        assert bool(st.finished.all())
    return logp, near, total, rec


# ---------------------------------------------------------------------------------------------------- cases
def _case(cid, kind, k, N, M, n=1, aug=8, xi=-1.0, clip=50.0, ensemble=True, gain=3.0, seed=1, edges=()):
    return dict(id=cid, kind=kind, k=k, N=N, M=M, n=n, aug=aug, xi=xi, clip=clip, ensemble=ensemble, gain=gain,
                seed=seed, edges=edges)


def n1(c):
    return c["N"] + (1 if c["kind"] == "cvrp" else 0)


CASES = [
    # every rollout_kernel<P, MAXE, RESIDENT> instantiation: resident at the bucket's limit, streaming in (limit, 128]
    _case("cvrp-me4-res", "cvrp", 31, 111, 24, seed=1),
    _case("cvrp-me4-stream", "cvrp", 31, 127, 24, seed=2),            # N1 128: the sampling limit
    _case("cvrp-me6-res", "cvrp", 40, 107, 24, seed=3),
    _case("cvrp-me6-stream", "cvrp", 40, 112, 24, seed=4),
    _case("cvrp-me8-res", "cvrp", 50, 103, 24, seed=5),
    _case("cvrp-me8-stream", "cvrp", 50, 104, 24, seed=6),
    _case("tsp-me4-res", "tsp", 30, 112, 24, seed=7),
    _case("tsp-me4-stream", "tsp", 30, 128, 24, seed=8),
    _case("tsp-me6-res", "tsp", 33, 108, 24, seed=9),
    _case("tsp-me6-stream", "tsp", 33, 109, 24, seed=10),
    _case("tsp-me8-res", "tsp", 49, 104, 24, seed=11),
    _case("tsp-me8-stream", "tsp", 49, 128, 24, seed=12),
    # row tiling: B = 1 runs 25 tiles of 4 rows, B = 64 two tiles of 52, M = 30 / 37 leave a partial last tile
    _case("cvrp-b1-m100", "cvrp", 40, 100, 100, aug=1, seed=13),
    _case("tsp-b64-m100", "tsp", 30, 100, 100, n=8, seed=14),
    _case("cvrp-m30", "cvrp", 40, 50, 30, seed=15),
    _case("tsp-m37", "tsp", 30, 50, 37, seed=16),
    # global policy and distance penalty only; other runtime constants
    _case("cvrp-no-local", "cvrp", 40, 60, 24, ensemble=False, seed=17),
    _case("tsp-xi-clip", "tsp", 30, 60, 24, xi=0.5, clip=10.0, seed=18),
    # draws at the top of the CDF (u = 1.0): (b, m, t) found by an exhaustive Philox search over seeds
    _case("tsp-top-225", "tsp", 30, 50, 50, seed=225, edges=((2, 11, 6),)),
    _case("tsp-top-512", "tsp", 30, 50, 50, seed=512, edges=((3, 36, 14),)),
    _case("cvrp-top-225", "cvrp", 40, 50, 50, seed=225, edges=((2, 11, 6),)),
    _case("cvrp-top-512", "cvrp", 40, 50, 50, seed=512, edges=((3, 36, 14),)),
]


def _model(c):
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    mp = dict(DEFAULT_MODEL_PARAMS[c["kind"]], local_size=[c["k"]], xi=c["xi"], logit_clipping=c["clip"],
              ensemble=c["ensemble"])
    return mp, synthetic_state_dict(c["kind"], seed=200 + c["seed"], gain=c["gain"], model_params=mp)


def _problem(kind, n, N, aug, seed):
    """fp32 aug-instances for the device and the same coordinates in fp64 for the oracle."""
    from elg_b200.synth import synthetic_cvrp_batch, synthetic_tsp_batch
    if kind == "cvrp":
        d = synthetic_cvrp_batch(n, N, seed=seed)
        p32 = O.load_cvrp(d["depot"], d["loc"], d["demand"], aug)
    else:
        p32 = O.load_tsp(synthetic_tsp_batch(n, N, seed=seed), aug)
    xy = p32.xy.double()
    p64 = O.Problem(kind, xy, None if p32.demand is None else p32.demand.double(), O.pairwise_dist(xy), None, aug)
    return p32, p64


def test_case_table_covers_every_instantiation():
    """The -me cases launch each of the 12 instantiations once: resident at the bucket's limit, streaming above it."""
    want = {"rollout_kernel<%d, %d, %s>" % (p, m, r) for p in (0, 1) for m in (4, 6, 8) for r in ("true", "false")}
    inst = [c for c in CASES if "-me" in c["id"]]
    assert {expected_kernel(c["kind"], c["k"], n1(c), "fp32", True) for c in inst} == want and len(inst) == 12
    for c in inst:
        top = RESIDENT_MAX_N1[maxe(c["kind"], c["k"])]
        assert n1(c) == top if c["id"].endswith("-res") else top < n1(c) <= 128, c["id"]
    assert all(n1(c) <= 128 for c in CASES) and any(n1(c) == 128 for c in inst)


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=lambda c: c["id"])
def test_sampled_rollout_replays_against_fp64(c):
    from elg_b200 import engine
    kind, M = c["kind"], c["M"]
    mp, sd = _model(c)
    p32, p64 = _problem(kind, c["n"], c["N"], c["aug"], 300 + c["seed"])
    B = p32.xy.shape[0]
    perm = O.start_permutation(kind, c["N"], M, seed=c["seed"])
    handle = engine.ModelHandle(kind, mp, sd, DEV)
    assert handle.has_local == c["ensemble"]
    batch = engine.encode(handle, p32.xy.to(DEV), None if p32.demand is None else p32.demand.to(DEV))
    seed = c["seed"]
    (t16, reward, logp, n_steps), found = launched_kernels(
        lambda: engine.rollout(batch, M, perm.tolist(), mode="sample", seed=seed))
    assert_kernel(found, expected_kernel(kind, c["k"], n1(c), "fp32", True))
    T = int(n_steps.max())
    tours, logp = t16[:, :, :T].long().cpu(), logp.double().cpu()
    # the same seed gives the same tours
    t16b, _, logpb, _ = engine.rollout(batch, M, perm.tolist(), mode="sample", seed=seed)
    assert torch.equal(t16b[:, :, :T].long().cpu(), tours) and torch.equal(logpb.double().cpu(), logp)
    W = O.Weights(sd, kind, mp, dtype=torch.float64)
    ref, near, total, rec = replay_rollout(W, p64, M, perm, tours, seed, c["clip"])
    assert total > 0 and near < AMBIGUOUS_MAX * total, (near, total)
    assert float((logp - ref).abs().max()) < LOGP_REL * max(1.0, float(ref.abs().max()))
    if kind == "cvrp":
        O.check_feasible_cvrp(tours, p64.demand)
    else:
        assert torch.equal(tours.sort(dim=2)[0], torch.arange(n1(c)).expand_as(tours))
    for b, m, t in c["edges"]:
        assert sample_uniform(seed, b * M + m, t) == U_TOP
        p, masked = rec[t]
        cand = (~masked[b, m]).nonzero().flatten()
        assert cand.numel() >= 2
        j = int(tours[b, m, t])               # the window at u = 1: F64[j] >= 1 - delta, p64[j] > 0 (replay_rollout)
        pj = float(p[b, m, j])
        if pj < 0.9:                                                   # the step's log p is part of the row's logp
            assert abs(float(logp[b, m] - ref[b, m])) < 0.5 * abs(np.log(pj)), (float(logp[b, m]), float(ref[b, m]), pj)


# ---------------------------------------------------------------------------------------------------- single steps
DECODE_GOLDEN = ["cvrp_n20", "cvrp_n50", "cvrp_n100", "tsp_n20", "tsp_n50", "tsp_n100"]
# (golden, step, seed, grow, uniform): grow = b * M + m of a row whose draw is the largest (U_TOP) or the smallest
# (U_BOTTOM) uniform at (seed, step), found by an exhaustive Philox search over seeds
EDGE_DRAWS = [
    ("cvrp_n20", 5, 192360, 0, U_TOP), ("cvrp_n20", 12, 65787, 65, U_TOP),
    ("cvrp_n50", 10, 307990, 37, U_TOP), ("cvrp_n50", 30, 785914, 7, U_TOP),
    ("cvrp_n100", 7, 94404, 10, U_TOP), ("cvrp_n100", 40, 43490, 23, U_TOP),
    ("tsp_n20", 3, 187873, 20, U_TOP), ("tsp_n20", 10, 307990, 37, U_TOP),
    ("tsp_n50", 10, 307990, 37, U_TOP), ("tsp_n50", 30, 785914, 7, U_TOP),
    ("tsp_n100", 7, 94404, 10, U_TOP), ("tsp_n100", 40, 43490, 23, U_TOP),
    ("cvrp_n50", 10, 540583, 31, U_BOTTOM), ("tsp_n50", 10, 540583, 31, U_BOTTOM),
]


def _golden_state(name):
    """The recorded aug-instances of a golden case on the device and the fp64 oracle, with a probability function."""
    from elg_b200 import engine
    g = Golden(name)
    rows = g.rows_b
    prob64 = g.oracle_problem(torch.float64)
    sub = O.Problem(prob64.kind, prob64.xy[rows], None if prob64.demand is None else prob64.demand[rows],
                    prob64.dist[rows], None, 1)
    W = O.Weights(g.state_dict(), g.kind, g.model_params(), dtype=torch.float64)
    cache = O.decoder_cache(W, O.encode(W, sub))
    first = g.tours()[rows, :, 0] if g.kind == "tsp" else None
    if first is not None:
        O.set_first(W, cache, first)
    prob32 = g.oracle_problem()
    handle = engine.ModelHandle(g.kind, g.model_params(), g.state_dict(), DEV)
    batch = engine.encode(handle, prob32.xy[rows].contiguous().to(DEV),
                          None if prob32.demand is None else prob32.demand[rows].contiguous().to(DEV))
    return dict(g=g, W=W, sub=sub, cache=cache, first=first, batch=batch)


def _decode(gs, t, seed, step):
    """(selected (B, M), prob (B, M), p64 (B, M, N1), live (B, M), masked) of one sampled decode step at state t."""
    from elg_b200 import engine
    g = gs["g"]
    s = g.step(t)
    load = s["load"] if g.kind == "cvrp" else None
    logits = O.decode_logits(gs["W"], gs["sub"], gs["cache"], s["cur"], s["masked"], load)
    p64 = torch.softmax(logits, dim=2)
    bits = engine.pack_mask_bits(s["masked"].to(DEV))
    sel, pr, _ = engine.decode_step(gs["batch"], g.M, s["cur"].to(DEV), bits, load=None if load is None else load.to(DEV),
                                    first=None if gs["first"] is None else gs["first"].to(DEV), mode="sample",
                                    seed=seed, step=step)
    live = torch.ones(s["cur"].shape, dtype=torch.bool)    # a single step decides every row (finished: the depot)
    return sel.cpu(), pr.double().cpu(), p64, live, s["masked"]


def _check_step(gs, t, seed, step, clip):
    sel, pr, p64, live, masked = _decode(gs, t, seed, step)
    B, M = sel.shape
    u = sample_uniform(seed, np.arange(B * M, dtype=np.uint64), step)
    near, total = check_draws(p64.reshape(B * M, -1), sel.reshape(-1), u, live.reshape(-1), clip, "t=%d" % t)
    want = p64.gather(2, sel[:, :, None]).squeeze(2)
    assert float(((pr - want).abs() / want).max()) < 4e-3
    return sel, pr, p64, masked, near, total


@pytest.mark.gpu
@pytest.mark.parametrize("name", DECODE_GOLDEN)
def test_decode_step_draws_at_golden_states(name):
    gs = _golden_state(name)
    g = gs["g"]
    clip = float(g.model_params()["logit_clipping"])
    near = total = moved = 0
    steps = g.steps[:: max(1, len(g.steps) // 5)]
    for i, t in enumerate(steps):
        for seed in (7 + i, 2 ** 40 + 3 * i):                 # a seed above 2^32 exercises the key's high word
            sel, _, p64, _, n, c = _check_step(gs, t, seed, t, clip)
            near, total = near + n, total + c
            again, _, _, _, _, _ = _check_step(gs, t, seed, t, clip)
            assert torch.equal(again, sel)                      # the same (seed, step): the same draws
            # another step draws other uniforms: wherever the new uniform lies outside the first node's CDF interval
            # (by more than delta), the node must change.  Near-deterministic rows keep their node either way.
            other, _, _, _, _, _ = _check_step(gs, t, seed, t + 1000, clip)
            B, M = sel.shape
            u2 = torch.as_tensor(sample_uniform(seed, np.arange(B * M, dtype=np.uint64), t + 1000).astype(np.float64))
            Fj = p64.cumsum(2).gather(2, sel[:, :, None]).squeeze(2).reshape(-1)
            Fprev = Fj - p64.gather(2, sel[:, :, None]).squeeze(2).reshape(-1)
            must = ((u2 < Fprev - delta(clip)) | (u2 > Fj + delta(clip))).reshape(B, M)
            assert bool((other[must] != sel[must]).all())
            moved += int(must.sum())
    assert total > 0 and near < AMBIGUOUS_MAX * total, (near, total)
    assert moved > 0                                            # the step word reaches the draw


@pytest.mark.gpu
@pytest.mark.parametrize("edge", EDGE_DRAWS, ids=lambda e: "%s-t%d-%s" % (e[0], e[1], "top" if e[4] == 1 else "bottom"))
def test_decode_step_at_the_ends_of_the_cdf(edge):
    name, t, seed, grow, uval = edge
    assert sample_uniform(seed, grow, t) == uval
    gs = _golden_state(name)
    g = gs["g"]
    sel, pr, p64, masked, _, _ = _check_step(gs, t, seed, t, float(g.model_params()["logit_clipping"]))
    b, m = divmod(grow, g.M)
    cand = (~masked[b, m]).nonzero().flatten()
    j, pj = int(sel[b, m]), float(p64[b, m, int(sel[b, m])])
    # _check_step asserted the window: at u = 1 a node of positive probability with F64[j] >= 1 - delta, in fp32 the
    # first one whose running sum reaches the total; at u = 2^-25 one with F64[j - 1] <= 2^-25 + delta
    if uval == U_TOP:
        assert float(p64[b, m].cumsum(0)[j]) >= 1 - delta(50.0)
    else:
        assert float(p64[b, m, :j].sum()) <= 2.0 ** -25 + delta(50.0), (j, cand.tolist())
    assert cand.numel() == 1 or pj > 0.996 or float(pr[b, m]) < 1.0, (j, pj)     # its own probability, not 1
    assert abs(float(pr[b, m]) - pj) < 4e-3 * pj


@pytest.mark.gpu
def test_decode_step_draws_at_a_streaming_size_state():
    """One state of a 120-customer cvrp instance (N1 = 121: the streaming template for local_size 40)."""
    from elg_b200 import engine
    c = _case("cvrp-stream-step", "cvrp", 40, 120, 16, seed=19)
    mp, sd = _model(c)
    p32, p64 = _problem("cvrp", 1, 120, 8, 319)
    perm = O.start_permutation("cvrp", 120, 16, seed=19)
    W = O.Weights(sd, "cvrp", mp, dtype=torch.float64)
    rec = {}

    def hook(st, logits):
        if st.count == 30:
            rec.update(cur=st.cur.clone(), masked=st.masked.clone(), load=st.load.clone(), p=torch.softmax(logits, 2))
    O.rollout(W, p64, 16, perm, "greedy", hook=hook, max_steps=31)
    handle = engine.ModelHandle("cvrp", mp, sd, DEV)
    batch = engine.encode(handle, p32.xy.to(DEV), p32.demand.to(DEV))
    bits = engine.pack_mask_bits(rec["masked"].to(DEV))
    B, M = rec["cur"].shape
    near = total = 0
    for seed, step in ((5, 30), (5, 31), (2 ** 33 + 1, 30)):
        (sel, pr, _), found = launched_kernels(lambda: engine.decode_step(
            batch, M, rec["cur"].to(DEV), bits, load=rec["load"].float().to(DEV), mode="sample", seed=seed, step=step))
        assert_kernel(found, "rollout_kernel<1, 6, false>")
        sel, pr = sel.cpu(), pr.double().cpu()
        u = sample_uniform(seed, np.arange(B * M, dtype=np.uint64), step)
        n, cnt = check_draws(rec["p"].reshape(B * M, -1), sel.reshape(-1), u, torch.ones(B * M, dtype=torch.bool), 50.0)
        near, total = near + n, total + cnt
        want = rec["p"].gather(2, sel[:, :, None]).squeeze(2)
        assert float(((pr - want).abs() / want).max()) < 4e-3
    assert near < AMBIGUOUS_MAX * total, (near, total)
