"""Edge cases of the CUDA path: tiny / ragged shapes against the oracle, and loud failures outside the envelope."""
import pytest
import torch

from helpers import compare_tours
from oracle import elg_oracle as O
from test_gpu_model_config import assert_kernel, expected_kernel, launched_kernels

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _run(kind, N, M, n, aug, gain=3.0, seed=1, attention="fp32"):
    from elg_b200 import engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict, synthetic_tsp_batch
    mp = dict(DEFAULT_MODEL_PARAMS[kind])
    sd = synthetic_state_dict(kind, seed=100 + seed, gain=gain)
    W = O.Weights(sd, kind, mp)
    if kind == "cvrp":
        b = synthetic_cvrp_batch(n, N, seed=seed)
        prob = O.load_cvrp(b["depot"], b["loc"], b["demand"], aug)
    else:
        prob = O.load_tsp(synthetic_tsp_batch(n, N, seed=seed), aug)
    perm = O.start_permutation(kind, N, M, seed=seed)
    ref_t, _, ref_r = O.rollout(W, prob, M, perm, "greedy")
    handle = engine.ModelHandle(kind, mp, sd, DEV, attention=attention)
    batch = engine.encode(handle, prob.xy.to(DEV), None if prob.demand is None else prob.demand.to(DEV))
    (tours16, reward, _, n_steps), kernels = launched_kernels(lambda: engine.rollout(batch, M, perm.tolist()))
    T = int(n_steps.max())
    return tours16[:, :, :T].long().cpu(), reward.cpu(), ref_t, ref_r, prob, kernels


def _kernel(kind, N, M, n, aug, attention):
    """The decode kernel the released configuration (local_size 40 / 30) runs this shape on."""
    from elg_b200.synth import DEFAULT_MODEL_PARAMS
    return expected_kernel(kind, DEFAULT_MODEL_PARAMS[kind]["local_size"][0], N + (1 if kind == "cvrp" else 0), attention, True,
                           n * aug, M, torch.cuda.get_device_properties(DEV).multi_processor_count)


@pytest.mark.parametrize("kind,N,M,n,aug", [
    ("cvrp", 5, 1, 3, 1),       # one POMO row, tiny instance (local neighbourhood smaller than k)
    ("cvrp", 7, 5, 2, 8),       # M not a multiple of 4
    ("cvrp", 45, 45, 1, 8),     # k = 40 < N: neighbour list truncation
    ("cvrp", 107, 9, 1, 1),     # largest resident instance at k = 40 (N+1 = 108)
    ("cvrp", 108, 9, 1, 1),     # smallest streaming instance at k = 40 (N+1 = 109)
    ("cvrp", 111, 9, 1, 1),     # N+1 = 112: streaming at k = 40, the largest node count the resident kernels have slots for
    ("cvrp", 112, 9, 1, 1),     # N+1 = 113: beyond the resident kernels' node slots
    ("tsp", 4, 4, 2, 1),
    ("tsp", 31, 31, 1, 8),      # k = 30 = N-1
    ("tsp", 112, 7, 1, 1),      # resident limit
    ("tsp", 113, 7, 1, 1),      # streaming
    ("tsp", 129, 129, 1, 1),    # 5 mask words, M > 128
])
def test_ragged_shapes_match_oracle(kind, N, M, n, aug):
    tours, reward, ref_t, ref_r, prob, kernels = _run(kind, N, M, n, aug)
    assert_kernel(kernels, _kernel(kind, N, M, n, aug, "fp32"))
    frac, same = compare_tours(tours, ref_t)
    assert frac >= 0.9, frac
    assert ((reward - ref_r).abs() / ref_r.abs())[same].max() < 1e-4
    if kind == "cvrp":
        O.check_feasible_cvrp(tours, prob.demand)
    else:
        assert torch.equal(tours.sort(dim=2)[0], torch.arange(N).expand_as(tours))


@pytest.mark.parametrize("kind,N,M,n,aug", [
    ("cvrp", 112, 9, 1, 1),     # N+1 = 113: one key tile with 113 live keys, one row tile with 9 live rows
    ("cvrp", 128, 40, 1, 8),    # N+1 = 129: the second key tile holds a single node
    ("cvrp", 200, 130, 1, 1),   # two row tiles (128 + 2 rows), two key tiles
    ("cvrp", 300, 64, 1, 8),    # three key tiles, neighbour lists of more than two 128-entry chunks late in the rollout
    ("tsp", 113, 7, 1, 1),
    ("tsp", 129, 129, 1, 1),    # 2 row tiles, 2 key tiles
    ("tsp", 260, 50, 1, 8),
])
def test_ragged_shapes_streamed_tensor_core_kernel(kind, N, M, n, aug):
    """Large instances on the streamed tensor-core kernel (rollout_stc.cu; attention = auto) against the oracle."""
    tours, reward, ref_t, ref_r, prob, kernels = _run(kind, N, M, n, aug, attention="auto")
    assert_kernel(kernels, "rollout_stc_kernel<%d>" % (1 if kind == "cvrp" else 0))
    frac, same = compare_tours(tours, ref_t)
    assert frac >= 0.9, frac
    assert ((reward - ref_r).abs() / ref_r.abs())[same].max() < 1e-4
    if kind == "cvrp":
        O.check_feasible_cvrp(tours, prob.demand)
    else:
        assert torch.equal(tours.sort(dim=2)[0], torch.arange(N).expand_as(tours))


def test_streamed_kernel_is_the_one_that_runs():
    """The dispatch really takes the streamed tensor-core kernel for a large greedy rollout: same tours as the fp32-pipe
    kernel, and the scratch it needs was requested."""
    from elg_b200 import _lib, engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS
    desc = engine.make_desc("cvrp", dict(DEFAULT_MODEL_PARAMS["cvrp"]))
    assert int(_lib.lib.elg_et_bytes(desc, 8, 201)) == 8 * 2 * 3 * 65536
    assert int(_lib.lib.elg_rollout_ws_bytes(desc, 8, 200, 201)) > 0 and int(_lib.lib.elg_rollout_ws_bytes(desc, 8, 100, 101)) == 0
    a = _run("cvrp", 150, 60, 1, 8, attention="auto")
    b = _run("cvrp", 150, 60, 1, 8, attention="fp32")
    assert_kernel(a[5], "rollout_stc_kernel<1>")
    assert_kernel(b[5], "rollout_kernel<1, 6, false>")
    frac, _ = compare_tours(a[0], b[0])
    assert frac >= 0.97, frac


@pytest.mark.parametrize("kind,N,M,n,aug", [
    ("cvrp", 5, 1, 3, 1),       # N+1 = 6 -> one 16-column MMA tile, one live TMEM lane
    ("cvrp", 7, 5, 2, 8),
    ("cvrp", 15, 15, 2, 8),     # N+1 = 16: no padded key columns
    ("cvrp", 45, 45, 1, 8),     # k = 40 < N; rows in two TMEM lane quadrants
    ("cvrp", 70, 66, 1, 8),     # rows in three quadrants, M not a multiple of 4
    ("cvrp", 107, 107, 1, 1),   # resident limit at k = 40 (N+1 = 108), 107 rows in one CTA
    ("tsp", 4, 4, 2, 1),
    ("tsp", 31, 31, 1, 8),
    ("tsp", 100, 100, 1, 8),
    ("tsp", 112, 112, 1, 1),    # 112 nodes, 112 rows: every TMEM column of the S buffers in use
])
def test_ragged_shapes_tensor_core_kernel(kind, N, M, n, aug):
    tours, reward, ref_t, ref_r, prob, kernels = _run(kind, N, M, n, aug, attention="tensor")
    want = _kernel(kind, N, M, n, aug, "tensor")
    assert want.startswith("rollout_tc_kernel<")
    assert_kernel(kernels, want)
    frac, same = compare_tours(tours, ref_t)
    assert frac >= 0.9, frac
    assert ((reward - ref_r).abs() / ref_r.abs())[same].max() < 1e-4
    if kind == "cvrp":
        O.check_feasible_cvrp(tours, prob.demand)
    else:
        assert torch.equal(tours.sort(dim=2)[0], torch.arange(N).expand_as(tours))


def test_automatic_kernel_choice_agrees_with_both():
    """160 aug-instances >= 148 SMs -> the library picks the tensor-core kernel by itself; forcing either kernel gives the
    same tours on (all but a handful of) rows and the same best costs."""
    from elg_b200 import engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict
    mp, sd = dict(DEFAULT_MODEL_PARAMS["cvrp"]), synthetic_state_dict("cvrp", seed=7, gain=3.0)
    b = synthetic_cvrp_batch(20, 50, seed=3)
    prob = O.load_cvrp(b["depot"], b["loc"], b["demand"], 8)
    perm = O.start_permutation("cvrp", 50, 50, seed=3)
    out = {}
    for att in ("auto", "tensor", "fp32"):
        h = engine.ModelHandle("cvrp", mp, sd, DEV, attention=att)
        batch = engine.encode(h, prob.xy.to(DEV), prob.demand.to(DEV))
        t16, rew, _, ns = engine.rollout(batch, 50, perm.tolist())
        out[att] = (t16[:, :, :int(ns.max())].long().cpu(), rew.cpu())
    assert torch.equal(out["auto"][0], out["tensor"][0]) and torch.equal(out["auto"][1], out["tensor"][1])
    frac, same = compare_tours(out["tensor"][0], out["fp32"][0])
    assert frac >= 0.97, frac
    best_t, best_f = out["tensor"][1].max(1)[0], out["fp32"][1].max(1)[0]
    assert ((best_t - best_f).abs() / best_f.abs()).max() < 2e-3
    O.check_feasible_cvrp(out["tensor"][0], prob.demand)


def test_out_of_envelope_fails_loudly():
    from elg_b200 import _lib, engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    mp = dict(DEFAULT_MODEL_PARAMS["tsp"])
    handle = engine.ModelHandle("tsp", mp, synthetic_state_dict("tsp"), DEV)
    xy = torch.rand(1, 130, 2, device=DEV)
    batch = engine.encode(handle, xy)
    with pytest.raises(_lib.ElgError):                                   # sampling is limited to 128 nodes
        engine.rollout(batch, 8, list(range(8)), mode="sample")
    with pytest.raises(ValueError):
        engine.rollout(batch, 8, list(range(7)))                          # wrong start-node count
    with pytest.raises(_lib.ElgError):
        engine.encode(handle, torch.rand(1, 20, 2))                       # CPU tensor: no CPU path
    big = torch.rand(1, 8200, 2, device=DEV)
    with pytest.raises(_lib.ElgError):                                   # beyond ELG_MAX_NODES
        engine.rollout(engine.encode(handle, big), 4, [0, 1, 2, 3])


@pytest.mark.parametrize("kind", ["cvrp", "tsp"])
def test_model_without_local_policy_matches_oracle(kind):
    """The reference's decoder before add_local_policy (self.local False, CVRP/models.py:409): global policy + distance
    penalty.  The drop-in model packs no local weights, the library zeroes the local tables."""
    import random
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict, synthetic_tsp_batch
    mp = dict(DEFAULT_MODEL_PARAMS[kind])
    sd = {k: v for k, v in synthetic_state_dict(kind, seed=9, gain=3.0).items() if ".local_polic" not in k}
    if kind == "cvrp":
        from elg_b200.cvrp import CVRPEnv as Env, CVRPModel as Model, rollout
        data = synthetic_cvrp_batch(3, 30, seed=2)
        prob = O.load_cvrp(data["depot"], data["loc"], data["demand"], 8)
    else:
        from elg_b200.tsp import TSPEnv as Env, TSPModel as Model, rollout
        data = synthetic_tsp_batch(3, 30, seed=2)
        prob = O.load_tsp(data, 8)
    model = Model(**mp)                      # no add_local_policy
    model.load_state_dict(sd)
    model = model.to(DEV)
    env = Env(30, DEV)
    env.load_random_problems(data, 8)
    reset_state, _, _ = env.reset()
    random.seed(3)
    model.pre_forward(reset_state)
    tours, _, reward = rollout(model, env, "greedy")
    W = O.Weights(sd, kind, dict(mp, ensemble=False))
    ref_t, _, ref_r = O.rollout(W, prob, 30, O.start_permutation(kind, 30, 30, seed=3), "greedy")
    T = max(tours.shape[2], ref_t.shape[2])
    a = torch.zeros(24, 30, T, dtype=torch.long); a[:, :, :tours.shape[2]] = tours.cpu()
    b = torch.zeros(24, 30, T, dtype=torch.long); b[:, :, :ref_t.shape[2]] = ref_t
    same = (a == b).all(dim=2)
    assert float(same.float().mean()) >= 0.97
    assert float(((reward.cpu() - ref_r).abs() / ref_r.abs())[same].max()) < 1e-4


@pytest.mark.parametrize("kind", ["cvrp", "tsp"])
def test_encoder_tables_do_not_depend_on_the_batch(kind):
    """The persistent encoder kernels (tc_gemm_kernel, tc_ffn_kernel: one CTA per SM walking 128-row tiles through mbarrier
    rings) give every instance the same tables whether it is encoded in a batch of 200 (20,200 rows = 158 tiles: several
    tiles per CTA, a partial last tile, instances straddling tile boundaries) or in a batch of 3 (one CTA, partial tiles)."""
    from elg_b200 import engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict, synthetic_tsp_batch
    mp = dict(DEFAULT_MODEL_PARAMS[kind])
    handle = engine.ModelHandle(kind, mp, synthetic_state_dict(kind, seed=11, gain=2.0), DEV)
    n = 200
    if kind == "cvrp":
        d = {k: v.to(DEV) for k, v in synthetic_cvrp_batch(n, 100, seed=7).items()}
        xy, dem = engine.load_problems("cvrp", d["loc"], d["depot"], d["demand"], aug=1)
    else:
        xy, dem = engine.load_problems("tsp", synthetic_tsp_batch(n, 100, seed=7).to(DEV), aug=1)
    big = engine.encode(handle, xy, dem)
    torch.cuda.synchronize()
    for lo in (0, 98, 197):
        sl = slice(lo, lo + 3)
        small = engine.encode(handle, xy[sl].contiguous(), None if dem is None else dem[sl].contiguous())
        torch.cuda.synchronize()
        for name in ("enc", "k", "v", "qtab", "eb") + (("qfirst",) if kind == "tsp" else ()):
            a, b = getattr(big, name)[sl], getattr(small, name)
            assert torch.equal(a, b), (name, lo, float((a - b).abs().max()))


@pytest.mark.parametrize("kind", ["cvrp", "tsp"])
def test_decoder_tables_with_separately_allocated_buffers(kind):
    """elg_encode writes K', V, qtab (qfirst) in ONE GEMM launch when the caller's buffers are equally spaced planes (the
    Python engine's are) and in one launch per table otherwise (any C-ABI caller with its own allocations): same bits."""
    import ctypes as C
    from elg_b200 import _lib, engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict, synthetic_tsp_batch
    mp = dict(DEFAULT_MODEL_PARAMS[kind])
    handle = engine.ModelHandle(kind, mp, synthetic_state_dict(kind, seed=12, gain=2.0), DEV)
    if kind == "cvrp":
        d = {k: v.to(DEV) for k, v in synthetic_cvrp_batch(5, 60, seed=8).items()}
        xy, dem = engine.load_problems("cvrp", d["loc"], d["depot"], d["demand"], aug=8)
    else:
        xy, dem = engine.load_problems("tsp", synthetic_tsp_batch(5, 60, seed=8).to(DEV), aug=8)
    ref = engine.encode(handle, xy, dem)
    torch.cuda.synchronize()
    other = engine.EncodedBatch(handle, xy, dem)
    n = ref.k.numel()
    buf = torch.empty(4 * n + 4096, device=DEV)               # tables carved out at irregular (16-byte aligned) offsets
    other.k = buf[0:n].view_as(ref.k)
    other.v = buf[n + 256:2 * n + 256].view_as(ref.k)
    other.qtab = buf[2 * n + 1024:3 * n + 1024].view_as(ref.k)
    if kind == "tsp":
        other.qfirst = buf[3 * n + 2048:4 * n + 2048].view_as(ref.k)
    assert other.v.data_ptr() - other.k.data_ptr() != other.qtab.data_ptr() - other.v.data_ptr()
    other.tables = _lib.Tables(*[engine._ptr(x).value for x in (other.xy, other.demand, other.unscaled, other.enc, other.k, other.v,
                                                                 other.e, other.eb, other.qtab, other.qfirst, other.nbr, other.et, None)])
    nbytes = int(_lib.lib.elg_encode_workspace_bytes(handle.desc, other.B, other.N1))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    with torch.cuda.device(DEV):
        _lib.check(_lib.lib.elg_encode(handle.desc, engine._ptr(handle.weights), engine._ptr(handle.derived), other.tables, other.B,
                                       other.N1, engine._ptr(ws), nbytes, engine._stream(torch.device(DEV))))
    torch.cuda.synchronize()
    for name in ("enc", "k", "v", "qtab", "eb", "e") + (("qfirst",) if kind == "tsp" else ()):
        assert torch.equal(getattr(ref, name), getattr(other, name)), name
