"""Model configurations the library accepts beyond the released config.yml, on every kernel they select.

check_desc admits local_size 1..63 (cvrp) / 1..64 (tsp), any xi and logit_clipping, positional off, 1..16 encoder layers
and any multiple of 128 for ff_hidden_dim.  The local sequence length KT (local_size, plus the depot for cvrp) picks the
template of every decode kernel (MAXE = 4 / 6 / 8 for KT <= 32 / 48 / 64) and moves the resident / streaming boundary;
ff_hidden_dim picks the fused or the two-GEMM feed-forward of the encoder.  Each case below names the exact kernel
instantiation it launches (read back through torch.profiler) and compares it with the fp64 oracle.

The CPU tests pin the parameter bounds, the resident boundaries and the coverage of the case table.
"""
import random
import re

import pytest
import torch

from helpers import compare_tours, tie_rows, top2_margin
from oracle import elg_oracle as O

DEV = "cuda:0"
LOGIT_MAX_ATOL = 2e-3        # test_gpu_parity's bars at logit_clipping 50; scaled by clip / 50 here
LOGIT_MEAN_ATOL = 3e-5
PROBLEM_ID = {"tsp": 0, "cvrp": 1}
N_RES_MAX = 112              # node slots of the resident kernels
RESIDENT_MAX_N1 = {4: 112, 6: 108, 8: 104}      # largest resident N1 per MAXE bucket (the tables + the largest row tile)


# ---------------------------------------------------------------------------------------- dispatch, restated
def local_len(kind, k):
    return k + (1 if kind == "cvrp" else 0)


def maxe(kind, k):
    kt = local_len(kind, k)
    return 4 if kt <= 32 else (6 if kt <= 48 else 8)


def is_resident(kind, k, N1):
    return N1 <= RESIDENT_MAX_N1[maxe(kind, k)]


def tc_maxe(kind, k):
    """MAXE of rollout_tc_kernel; 0 = the local sequence does not fit its tensor-memory plan (KT > 48)."""
    kt = local_len(kind, k)
    return 4 if kt <= 32 else (6 if kt <= 48 else 0)


def stc_eligible(kind, k, N1):
    """rollout_stc_kernel: large instances with a local sequence of at most 44 positions (greedy, fused rollouts)."""
    return N1 > N_RES_MAX and local_len(kind, k) <= 44


def expected_kernel(kind, k, N1, attention, fused, B=1, M=1, sms=148):
    """The decode kernel elg_rollout / elg_decode_step launch for this shape (rollout.cu launch_rollout)."""
    p = PROBLEM_ID[kind]
    res = is_resident(kind, k, N1)
    me = tc_maxe(kind, k)
    if attention != "fp32" and res and me:
        tiles = (M + 111) // 112
        if attention == "tensor" or B * tiles >= sms:
            return "rollout_tc_kernel<%d, %d, %d>" % (p, me, 112 if ((N1 + 15) & ~15) == 112 else 0)
    if fused and attention != "fp32" and stc_eligible(kind, k, N1):
        return "rollout_stc_kernel<%d>" % p
    return "rollout_kernel<%d, %d, %s>" % (p, maxe(kind, k), "true" if res else "false")


ALL_INSTANTIATIONS = ({"rollout_kernel<%d, %d, %s>" % (p, m, r) for p in (0, 1) for m in (4, 6, 8) for r in ("true", "false")} |
                      {"rollout_tc_kernel<%d, %d, %d>" % (p, m, n) for p in (0, 1) for m in (4, 6) for n in (112, 0)} |
                      {"rollout_stc_kernel<%d>" % p for p in (0, 1)})


# ---------------------------------------------------------------------------------------- kernel identity
_KERNEL = re.compile(r"elg::(rollout(?:_tc|_stc)?_kernel)<([^>]*)>")


def launched_kernels(fn):
    """Run fn() under torch.profiler (CUDA activity) -> (fn's result, set of the elg decode kernels that launched, written
    like 'rollout_kernel<1, 8, false>').  Fails when the profiler recorded no CUDA activity at all.

    In a long run of back-to-back sessions torch.profiler now and then hands back a session without any CUDA activity
    (observed on a B200 during the full GPU suite).  fn must therefore be repeatable -- every call here recomputes its
    outputs from unchanged inputs -- and is run again, in a fresh session, up to twice before the helper fails."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]
        if names:
            break
    assert names, "torch.profiler recorded no CUDA activity: cannot tell which kernel ran"
    found = set()
    for n in names:
        m = _KERNEL.search(n)
        if m:
            args = [re.sub(r"^\(\w+\)", "", a.strip()) for a in m.group(2).split(",")]
            found.add("%s<%s>" % (m.group(1), ", ".join(args)))
    return out, found


def assert_kernel(found, want):
    assert found == {want}, "expected %s to run, profiler saw %s" % (want, sorted(found))


# ---------------------------------------------------------------------------------------- case table
def _case(cid, kind, k, N, M, n=1, aug=8, xi=-1.0, clip=50.0, positional=True, gain=3.0, seed=1, tf_steps=36):
    return dict(id=cid, kind=kind, k=k, N=N, M=M, n=n, aug=aug, xi=xi, clip=clip, positional=positional, gain=gain,
                seed=seed, tf_steps=tf_steps)


CASES = [
    # cvrp: local_size at both sides of every MAXE bucket, the stc cut-off (K1 <= 44) and KT_MAX; per bucket N1 at the
    # largest resident value, one above it and 129 (two key tiles)
    _case("cvrp-k1-n20", "cvrp", 1, 20, 20, n=2, gain=2.0, seed=1),
    _case("cvrp-k8-n111", "cvrp", 8, 111, 24, gain=3.0, seed=2),                 # N1 112: largest resident, MAXE 4
    _case("cvrp-k8-n112", "cvrp", 8, 112, 24, gain=4.0, seed=3),                 # N1 113: streaming / stc
    _case("cvrp-k31-n128", "cvrp", 31, 128, 24, xi=0.0, gain=2.0, seed=4),       # KT 32, N1 129
    _case("cvrp-k31-n60", "cvrp", 31, 60, 30, xi=0.0, clip=10.0, gain=3.0, seed=5),
    _case("cvrp-k32-n107", "cvrp", 32, 107, 24, gain=4.0, seed=6),               # KT 33: MAXE 6, N1 108 largest resident
    _case("cvrp-k32-n108", "cvrp", 32, 108, 24, gain=2.0, seed=7),               # N1 109: streaming below N_RES_MAX
    _case("cvrp-k43-n128", "cvrp", 43, 128, 24, xi=0.5, positional=False, gain=3.0, seed=8),   # K1 44: last stc size
    _case("cvrp-k44-n128", "cvrp", 44, 128, 24, xi=-3.0, gain=4.0, seed=9),      # K1 45: fp32-pipe streaming kernel
    _case("cvrp-k47-n60", "cvrp", 47, 60, 30, clip=200.0, gain=2.0, seed=10),    # KT 48: last tensor-core size
    _case("cvrp-k48-n103", "cvrp", 48, 103, 24, clip=10.0, gain=3.0, seed=11),   # KT 49: MAXE 8, N1 104 largest resident
    _case("cvrp-k50-n104", "cvrp", 50, 104, 24, gain=4.0, seed=12),              # N1 105: streaming
    _case("cvrp-k63-n128", "cvrp", 63, 128, 24, xi=0.5, gain=2.0, seed=13),      # KT_MAX, N1 129
    _case("cvrp-k63-n40", "cvrp", 63, 40, 40, positional=False, gain=3.0, seed=14),   # fewer customers than k
    # BASELINE.json "CVRP1000 generalization inference (local kNN policy k=50 dominant)": KT 51
    _case("cvrp-k50-n1000", "cvrp", 50, 1000, 8, gain=3.0, seed=15, tf_steps=40),
    # tsp
    _case("tsp-k1-n20", "tsp", 1, 20, 20, n=2, gain=2.0, seed=21),
    _case("tsp-k32-n112", "tsp", 32, 112, 24, xi=0.5, gain=3.0, seed=22),        # KT 32: N1 112 largest resident
    _case("tsp-k32-n113", "tsp", 32, 113, 24, clip=10.0, gain=4.0, seed=23),
    _case("tsp-k32-n129", "tsp", 32, 129, 24, clip=200.0, gain=2.0, seed=24),
    _case("tsp-k33-n108", "tsp", 33, 108, 24, positional=False, gain=3.0, seed=25),   # MAXE 6, largest resident
    _case("tsp-k33-n109", "tsp", 33, 109, 24, gain=4.0, seed=26),
    _case("tsp-k44-n129", "tsp", 44, 129, 24, xi=-3.0, gain=2.0, seed=27),       # last stc size
    _case("tsp-k45-n129", "tsp", 45, 129, 24, xi=0.0, gain=3.0, seed=28),
    _case("tsp-k48-n64", "tsp", 48, 64, 32, xi=-3.0, gain=4.0, seed=29),         # KT 48: last tensor-core size
    _case("tsp-k49-n104", "tsp", 49, 104, 24, gain=2.0, seed=30),                # MAXE 8, largest resident
    _case("tsp-k49-n105", "tsp", 49, 105, 24, gain=3.0, seed=31),
    _case("tsp-k64-n129", "tsp", 64, 129, 24, positional=False, gain=4.0, seed=32),   # KT_MAX
    _case("tsp-k64-n64", "tsp", 64, 64, 40, clip=200.0, gain=2.0, seed=33),      # k = N: every node is a neighbour
]


def case_params(c):
    from elg_b200.synth import DEFAULT_MODEL_PARAMS
    return dict(DEFAULT_MODEL_PARAMS[c["kind"]], local_size=[c["k"]], xi=c["xi"], logit_clipping=c["clip"],
                positional=c["positional"])


def case_n1(c):
    return c["N"] + (1 if c["kind"] == "cvrp" else 0)


def decode_attentions(c):
    """Attention modes a single decode step is replayed with: fp32 always, the tensor-core kernel where it is eligible."""
    out = ["fp32"]
    if is_resident(c["kind"], c["k"], case_n1(c)) and tc_maxe(c["kind"], c["k"]):
        out.append("tensor")
    return out


def rollout_attentions(c):
    """fp32 and tensor forced, when they pick different kernels, plus auto."""
    kind, k, N1 = c["kind"], c["k"], case_n1(c)
    out = ["fp32"]
    if expected_kernel(kind, k, N1, "tensor", True) != expected_kernel(kind, k, N1, "fp32", True):
        out.append("tensor")
    return out + ["auto"]


def case_kernels(c, sms=148):
    kind, k, N1, B = c["kind"], c["k"], case_n1(c), c["n"] * c["aug"]
    s = {expected_kernel(kind, k, N1, a, False, B, c["M"], sms) for a in decode_attentions(c)}
    s |= {expected_kernel(kind, k, N1, a, True, B, c["M"], sms) for a in rollout_attentions(c)}
    return s


# ---------------------------------------------------------------------------------------- CPU tests
def _desc(kind, **over):
    from elg_b200 import engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS
    mp = dict(DEFAULT_MODEL_PARAMS[kind])
    mp.update(over)
    return engine.make_desc(kind, mp)


@pytest.mark.parametrize("kind,k_max", [("cvrp", 63), ("tsp", 64)])
def test_local_size_bounds(kind, k_max):
    """cvrp's local sequence holds the depot too, so it admits one neighbour fewer; the message names the problem's bound."""
    from elg_b200 import _lib
    L = _lib.WeightLayout()
    for k in (1, k_max):
        assert _lib.lib.elg_weight_layout(_desc(kind, local_size=[k]), L) == 0, _lib.lib.elg_last_error()
    for k in (0, k_max + 1):
        assert _lib.lib.elg_weight_layout(_desc(kind, local_size=[k]), L) != 0
        msg = _lib.lib.elg_last_error().decode()
        assert "outside [1,%d]" % k_max in msg and kind in msg, msg


@pytest.mark.parametrize("kind", ["cvrp", "tsp"])
def test_resident_boundary_per_local_sequence_length(kind):
    """elg_rollout_resident (the predicate elg_encode, elg_rollout and the training path share) against RESIDENT_MAX_N1."""
    from elg_b200 import _lib
    ks = (1, 8, 31, 32, 43, 44, 47, 48, 50, 63) if kind == "cvrp" else (1, 32, 33, 44, 45, 48, 49, 64)
    for k in ks:
        d = _desc(kind, local_size=[k])
        got = [n1 for n1 in range(2, 140) if _lib.lib.elg_rollout_resident(d, n1) == 1]
        assert got == list(range(2, RESIDENT_MAX_N1[maxe(kind, k)] + 1)), (k, got[-1:])


def test_case_table_covers_every_decode_instantiation():
    """Between them the cases launch all 12 rollout_kernel, all 8 rollout_tc_kernel and both rollout_stc_kernel
    instantiations, at the local sizes, shapes and runtime constants the configuration space asks for."""
    seen = set()
    for c in CASES:
        seen |= case_kernels(c)
    assert seen == ALL_INSTANTIATIONS, sorted(ALL_INSTANTIATIONS ^ seen)
    ks = {kind: {c["k"] for c in CASES if c["kind"] == kind} for kind in ("cvrp", "tsp")}
    assert {1, 8, 31, 32, 43, 44, 47, 48, 50, 63} <= ks["cvrp"]
    assert {1, 32, 33, 44, 45, 48, 49, 64} <= ks["tsp"]
    for kind in ("cvrp", "tsp"):
        for me, top in RESIDENT_MAX_N1.items():
            n1s = {case_n1(c) for c in CASES if c["kind"] == kind and maxe(kind, c["k"]) == me}
            assert {top, top + 1, 129} <= n1s, (kind, me, n1s)
    assert any(c["kind"] == "cvrp" and c["k"] == 50 and c["N"] == 1000 for c in CASES)
    # every non-default runtime constant on each kernel family: the fp32-pipe kernel on a resident and a streaming shape,
    # the tensor-core kernel (resident only) and the streamed tensor-core kernel (large instances only)
    knobs = [("xi", 0.0), ("xi", -3.0), ("xi", 0.5), ("clip", 10.0), ("clip", 200.0), ("positional", False)]
    for key, val in knobs:
        on = [c for c in CASES if c[key] == val]
        fams = set()
        for c in on:
            fams |= {re.sub(r"<.*", "", kn) + ("/resident" if "true" in kn else "/streaming" if "false" in kn else "")
                     for kn in case_kernels(c)}
        assert {"rollout_kernel/resident", "rollout_kernel/streaming", "rollout_tc_kernel", "rollout_stc_kernel"} <= fams, \
            (key, val, fams)
    assert len({c["id"] for c in CASES}) == len(CASES)
    assert all(2.0 <= c["gain"] <= 4.0 for c in CASES)


# ---------------------------------------------------------------------------------------- GPU: decode + rollout
def _problem(c, dtype):
    from elg_b200.synth import synthetic_cvrp_batch, synthetic_tsp_batch
    if c["kind"] == "cvrp":
        b = synthetic_cvrp_batch(c["n"], c["N"], seed=c["seed"])
        return O.load_cvrp(b["depot"], b["loc"], b["demand"], c["aug"], dtype)
    return O.load_tsp(synthetic_tsp_batch(c["n"], c["N"], seed=c["seed"]), c["aug"], dtype)


def _record_steps(c):
    """3-4 step counts spread over the first tf_steps decisions."""
    first = 2 if c["kind"] == "cvrp" else 1
    L = min(c["tf_steps"], c["N"] - 2)
    return sorted({first, first + L // 3, first + (2 * L) // 3, first + L - 1})


@pytest.fixture(scope="module", params=CASES, ids=lambda c: c["id"])
def oracle_case(request):
    """Oracle side of one case (CPU): fp64 states + logits at the recorded steps, the fp32 oracle's full greedy rollout."""
    from elg_b200.synth import synthetic_state_dict
    c = request.param
    mp = case_params(c)
    sd = synthetic_state_dict(c["kind"], seed=100 + c["seed"], gain=c["gain"], model_params=mp)
    prob32, prob64 = _problem(c, torch.float32), _problem(c, torch.float64)
    perm = O.start_permutation(c["kind"], c["N"], c["M"], seed=c["seed"])
    steps = _record_steps(c)
    rec = {}

    def hook(st, logits):
        if st.count in steps:
            rec[st.count] = dict(cur=st.cur.clone(), masked=st.masked.clone(), logits=logits.clone(),
                                 load=None if c["kind"] == "tsp" else st.load.clone())
    O.rollout(O.Weights(sd, c["kind"], mp, torch.float64), prob64, c["M"], perm, "greedy", hook=hook, max_steps=max(steps) + 1)
    assert sorted(rec) == steps
    ref_t, _, ref_r = O.rollout(O.Weights(sd, c["kind"], mp), prob32, c["M"], perm, "greedy")
    return dict(c=c, mp=mp, sd=sd, prob=prob32, perm=perm, rec=rec, ref_t=ref_t, ref_r=ref_r)


def _encoded(oc, attention):
    from elg_b200 import engine
    c, prob = oc["c"], oc["prob"]
    handle = engine.ModelHandle(c["kind"], oc["mp"], oc["sd"], DEV, attention=attention)
    return engine, engine.encode(handle, prob.xy.to(DEV), None if prob.demand is None else prob.demand.to(DEV))


@pytest.mark.gpu
def test_teacher_forced_logits_against_fp64(oracle_case):
    oc = oracle_case
    c, prob = oc["c"], oc["prob"]
    kind, N1, M = c["kind"], case_n1(c), c["M"]
    scale = c["clip"] / 50.0
    bar_max, bar_mean = LOGIT_MAX_ATOL * scale, LOGIT_MEAN_ATOL * scale
    first = oc["perm"][None, :].expand(prob.xy.shape[0], M).to(DEV) if kind == "tsp" else None
    for attention in decode_attentions(c):
        engine, batch = _encoded(oc, attention)
        want = expected_kernel(kind, c["k"], N1, attention, False)
        worst, total, count = 0.0, 0.0, 0
        for t, s in sorted(oc["rec"].items()):
            bits = engine.pack_mask_bits(s["masked"].to(DEV))
            load = None if kind == "tsp" else s["load"].float().to(DEV)
            (sel, _, logits), found = launched_kernels(
                lambda: engine.decode_step(batch, M, s["cur"].to(DEV), bits, load=load, first=first, want_logits=True))
            assert_kernel(found, want)
            logits, sel, ref = logits.cpu().double(), sel.cpu(), s["logits"]
            live = ~tie_rows(prob, kind, s["cur"], s["masked"], c["k"])
            assert live.float().mean() > 0.9
            assert torch.equal(torch.isinf(logits)[live], torch.isinf(ref)[live]), (attention, t)
            fin = ~torch.isinf(ref) & live[:, :, None]
            err = (logits[fin] - ref[fin]).abs()
            worst, total, count = max(worst, float(err.max())), total + float(err.sum()), count + err.numel()
            clear = (top2_margin(ref) > 2 * bar_max) & live
            assert torch.equal(sel[clear], ref.argmax(dim=2)[clear]), (attention, t)
        assert worst < bar_max, (attention, worst)
        assert total / count < bar_mean, (attention, total / count)


@pytest.mark.gpu
def test_fused_rollout_against_oracle(oracle_case):
    oc = oracle_case
    c, prob = oc["c"], oc["prob"]
    kind, N1, M = c["kind"], case_n1(c), c["M"]
    B = prob.xy.shape[0]
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    ref_t, ref_r = oc["ref_t"], oc["ref_r"]
    out = {}
    for attention in rollout_attentions(c):
        engine, batch = _encoded(oc, attention)
        (t16, reward, _, n_steps), found = launched_kernels(lambda: engine.rollout(batch, M, oc["perm"].tolist()))
        kn = expected_kernel(kind, c["k"], N1, attention, True, B, M, sms)
        assert_kernel(found, kn)
        tours, reward = t16[:, :, :int(n_steps.max())].long().cpu(), reward.cpu()
        out[attention] = (kn, tours, reward)
        frac, same = compare_tours(tours, ref_t)
        assert frac >= 0.95, (attention, frac)
        assert ((reward - ref_r).abs() / ref_r.abs())[same].max() < 1e-4, attention
        _, got = O.best_of(reward, c["aug"], c["n"])
        _, want = O.best_of(ref_r, c["aug"], c["n"])
        assert ((got - want).abs() / want).max() < 5e-3, attention
        if kind == "cvrp":
            O.check_feasible_cvrp(tours, prob.demand)
        else:
            assert torch.equal(tours.sort(dim=2)[0], torch.arange(N1).expand_as(tours))
        own = O.tour_length(prob.xy.double(), tours)          # every reward is its own tour's length
        assert ((own + reward.double()).abs() / own).max() < 5e-6, attention
    # one kernel, one answer; two kernels: the gate of the other two-kernel checks
    kernels = {}
    for attention, (kn, tours, reward) in out.items():
        if kn in kernels:
            assert torch.equal(tours, kernels[kn][0]) and torch.equal(reward, kernels[kn][1]), attention
        else:
            kernels[kn] = (tours, reward)
    runs = list(kernels.values())
    for (ta, ra), (tb, rb) in zip(runs, runs[1:]):
        frac, _ = compare_tours(ta, tb)
        assert frac >= 0.97, frac
        best_a, best_b = ra.max(1)[0], rb.max(1)[0]
        assert ((best_a - best_b).abs() / best_b.abs()).max() < 2e-3


# ---------------------------------------------------------------------------------------- GPU: encoder
ENC_CASES = [("cvrp", 128, 1, 60), ("tsp", 128, 16, 60), ("tsp", 256, 1, 60), ("cvrp", 256, 16, 60),
             ("cvrp", 384, 1, 120), ("tsp", 384, 16, 120), ("cvrp", 384, 6, 60), ("tsp", 1024, 1, 60), ("cvrp", 1024, 16, 120)]
UNFUSED_FF = (128, 384, 1024)       # not a multiple of 256 at most 512: the two-GEMM feed-forward (encoder.cu)
TS_XIN, TS_QKV, TS_ATT, TS_T1, TS_X1, TS_HID, TS_T2 = range(7)


def train_saved_off(l, rows, ff, which):
    """Float offset of one activation of layer l in the elg_encode_train buffer (common.cuh train_saved_off)."""
    part = (0, 128, 4 * 128, 5 * 128, 6 * 128, 7 * 128, 7 * 128 + ff)
    return (l * (8 * 128 + ff) + part[which]) * rows


def _enc_setup(kind, ff, layers, N):
    from elg_b200 import engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict, synthetic_tsp_batch
    mp = dict(DEFAULT_MODEL_PARAMS[kind], ff_hidden_dim=ff, encoder_layer_num=layers)
    sd = synthetic_state_dict(kind, seed=ff + layers, gain=2.0, model_params=mp)
    if kind == "cvrp":
        b = synthetic_cvrp_batch(3, N, seed=layers)
        p32, p64 = (O.load_cvrp(b["depot"], b["loc"], b["demand"], 1, dt) for dt in (torch.float32, torch.float64))
    else:
        x = synthetic_tsp_batch(3, N, seed=layers)
        p32, p64 = (O.load_tsp(x, 1, dt) for dt in (torch.float32, torch.float64))
    h = engine.ModelHandle(kind, mp, sd, DEV)
    return engine, mp, sd, h, p32, p64


@pytest.mark.gpu
@pytest.mark.parametrize("kind,ff,layers,N", ENC_CASES, ids=lambda v: str(v))
def test_encoder_against_fp64(kind, ff, layers, N):
    """batch.enc against the fp64 oracle; the bar is the larger of 5e-5 and 4x the fp32 oracle's own error, so that deep
    encoders (16 layers) are judged by what fp32 arithmetic can reach."""
    engine, mp, sd, h, p32, p64 = _enc_setup(kind, ff, layers, N)
    batch = engine.encode(h, p32.xy.to(DEV), None if p32.demand is None else p32.demand.to(DEV))
    torch.cuda.synchronize()
    truth = O.encode(O.Weights(sd, kind, mp, torch.float64), p64)
    own = float((O.encode(O.Weights(sd, kind, mp), p32).double() - truth).abs().max())
    err = float((batch.enc.cpu().double() - truth).abs().max())
    assert err < max(5e-5, 4 * own), (err, own)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,ff,layers,N", [c for c in ENC_CASES if c[1] in UNFUSED_FF], ids=lambda v: str(v))
def test_encode_train_equals_encode_on_unfused_feed_forward(kind, ff, layers, N):
    """elg_encode_train keeps every layer's activations at train_saved_off(l, ff) and computes the same tables as
    elg_encode bit for bit; the saved activations are consistent with the layer they belong to (any ff, any depth)."""
    engine, mp, sd, h, p32, _ = _enc_setup(kind, ff, layers, N)
    xy, dem = p32.xy.to(DEV), None if p32.demand is None else p32.demand.to(DEV)
    a = engine.encode(h, xy, dem)
    b, saved = engine.encode_train(h, xy, dem)
    torch.cuda.synchronize()
    for name in ("enc", "k", "v", "qtab", "eb", "e"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    B, N1 = xy.shape[0], xy.shape[1]
    rows = B * N1
    sv = saved.view(torch.float32).cpu().double()

    def act(l, which, width=128):
        o = train_saved_off(l, rows, ff, which)
        return sv[o:o + rows * width].reshape(B, N1, width)
    W = O.Weights(sd, kind, mp, torch.float64)
    for l in sorted({0, layers // 2, layers - 1}):
        p = "encoder.layers.%d." % l
        x1, hid, t2 = act(l, TS_X1), act(l, TS_HID, ff), act(l, TS_T2)
        want_hid = torch.relu(x1 @ W[p + W.ff + ".W1.weight"].T + W[p + W.ff + ".W1.bias"])
        assert float((hid - want_hid).abs().max()) < 1e-4 * max(1.0, float(want_hid.abs().max()))
        want_t2 = x1 + hid @ W[p + W.ff + ".W2.weight"].T + W[p + W.ff + ".W2.bias"]
        assert float((t2 - want_t2).abs().max()) < 1e-4 * max(1.0, float(want_t2.abs().max()))
        x_next = a.enc.cpu().double() if l == layers - 1 else act(l + 1, TS_XIN)
        want_x = O._instance_norm(t2, W[p + W.norm2 + ".norm.weight"], W[p + W.norm2 + ".norm.bias"])
        assert float((x_next - want_x).abs().max()) < 1e-4, l


# ---------------------------------------------------------------------------------------- GPU: training path
TRAIN_CASES = [
    # kind, overrides, N (N1 = the resident limit of the KT bucket), n, M
    ("cvrp", dict(local_size=[8], ff_hidden_dim=256, encoder_layer_num=1), 111, 2, 24),
    ("cvrp", dict(local_size=[50], ff_hidden_dim=384, encoder_layer_num=3, positional=False, xi=0.0, logit_clipping=10.0),
     103, 2, 24),
    ("tsp", dict(local_size=[33], ff_hidden_dim=384, encoder_layer_num=1, xi=0.0), 108, 2, 24),
    ("tsp", dict(local_size=[64], ff_hidden_dim=256, encoder_layer_num=3, positional=False, logit_clipping=10.0), 104, 2, 24),
]


def _trainer(kind, over):
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    from elg_b200.trainer import Trainer
    mp = dict(DEFAULT_MODEL_PARAMS[kind], **over)
    sd = synthetic_state_dict(kind, seed=11, gain=1.5, model_params=mp)
    return mp, sd, Trainer(kind, mp, sd, DEV)


def _train_id(v):
    return "%s-k%d-ff%d-l%d-n%d" % (v[0], v[1]["local_size"][0], v[1]["ff_hidden_dim"], v[1]["encoder_layer_num"], v[2])


@pytest.mark.gpu
@pytest.mark.parametrize("case", TRAIN_CASES, ids=_train_id)
def test_training_step_against_oracle_autograd(case):
    """A sampled rollout + elg_reinforce_backward at the resident limit of each local-sequence bucket: log-probs, loss and
    every parameter gradient against the oracle's autograd replaying the same tours (test_gpu_train's bars)."""
    import train_helpers as TH
    from elg_b200.synth import synthetic_cvrp_batch, synthetic_tsp_batch
    kind, over, N, n, M = case
    mp, sd, tr = _trainer(kind, over)
    assert is_resident(kind, mp["local_size"][0], N + (1 if kind == "cvrp" else 0))
    if kind == "cvrp":
        data = synthetic_cvrp_batch(n, N, seed=17)
        prob = O.load_cvrp(data["depot"], data["loc"], data["demand"], 1)
    else:
        data = synthetic_tsp_batch(n, N, seed=17)
        prob = O.load_tsp(data, 1)
    random.seed(6)
    out = tr.forward_backward(data, M, seed=77)
    torch.cuda.synchronize()
    tours = out["tours"][:, :, :out["T"]].long().cpu()
    if kind == "cvrp":
        O.check_feasible_cvrp(tours, prob.demand)
    J, logp, ref, _ = TH.oracle_grads(kind, mp, sd, prob, M, tours, out["reward"].cpu(), True)
    assert float((out["logp"].cpu() - logp).abs().max()) < 5e-3 * max(1.0, float(logp.abs().max()))
    assert abs(float(out["loss"]) - float(J)) < 5e-3 * max(1.0, abs(float(J)))
    eo = TH.grad_errors_l2(tr.unpack(out["grads"]), ref)
    assert max(eo.values()) < 2e-2, sorted(eo.items(), key=lambda kv: -kv[1])[:3]


@pytest.mark.gpu
@pytest.mark.parametrize("case", TRAIN_CASES, ids=_train_id)
def test_training_rejects_one_node_above_the_resident_limit(case):
    from elg_b200._lib import ElgError
    from elg_b200.synth import synthetic_cvrp_batch, synthetic_tsp_batch
    kind, over, N, n, M = case
    mp, sd, tr = _trainer(kind, over)
    assert not is_resident(kind, mp["local_size"][0], N + 1 + (1 if kind == "cvrp" else 0))
    data = synthetic_cvrp_batch(1, N + 1, seed=1) if kind == "cvrp" else synthetic_tsp_batch(1, N + 1, seed=1)
    with pytest.raises(ElgError):
        tr.forward_backward(data, 8, seed=5)


# ---------------------------------------------------------------------------------------- GPU: drop-in classes
@pytest.mark.gpu
def test_drop_in_model_passes_the_knobs_through():
    """CVRPModel / CVRPEnv / rollout with local_size [50], xi and logit_clipping changed give the tours and rewards of
    engine.rollout on a handle built from the same model_params."""
    from elg_b200 import engine
    from elg_b200.cvrp import CVRPEnv, CVRPModel, rollout
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict
    N, M = 100, 50
    mp = dict(DEFAULT_MODEL_PARAMS["cvrp"], local_size=[50], xi=0.5, logit_clipping=20)
    sd = synthetic_state_dict("cvrp", seed=41, gain=3.0, model_params=mp)
    data = synthetic_cvrp_batch(2, N, seed=42)
    model = CVRPModel(**mp)
    model.decoder.add_local_policy(DEV)
    model.load_state_dict(sd)
    model = model.to(DEV)
    env = CVRPEnv(M, DEV)
    env.load_random_problems(data, 8)
    reset_state, _, _ = env.reset()
    random.seed(3)
    model.pre_forward(reset_state)
    tours, _, reward = rollout(model, env, "greedy")
    d = model._handle.desc
    assert (d.local_k, d.xi, d.clip) == (50, 0.5, 20.0)
    handle = engine.ModelHandle("cvrp", mp, sd, DEV)
    xy, dem = engine.load_problems("cvrp", data["loc"].to(DEV), data["depot"].to(DEV), data["demand"].to(DEV), 8)
    batch = engine.encode(handle, xy, dem)
    t16, rew, _, n_steps = engine.rollout(batch, M, O.start_permutation("cvrp", N, M, seed=3).tolist())
    T = int(n_steps.max())
    assert tours.shape[2] == T
    assert torch.equal(tours.cpu(), t16[:, :, :T].long().cpu())
    assert torch.equal(reward.cpu(), rew.cpu())
