"""TSP local search with 2-opt and Or-opt moves on the GPU (elg_tsp_local_search, engine.tsp_local_search,
elg_b200.tsp.tsp_local_search, the drivers' opt-in stage) against the CPU oracle (tests/tsp_ls_oracle.py).

Under the rounded library metric every edge is an integer, so gains are exact in fp32 and fp64 alike and the kernel must
make the oracle's moves exactly.  Under the scaled metric fp32 gains can order near-ties differently from fp64 ones, so
there the invariants are checked instead.  max_segment = 0 must be elg_two_opt bit for bit in both metrics."""
import json
import os
import random

import numpy as np
import pytest
import torch

import tsp_ls_oracle as LS
from test_gpu_two_opt import _greedy_rows, _lib_rows

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "tests", "golden", "lib")


def _check_invariants(xy, rows, out, length, iters, max_iterations, optimum_rows=None):
    """Permutation with position 0 fixed, length as tour_length measures it, no longer than the input; tours that stopped
    before the cap have no variant with an fp64 gain below -1e-5 (checked on the rows listed in optimum_rows)."""
    from elg_b200 import engine
    rows, out = rows.cpu(), out.cpu()
    assert torch.equal(out.sort(1)[0], rows.sort(1)[0]) and torch.equal(out[:, 0], rows[:, 0])
    assert torch.equal(length.cpu(), engine.tour_length(xy, out.to(DEV)[:, None])[:, 0].cpu())       # bit for bit
    assert (length.cpu() <= engine.tour_length(xy, rows.to(DEV)[:, None])[:, 0].cpu()).all()
    xc = xy.cpu()
    for r in (range(len(out)) if optimum_rows is None else optimum_rows):
        if int(iters[r]) < max_iterations:
            assert LS.best_move(xc[r if xc.shape[0] > 1 else 0], out[r], 3, exact=True)[0] >= -1e-5


# ------------------------------------------------------------------------------------------------ 1. exact parity

@pytest.mark.parametrize("name,cap", [("eil51", 1000), ("kroA100", 1000), ("a280", 30), ("rat575", 20), ("pr1002", 4)])
def test_rounded_metric_identical_to_oracle(name, cap):
    from elg_b200 import engine
    xy, rows, _, _ = _lib_rows("tsplib", name)
    out, length, iters = engine.tsp_local_search(xy, rows, max_iterations=cap, rounding=True)
    ref_t, ref_len, ref_it = LS.tsp_local_search(xy.cpu(), rows.cpu(), cap, rounding=True)
    assert torch.equal(iters.cpu().long(), ref_it)
    assert torch.equal(out.cpu(), ref_t)
    assert torch.equal(length.cpu(), ref_len)
    if cap == 1000:
        assert int(iters.max()) < cap                                       # every tour ran to convergence
    else:
        assert int(iters.min()) == cap


def test_max_segment_zero_is_two_opt():
    from elg_b200 import engine
    xy, _, rows = _greedy_rows("tsp", 100, 64, seed=3)                     # scaled metric
    a = engine.tsp_local_search(xy, rows, max_segment=0)
    b = engine.two_opt("tsp", xy, rows)
    assert all(torch.equal(x, y) for x, y in zip(a, b)) and int(a[2].sum()) > 0
    for name in ("eil51", "a280"):                                         # rounded metric
        xy, rows, _, _ = _lib_rows("tsplib", name)
        a = engine.tsp_local_search(xy, rows, max_segment=0, rounding=True)
        b = engine.two_opt("tsp", xy, rows, rounding=True)
        assert all(torch.equal(x, y) for x, y in zip(a, b)) and int(a[2].sum()) > 0


def test_shorter_segments_match_the_oracle():
    from elg_b200 import engine
    xy, rows, _, _ = _lib_rows("tsplib", "kroA100")
    for ms in (1, 2):
        out, length, iters = engine.tsp_local_search(xy, rows, max_segment=ms, rounding=True)
        ref = LS.tsp_local_search(xy.cpu(), rows.cpu(), 1000, max_segment=ms, rounding=True)
        assert torch.equal(out.cpu(), ref[0]) and torch.equal(length.cpu(), ref[1]) and torch.equal(iters.cpu().long(), ref[2])


# ------------------------------------------------------------------------------------------------ 2. random instances

def test_tsp100_x8000_invariants():
    from elg_b200 import engine
    xy, _, rows = _greedy_rows("tsp", 100, 1000, seed=100)
    out, length, iters = engine.tsp_local_search(xy, rows)
    _check_invariants(xy, rows, out, length, iters, 1000, optimum_rows=range(0, 8000, 40))
    two = engine.two_opt("tsp", xy, rows)[1]
    assert float(length.mean()) < float(two.mean())


def test_tsp1000_x8_invariants():
    from elg_b200 import engine
    xy, _, rows = _greedy_rows("tsp", 1000, 1, seed=1000)
    out, length, iters = engine.tsp_local_search(xy, rows, max_iterations=3000)
    _check_invariants(xy, rows, out, length, iters, 3000)
    assert int(iters.min()) > 0


# ------------------------------------------------------------------------------------------------ 3. edges

@pytest.mark.parametrize("N1", [3, 4, 5, 6])
def test_tiny_tours(N1):
    from elg_b200 import engine
    g = torch.Generator().manual_seed(N1)
    xy = torch.floor(torch.rand(64, N1, 2, generator=g) * 100)
    rows = torch.stack([torch.randperm(N1, generator=g) for _ in range(64)])
    out, length, iters = engine.tsp_local_search(xy.to(DEV), rows.to(DEV), rounding=True)
    ref_t, ref_len, ref_it = LS.tsp_local_search(xy, rows, 1000, rounding=True)
    assert torch.equal(out.cpu(), ref_t) and torch.equal(iters.cpu().long(), ref_it) and torch.equal(length.cpu(), ref_len)
    if N1 >= 5:
        assert int(iters.sum()) > 0
    scaled = engine.tsp_local_search((xy / 100).to(DEV), rows.to(DEV))
    _check_invariants((xy / 100).to(DEV), rows, *scaled, 1000)


def test_padding_shared_coordinates_and_inst():
    from elg_b200 import engine
    g = torch.Generator().manual_seed(9)
    N1, R = 40, 24
    xy = torch.floor(torch.rand(1, N1, 2, generator=g) * 1000)
    rows = torch.stack([torch.randperm(N1, generator=g) for _ in range(R)])
    out, length, iters = engine.tsp_local_search(xy.to(DEV), rows.to(DEV), rounding=True)         # Bxy = 1
    ref = LS.tsp_local_search(xy, rows, 1000, rounding=True)
    assert torch.equal(out.cpu(), ref[0]) and torch.equal(length.cpu(), ref[1]) and torch.equal(iters.cpu().long(), ref[2])
    same = engine.tsp_local_search(xy.expand(R, -1, -1).to(DEV), rows.to(DEV), rounding=True)       # Bxy = R
    assert all(torch.equal(a, b) for a, b in zip(same, (out, length, iters)))
    other = torch.floor(torch.rand(2, N1, 2, generator=g) * 1000)
    inst = torch.ones(R, dtype=torch.int32)
    by_inst = engine.tsp_local_search(torch.cat((other[:1], xy, other[1:])).to(DEV), rows.to(DEV), inst=inst.to(DEV),
                                      rounding=True)
    assert all(torch.equal(a, b) for a, b in zip(by_inst, (out, length, iters)))
    pad = torch.randint(0, N1, (R, 9), generator=g)                         # L > N1: positions N1.. are left as they are
    p_out, p_len, p_it = engine.tsp_local_search(xy.to(DEV), torch.cat((rows, pad), 1).to(DEV), rounding=True)
    assert torch.equal(p_out[:, :N1], out) and torch.equal(p_out[:, N1:].cpu(), pad)
    assert torch.equal(p_len, length) and torch.equal(p_it, iters)


def test_largest_instance_against_oracle():
    """N1 = 8192: 112 KB of shared memory, one CTA per tour."""
    from elg_b200 import engine
    g = torch.Generator().manual_seed(11)
    N1 = 8192
    xy = torch.floor(torch.rand(1, N1, 2, generator=g) * 10000)
    rows = torch.randperm(N1, generator=g)[None]
    out, length, iters = engine.tsp_local_search(xy.to(DEV), rows.to(DEV), max_iterations=2, rounding=True)
    ref_t, ref_len, ref_it = LS.tsp_local_search(xy, rows, 2, rounding=True)
    assert int(iters[0]) == 2
    assert torch.equal(out.cpu(), ref_t) and torch.equal(length.cpu(), ref_len)


def test_too_many_nodes_fails_loudly():
    from elg_b200 import _lib, engine
    xy = torch.rand(1, 8193, 2, device=DEV)
    with pytest.raises(_lib.ElgError, match="8192"):
        engine.tsp_local_search(xy, torch.arange(8193, device=DEV)[None])


# ------------------------------------------------------------------------------------------------ 4. determinism

def test_deterministic_and_idempotent():
    from elg_b200 import engine
    xy, _, rows = _greedy_rows("tsp", 200, 16, seed=5)
    a = engine.tsp_local_search(xy, rows)
    b = engine.tsp_local_search(xy, rows.to(torch.int16))
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert int(a[2].max()) < 1000
    again = engine.tsp_local_search(xy, a[0])
    assert int(again[2].sum()) == 0 and torch.equal(again[0], a[0]) and torch.equal(again[1], a[1])


# ------------------------------------------------------------------------------------------------ 5. drop-in function

def test_dropin_numpy_and_torch():
    from elg_b200 import engine
    from elg_b200.tsp import tsp_local_search
    xy, _, rows = _greedy_rows("tsp", 50, 1, seed=9)
    pts = xy[0]                                                            # augmentation 0 = the instance itself
    want, _, it = engine.tsp_local_search(pts[None], rows, max_iterations=500)
    closed = torch.cat((rows, rows[:, :1]), 1)
    want = torch.cat((want, want[:, :1]), 1)
    t_np, n_np = tsp_local_search(pts.cpu().numpy(), closed.cpu().numpy().astype(np.int32), max_iterations=500)
    assert isinstance(t_np, np.ndarray) and t_np.dtype == np.int32 and n_np == int(it.max()) > 0
    assert np.array_equal(t_np, want.cpu().numpy())
    t_pt, n_pt = tsp_local_search(pts, closed, max_iterations=500, device=DEV)
    assert torch.is_tensor(t_pt) and t_pt.device == closed.device and torch.equal(t_pt, want) and n_pt == n_np
    t_cpu, _ = tsp_local_search(pts.cpu(), closed.cpu(), max_iterations=500)
    assert t_cpu.device.type == "cpu" and torch.equal(t_cpu, want.cpu())
    from elg_b200.tsp import batched_two_opt_torch
    two, _ = batched_two_opt_torch(pts, closed, max_iterations=500)
    assert torch.equal(tsp_local_search(pts, closed, max_iterations=500, max_segment=0)[0], two)


# ------------------------------------------------------------------------------------------------ 6. drivers

def _tsplib_driver(name, params):
    """The TSPLIB driver on one instance with extra config params -> (record, unscaled xy, best rows)."""
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    from elg_b200.tsp import TSPModel
    from elg_b200.tsp.test_tsplib import TSPLib_Tester
    with open(os.path.join(LIB, "tsplib_ref.json")) as f:
        ref = json.load(f)
    z = np.load(os.path.join(LIB, "tsplib_inputs.npz"))
    cfg = {"name": "ELG", "use_cuda": True, "cuda_device_num": 0, "load_checkpoint": None,
           "params": dict(aug_factor=8, **params), "model_params": dict(DEFAULT_MODEL_PARAMS["tsp"])}
    m = TSPModel(**cfg["model_params"])
    m.decoder.add_local_policy(DEV)
    m.load_state_dict(synthetic_state_dict("tsp", seed=ref["wseed"], gain=ref["gain"]))
    random.seed(ref["seed"])
    res = {}
    sols, rewards = TSPLib_Tester(cfg, model=m).test_on_one_ins(name, res, [z[name + "/coord"], float(z[name + "/opt"])])
    return res, sols[torch.arange(rewards.shape[0], device=DEV), rewards.argmax(1)]


def test_library_driver_refines_with_or_opt():
    xy, rows, res_off, opt = _lib_rows("tsplib", "eil51")
    res, rows_on = _tsplib_driver("eil51", {"tsp_local_search_iterations": 200})
    assert torch.equal(rows_on, rows) and res["best_cost"] == res_off["best_cost"]
    assert not any("tsp_ls" in k for k in res_off)
    _, ref_len, ref_it = LS.tsp_local_search(xy.cpu(), rows.cpu(), 200, rounding=True)
    assert res["best_cost_tsp_ls"] == float(ref_len.min()) <= res["best_cost"]
    assert res["gap_tsp_ls"] == (res["best_cost_tsp_ls"] - opt) / opt
    assert res["tsp_ls_iterations"] == int(ref_it.sum()) > 0 and res["tsp_ls_seconds"] > 0
    both, _ = _tsplib_driver("eil51", {"two_opt_iterations": 200, "tsp_local_search_iterations": 200})
    assert both["best_cost_tsp_ls"] == res["best_cost_tsp_ls"] and "best_cost_2opt" in both


def test_tsplib_driver_prints_and_records(tmp_path, capsys):
    import pickle
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    from elg_b200.tsp import TSPModel
    from elg_b200.tsp.test_tsplib import TSPLib_Tester
    z = np.load(os.path.join(LIB, "tsplib_inputs.npz"))
    d = tmp_path / "TSPLib"
    d.mkdir()
    for name in ("eil51", "st70"):
        with open(d / (name + ".pkl"), "wb") as f:
            pickle.dump([z[name + "/coord"], float(z[name + "/opt"])], f)
    for iters in (0, 100):
        cfg = {"name": "ELG", "use_cuda": True, "cuda_device_num": 0, "tsplib_path": str(d), "load_checkpoint": None,
               "params": {"aug_factor": 8, "tsp_local_search_iterations": iters},
               "model_params": dict(DEFAULT_MODEL_PARAMS["tsp"])}
        m = TSPModel(**cfg["model_params"])
        m.decoder.add_local_policy(DEV)
        m.load_state_dict(synthetic_state_dict("tsp", seed=3, gain=3.0))
        random.seed(1)
        results = TSPLib_Tester(cfg, model=m).test_on_tsplib(out_dir=str(tmp_path / ("out%d" % iters)))
        out = capsys.readouterr().out
        recs = [r["record"][0] for r in results]
        if iters:
            assert out.count("gap after 2-opt + or-opt") == 2 + 1 + 1
            assert all(r["best_cost_tsp_ls"] <= r["best_cost"] and r["tsp_ls_iterations"] > 0 for r in recs)
        else:
            assert "or-opt" not in out and not any("tsp_ls" in k for r in recs for k in r)


def test_test_py_with_or_opt(capsys):
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict, synthetic_tsp_batch
    from elg_b200.tsp import TSPEnv, TSPModel
    from elg_b200.tsp.test import test
    batch = synthetic_tsp_batch(4, 20, seed=8).to(DEV)
    model = TSPModel(**DEFAULT_MODEL_PARAMS["tsp"])
    model.decoder.add_local_policy(DEV)
    model.load_state_dict(synthetic_state_dict("tsp", seed=21, gain=3.0))
    model = model.to(DEV)
    env = TSPEnv(20, DEV)
    random.seed(5)
    avg = test([batch], model, env, 8)
    plain = capsys.readouterr().out
    assert "or-opt" not in plain
    random.seed(5)
    avg2 = test([batch], model, env, 8, two_opt_iterations=100, tsp_local_search_iterations=100)
    out = capsys.readouterr().out
    assert out.startswith(plain.split("Wall-clock")[0]) and float(avg2) == float(avg)
    lines = out.splitlines()
    assert lines[-2].startswith("2-opt Aug cost: ") and lines[-1].startswith("2-opt + or-opt Aug cost: ")
    assert float(lines[-1].split()[5].rstrip(",")) <= float(avg) + 1e-6
