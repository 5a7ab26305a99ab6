#!/usr/bin/env python
"""Benchmark of the ELG rollout hot path: CVRP100 ELG-POMO greedy multi-start inference,
POMO = 100, x8 augmentation, synthetic uniform instances, seeded random-init weights
(BASELINE.json configs[1]; the released checkpoints are not available offline).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py ... --dump-outputs DIR                   # + the last timed step's costs, rewards and tours as .npy
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on host cores
                                                             # (CPU oracle port; the reference is Python
                                                             # and cannot travel to the GPU box)

A "step" is one evaluation batch through the reference's test() loop body: load + x8 augmentation,
encoder, the whole greedy rollout, best-of-POMO and best-of-augmentation.  `value` = instances/s
with the instances already resident in HBM; `e2e` = the same call fed from pinned HOST buffers
with the H2D copy of the instances and the D2H copy of rewards/costs inside the timed region.
Every step uses fresh instances; one batch's decoder tables are ~2 GB, far larger than L2.
Rank layout (N > 1): one process per GPU, instances sharded across ranks, no data-path collective;
time = max over ranks of the CUDA-event time, bracketed by barrier + synchronize.
"""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_NODES, POMO, AUG = 100, 100, 8
WEIGHT_SEED, INSTANCE_SEED = 1234, 1234
ALG_BYTES_PER_AUG_STEP = 161548        # SURVEY.md 8(d): K+V+enc re-read + node statics + row state, CVRP100
ALG_FLOP_PER_ROW_STEP = 329088         # SURVEY.md 8(d): reference arithmetic per decode row-step, CVRP100
SMS, LANES = 148, 128
FP32_PEAK_TFLOPS = SMS * LANES * 2 * 1.965e9 / 1e12
# Per-pipe work of ONE decode row-step in the folded formulation the kernel computes (DESIGN.md 5.1 "Roofline", CVRP100:
# N+1 = 101 nodes, local sequence 41).  Tensor pipe: Q K^T, P V, O E'^T (3 x 12,928 MAC), the local policy's W (Wv PE)
# (1,312) and ol [PW | ZW] (1,440) = 41,536 MAC, each issued three times (split precision: lo*hi, hi*lo, hi*hi).
# FMA/ALU pipe (thread operations): query row, the two softmaxes around their exponentials, local scores / sums, final
# logits, fp32 -> fp16 hi/lo conversions, environment step and list walk on bit masks.  XU pipe: one exp2 per (head, key).
PIPE_TENSOR_FLOP = 41536 * 2 * 3
PIPE_FMA_OPS = 2 * (128 + 492 + 492 + 96 + 164) + 3232 + 656 + 303 + 3780 + 1200
PIPE_XU_OPS = 8 * 101 + 4 * 41
DUMP_BYTES = 64 << 20                  # --dump-outputs: all arrays together


def ncu_traffic():
    """dram__bytes of the rollout kernel per aug-instance from the committed ncu --set full capture of THIS kernel
    (profiles/ncu_traffic.json: {sha, kernel, dram_bytes_per_aug_instance, source}); None if there is no capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


def make_instances(n, seed):
    from elg_b200.synth import synthetic_cvrp_batch
    return synthetic_cvrp_batch(n, N_NODES, seed=seed)


# ------------------------------------------------------------------------------------------- CPU arms
def cpu_rollout_rate(n_inst, seed, threads=None, device=None, keep=None):
    """Reference algorithm (oracle port, torch eager): instances/s for one batch of n_inst on the host cores, or, with
    device='cuda:0', the same torch code on the GPU (SURVEY 8d "reference torch-CUDA eager", informative).  `keep` (dict)
    receives the tours / rewards / per-instance costs for the in-bench parity check."""
    import torch
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    from oracle import elg_oracle as O
    if threads:
        torch.set_num_threads(threads)
    W = O.Weights(synthetic_state_dict("cvrp", seed=WEIGHT_SEED), "cvrp", dict(DEFAULT_MODEL_PARAMS["cvrp"]))
    data = make_instances(n_inst, seed)
    ctx = torch.device(device) if device else torch.device("cpu")
    if device:
        W.sd = {k: v.to(device) for k, v in W.sd.items()}
        data = {k: v.to(device) for k, v in data.items()}
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    with torch.no_grad(), ctx:
        prob = O.load_cvrp(data["depot"], data["loc"], data["demand"], AUG)
        perm = O.start_permutation("cvrp", N_NODES, POMO, seed=seed)
        if device:
            perm = perm.to(device)
        tours, _, reward = O.rollout(W, prob, POMO, perm, "greedy")
        _, aug_cost = O.best_of(reward, AUG, n_inst)
        if device:
            torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if keep is not None:
        keep.update(tours=tours.cpu(), reward=reward.cpu(), aug_cost=aug_cost.cpu(), perm=perm.cpu())
    return n_inst / dt, dt, int(tours.shape[2])


def gpu_vs_oracle(model, env, dev, n_inst, seed, ref):
    """In-bench parity: the instances the CPU baseline just solved, through our CUDA path with the same start permutation."""
    import torch
    from elg_b200.cvrp.test import solve_batch
    data = {k: v.to(dev) for k, v in make_instances(n_inst, seed).items()}
    random.seed(seed)
    _, aug, sol, rew = solve_batch(model, env, data, AUG)
    sol, rew, aug = sol.cpu(), rew.cpu(), aug.cpu()
    rt = ref["tours"]
    T = max(sol.shape[2], rt.shape[2])
    a = torch.zeros(sol.shape[0], sol.shape[1], T, dtype=torch.long); a[:, :, :sol.shape[2]] = sol
    b = torch.zeros_like(a); b[:, :, :rt.shape[2]] = rt
    same = (a == b).all(dim=2)
    rel = ((rew - ref["reward"]).abs() / ref["reward"].abs())[same]
    return {"instances": n_inst, "rows": int(same.numel()), "rows_identical_frac": float(same.float().mean()),
            "reward_max_rel_err_on_identical_rows": float(rel.max()) if rel.numel() else None,
            "best_cost_max_rel_err": float(((aug - ref["aug_cost"]).abs() / ref["aug_cost"]).max()),
            "best_cost_identical": int(((aug - ref["aug_cost"]).abs() / ref["aug_cost"] < 1e-6).sum()),
            "checker": "oracle port (torch CPU) on the cpu_baseline sample, same weights / instances / start permutation"}


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path, timed on host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    torch.set_num_threads(os.cpu_count() or 1)      # torchrun exports OMP_NUM_THREADS=1: use every host core anyway
    cores = torch.get_num_threads()
    n = args.ref_batch
    times, T = [], 0
    for s in range(args.warmup + args.steps):
        rate, dt, T = cpu_rollout_rate(n, INSTANCE_SEED + s)
        if s >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = n * len(times) / total
    line = {"impl": "reference", "metric": "CVRP100 instances/s (POMO x8 aug, greedy)", "value": value, "unit": "instances/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
            "ms_per_decode_step": 1e3 * total / len(times) / max(T, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(n, 1),
            "cpu_baseline": {"value": value, "unit": "instances/s", "cores": cores, "kind": "port",
                             "sample": "%d CVRP100 instances per step (x8 aug x 100 POMO rows), %d steps" % (n, args.steps)},
            "e2e": {"value": value, "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "host_cpu_count": os.cpu_count()}
    print(json.dumps(line), flush=True)


def workload_config(batch_per_gpu, n_gpus):
    return {"workload": "CVRP100 ELG-POMO greedy multi-start inference, POMO=100, x8 augmentation, synthetic uniform instances",
            "problem_size": N_NODES, "pomo": POMO, "aug": AUG, "instances_per_step_per_gpu": batch_per_gpu,
            "weights": "seeded random init (released checkpoint not available offline)",
            "l2_policy": "fresh instances every step; per-step decoder tables (~2 GB) exceed L2",
            "parallelism": "instances sharded across %d GPU(s), no data-path collective" % n_gpus}


# ------------------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from elg_b200 import _lib, engine
    from elg_b200.cvrp import CVRPEnv, CVRPModel
    from elg_b200.cvrp.test import solve_batch
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = "cuda:%d" % local
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))

    mp = dict(DEFAULT_MODEL_PARAMS["cvrp"])
    model = CVRPModel(**mp)
    model.decoder.add_local_policy(dev)
    model.load_state_dict(synthetic_state_dict("cvrp", seed=WEIGHT_SEED))
    model = model.to(dev).eval().requires_grad_(False)
    env = CVRPEnv(POMO, dev)
    nb = args.batch
    total_steps = args.warmup + args.steps

    # synthetic instances: every (step, rank) gets its own seeded batch; host copies are pinned
    host = []
    for s in range(total_steps):
        d = make_instances(nb, INSTANCE_SEED + 7919 * s + rank)
        host.append({k: v.pin_memory() for k, v in d.items()})
    dev_batches = [{k: v.to(dev) for k, v in h.items()} for h in host]
    out_host = {"costs": torch.empty((2, nb), dtype=torch.float32).pin_memory(),
                "rewards": torch.empty((AUG * nb, POMO), dtype=torch.float32).pin_memory()}

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step_device(s):
        random.seed(INSTANCE_SEED + s)
        return solve_batch(model, env, dev_batches[s], AUG)

    def step_e2e(s):
        random.seed(INSTANCE_SEED + s)
        batch = {k: v.to(dev, non_blocking=True) for k, v in host[s].items()}
        no_aug, aug, _, rewards = solve_batch(model, env, batch, AUG)
        out_host["costs"][0].copy_(no_aug, non_blocking=True)
        out_host["costs"][1].copy_(aug, non_blocking=True)
        out_host["rewards"].copy_(rewards, non_blocking=True)
        return no_aug, aug

    def timed(fn):
        for s in range(args.warmup):
            fn(s)
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        engine.profile_events = []
        launches0 = _lib.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        costs = []
        for s in range(args.warmup, total_steps):
            out = fn(s)
            costs.append(out[1].mean())
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        launches = _lib.launch_count() - launches0
        events, engine.profile_events = engine.profile_events, None
        clocks = sampler.stop() if rank == 0 else None
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches, events, clocks, float(torch.stack(costs).mean()), out

    ms_dev, launches, events, clocks, mean_cost, last = timed(step_device)
    dump = sample_outputs(*last) if args.dump_outputs and rank == 0 else None
    del last
    ms_e2e, _, _, clocks_e2e, _, _ = timed(step_e2e)

    # rollout-kernel roofline numbers from the CUDA events recorded around each elg_rollout launch
    k_ms, aug_steps, row_steps, T_list = 0.0, 0, 0, []
    for e0, e1, n_steps, tiles in events:
        k_ms += e0.elapsed_time(e1)
        per_inst = n_steps.view(-1, tiles).max(dim=1)[0]
        aug_steps += int(per_inst.sum())
        row_steps += int(per_inst.sum()) * POMO
        T_list.append(int(n_steps.max()))
    peaks, peak_src = measured_peaks()
    ach_gbs = ALG_BYTES_PER_AUG_STEP * aug_steps / (k_ms * 1e-3) / 1e9
    ach_tf = ALG_FLOP_PER_ROW_STEP * row_steps / (k_ms * 1e-3) / 1e12

    # config 3 (REINFORCE training step, NCCL all-reduce of the gradient for N > 1) rides along so that every driver run
    # puts it on record; `--workload train` prints the same measurement as its own line
    train = None
    if not args.no_train:
        train = measure_train(args, world, rank, local, dev, short=True)

    if rank == 0:
        n_total = nb * world * args.steps
        value = n_total / (ms_dev * 1e-3)
        e2e = n_total / (ms_e2e * 1e-3)
        n_launch = max(len(events), 1)
        # per-pipe lower bounds of the rollout kernel for the row-steps it actually processed (all N GPUs of this rank's view
        # are identical, so rank 0's kernel stands for the job)
        sm_clock = (clocks or {}).get("sm_mhz") or 1965.0
        tc_peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
        t_tensor = PIPE_TENSOR_FLOP * row_steps / (tc_peak * 1e12) * 1e3                                  # ms
        t_fma = PIPE_FMA_OPS * row_steps / (SMS * LANES * sm_clock * 1e6) * 1e3
        t_xu = PIPE_XU_OPS * row_steps / (SMS * 16 * sm_clock * 1e6) * 1e3
        t_bound = max(t_tensor, t_fma, t_xu)
        bound_pipe = "fma" if t_bound == t_fma else ("tensor" if t_bound == t_tensor else "xu")
        traffic = ncu_traffic()
        line = {
            "metric": "CVRP100 instances/s (POMO x8 aug, greedy)", "value": value, "unit": "instances/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps,
            "ms_per_decode_step": k_ms / max(sum(T_list), 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(nb, world),
            "e2e": {"value": e2e, "unit": "instances/s", "h2d_bytes_per_step": nb * (2 + 2 * N_NODES + N_NODES) * 4,
                    "d2h_bytes_per_step": 2 * nb * 4 + AUG * nb * POMO * 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches,
            "clocks": clocks, "clocks_e2e": clocks_e2e,
            # The rollout kernel keeps K'/V/E' resident in shared memory, so it is compute-side bound; `frac` is the
            # per-pipe lower bound of its folded arithmetic over the measured time (DESIGN.md 5.1).  The tensor-pipe view
            # (achieved / peak in TFLOP/s) and the SURVEY 8(d) contract figures are kept beside it.
            "roofline": {"kernel": "rollout_tc_kernel<CVRP> (decode step + env step, whole rollout in one launch)",
                         "bound": "tensor", "achieved": PIPE_TENSOR_FLOP * row_steps / (k_ms * 1e-3) / 1e12,
                         "peak": tc_peak, "unit": "TFLOP/s",
                         "frac": t_tensor / k_ms, "peak_source": peak_src + (", sustained (kernel of a long step)" if "bf16_tflops_sustained" in peaks else ", burst"),
                         "traffic": (traffic["dram_bytes_per_aug_instance"] * nb * AUG) if traffic else None,
                         "traffic_source": ({k: traffic[k] for k in ("sha", "source") if k in traffic} if traffic else None),
                         "pipe_model": {"tensor_ms": t_tensor / n_launch, "fma_ms": t_fma / n_launch, "xu_ms": t_xu / n_launch,
                                        "bound_ms": t_bound / n_launch, "serial_ms": (t_tensor + t_fma + t_xu) / n_launch,
                                        "measured_ms": k_ms / n_launch, "binding_pipe": bound_pipe,
                                        "frac_of_bound": t_bound / k_ms, "frac_of_serial": (t_tensor + t_fma + t_xu) / k_ms,
                                        "per_row_step": {"tensor_flop_issued": PIPE_TENSOR_FLOP, "fma_alu_thread_ops": PIPE_FMA_OPS,
                                                         "xu_ops": PIPE_XU_OPS},
                                        "us_per_sm_step": k_ms * 1e3 * SMS / max(aug_steps, 1),
                                        "note": "lower bounds per pipe for the folded arithmetic (split-precision MMAs as issued, "
                                                "100 live rows); max() = perfect overlap of the pipes, serial = none"},
                         "row_steps_per_launch": row_steps / n_launch,
                         "aug_instance_steps_per_launch": aug_steps / n_launch,
                         "kernel_ms_per_launch": k_ms / n_launch,
                         "kernel_share_of_step": k_ms / ms_dev,
                         "contract_hbm": {"achieved": ach_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach_gbs / peaks["hbm_gbs"],
                                          "algorithmic_bytes_per_aug_instance_step": ALG_BYTES_PER_AUG_STEP,
                                          "note": "SURVEY 8(d) streaming model; the operands stay in shared memory, so these bytes "
                                                  "are by design not moved (see traffic)"},
                         "contract_fp32": {"achieved": ach_tf, "peak": FP32_PEAK_TFLOPS, "unit": "TFLOP/s",
                                           "frac": ach_tf / FP32_PEAK_TFLOPS, "flop_per_row_step": ALG_FLOP_PER_ROW_STEP,
                                           "note": "reference-arithmetic FLOPs (SURVEY 8d) / kernel time: a throughput-equivalent, "
                                                   "not a utilisation (the folds remove 2.4x of them, the contractions run on tcgen05)"}},
            "mean_aug_cost": mean_cost, "rollout_steps_T": T_list,
        }
        if train is not None:
            line["train"] = train
        if world == 1 and not args.no_cpu_baseline:
            torch.set_num_threads(os.cpu_count() or 1)
            ref = {}
            rate, dt, T = cpu_rollout_rate(args.cpu_sample, INSTANCE_SEED, keep=ref)
            line["cpu_baseline"] = {"value": rate, "unit": "instances/s", "cores": torch.get_num_threads(), "kind": "port",
                                    "sample": "%d CVRP100 instances (x8 aug x 100 POMO rows), one batch, %.1f s, T=%d; "
                                              "oracle port of the reference's torch-CPU path" % (args.cpu_sample, dt, T),
                                    "host_cpu_count": os.cpu_count()}
            try:
                line["parity"] = gpu_vs_oracle(model, env, dev, args.cpu_sample, INSTANCE_SEED, ref)
            except Exception as e:      # the bench line must survive a checker problem
                line["parity"] = {"error": repr(e)[:200]}
            try:
                cpu_rollout_rate(2, INSTANCE_SEED, device=dev)                      # warm-up (cuBLAS handles, allocator)
                n_eager = 8 * args.cpu_sample                                       # a batch large enough to amortise the launches
                rate_g, dt_g, T_g = cpu_rollout_rate(n_eager, INSTANCE_SEED, device=dev)
                line["ref_cuda_eager"] = {"value": rate_g, "unit": "instances/s", "kind": "port",
                                          "sample": "%d instances in one batch, the oracle port's torch code on %s (eager, fp32, no "
                                                    "TF32), %.1f s, T=%d; informative (SURVEY 8d), not the baseline" % (n_eager, dev, dt_g, T_g)}
            except Exception as e:
                line["ref_cuda_eager"] = {"error": repr(e)[:200]}
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def sample_outputs(no_aug_cost, aug_cost, tours, rewards):
    """What solve_batch() returned in the last timed step, as host arrays for --dump-outputs.  The costs are kept whole.
    Tours and rewards of more aug-instances than fit in DUMP_BYTES are cut to a fixed seeded sample of aug-instances: a
    prefix of one seeded permutation, so the sample of a longer rollout is a subset of that of a shorter one.  `rows`
    lists the sampled aug-instances (row a * batch + i = augmentation a of instance i)."""
    import torch
    A, M, T = tours.shape
    room = DUMP_BYTES - 2 * 4 * no_aug_cost.numel()
    k = min(A, room // (4 * M * (T + 1) + 8))
    rows = torch.randperm(A, generator=torch.Generator().manual_seed(0))[:k].sort()[0]
    idx = rows.to(tours.device)
    return {"no_aug_cost": no_aug_cost.float().cpu().numpy(), "aug_cost": aug_cost.float().cpu().numpy(),
            "rewards": rewards[idx].float().cpu().numpy(), "tours": tours[idx].float().cpu().numpy(),
            "rows": rows.double().numpy()}


def write_outputs(dirname, arrays):
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


# ------------------------------------------------------------------------------------------- training workload
TRAIN_METRIC = "CVRP100 REINFORCE training instances/s (POMO=100 shared baseline, sample rollout + backward + Adam)"


def train_config(batch_per_gpu, n_gpus):
    return {"workload": "CVRP100 REINFORCE training step with POMO shared baseline, batch %d x 100 rollouts per GPU, "
                        "data-parallel with one NCCL all-reduce of the packed gradient" % batch_per_gpu,
            "problem_size": N_NODES, "pomo": POMO, "aug": 1, "instances_per_step_per_gpu": batch_per_gpu,
            "weights": "seeded random init", "l2_policy": "fresh instances every step; per-step activations + row-step "
            "buffers (> 1 GB) exceed L2", "parallelism": "dp%d" % n_gpus}


def run_train(args):
    """`--workload train`: BASELINE.json configs[2] as its own bench line."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = "cuda:%d" % local
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    line = measure_train(args, world, rank, local, dev, short=False)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure_train(args, world, rank, local, dev, short):
    """BASELINE.json configs[2]: one step = generate/load a batch, encoder (activations kept), sample rollout, REINFORCE
    backward, all-reduce of the gradient (N > 1), Adam, re-fold of the decoder tables.  Returns the bench line (rank 0;
    None elsewhere); short = the condensed form embedded in the inference line."""
    import torch
    import torch.distributed as dist
    from elg_b200 import _lib, engine
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    from elg_b200.trainer import Trainer
    tr = Trainer("cvrp", dict(DEFAULT_MODEL_PARAMS["cvrp"]), synthetic_state_dict("cvrp", seed=WEIGHT_SEED), dev,
                 chunk_steps=args.chunk_steps)
    nb = args.train_batch
    steps = min(args.steps, 10) if short else args.steps
    total_steps = args.warmup + steps
    host = [{k: v.pin_memory() for k, v in make_instances(nb, INSTANCE_SEED + 7919 * s + rank).items()} for s in range(total_steps)]
    dev_batches = [{k: v.to(dev) for k, v in h.items()} for h in host]
    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step_device(s):
        random.seed(INSTANCE_SEED + s)
        return tr.step(dev_batches[s], POMO, seed=INSTANCE_SEED + s)

    def step_e2e(s):
        random.seed(INSTANCE_SEED + s)
        out = tr.step({k: v.to(dev, non_blocking=True) for k, v in host[s].items()}, POMO, seed=INSTANCE_SEED + s)
        loss_host.copy_(out["loss"], non_blocking=True)
        return out

    def timed(fn):
        for s in range(args.warmup):
            fn(s)
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        launches0 = _lib.launch_count()
        engine.train_profile_events = []
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        costs, Ts = [], []
        for s in range(args.warmup, total_steps):
            out = fn(s)
            costs.append(-out["reward"].mean())
            Ts.append(out["T"])
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        launches = _lib.launch_count() - launches0
        events, engine.train_profile_events = engine.train_profile_events, None
        clocks = sampler.stop() if rank == 0 else None
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches, clocks, [float(c) for c in costs], Ts, events

    # The first pass through the timed loop runs its first two steps 30 and 5 ms long whatever the warm-up count, input
    # residency or clock sampler (per-step CUDA events: 56.5 29.1 24.4 24.3 ... against 24.0 24.2 23.9 ... for any later
    # pass over identical work), i.e. +7 % on a 10-step region.  So one full pass is discarded, and every kept pass starts
    # from the same weights and optimizer state.
    ck0 = tr.checkpoint()
    timed(step_device)
    tr.load_checkpoint(ck0)
    ms_dev, launches, clocks, costs, Ts, events = timed(step_device)
    tr.load_checkpoint(ck0)
    ms_e2e, _, clocks_e2e, _, _, _ = timed(step_e2e)
    bwd_ms = sum(e0.elapsed_time(e1) for e0, e1, _ in events)
    row_steps = sum(n for _, _, n in events)
    # the gradient all-reduce on its own (N > 1): one NCCL sum of the packed parameter vector, timed with CUDA events
    ar_ms = 0.0
    if world > 1:
        from elg_b200.dist import allreduce_mean_gradient
        g = torch.zeros_like(tr.grads)
        for _ in range(3):
            allreduce_mean_gradient(g)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            allreduce_mean_gradient(g)
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) / 20], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ar_ms = float(t.item())
    if rank != 0:
        return None
    n_total = nb * world * steps
    grad_bytes = int(tr.grads.numel()) * 4
    if short:
        return {"metric": TRAIN_METRIC, "value": n_total / (ms_dev * 1e-3), "unit": "instances/s", "n_gpus": world, "steps": steps,
                "warmup": args.warmup, "ms_per_step": ms_dev / steps, "scaling": "weak",
                "e2e": {"value": n_total / (ms_e2e * 1e-3), "unit": "instances/s", "ms_per_step": ms_e2e / steps,
                        "h2d_bytes_per_step": nb * (2 + 2 * N_NODES + N_NODES) * 4, "d2h_bytes_per_step": 8},
                "instances_per_step_per_gpu": nb, "backward_ms_per_step": bwd_ms / max(len(events), 1),
                "allreduce_ms": ar_ms, "grad_allreduce_bytes": grad_bytes if world > 1 else 0, "collective": "NCCL all-reduce (sum) of the "
                "packed gradient, 1/world folded into the Adam kernel" if world > 1 else "none (1 GPU)",
                "gpu_launches": launches, "mean_sampled_cost_first_last": [costs[0], costs[-1]], "rollout_steps_T": Ts,
                "config": train_config(nb, world)["workload"]}
    line = {"metric": TRAIN_METRIC, "value": n_total / (ms_dev * 1e-3), "unit": "instances/s", "n_gpus": world,
            "steps": steps, "warmup": args.warmup, "ms_per_step": ms_dev / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": train_config(nb, world),
            "e2e": {"value": n_total / (ms_e2e * 1e-3), "unit": "instances/s",
                    "h2d_bytes_per_step": nb * (2 + 2 * N_NODES + N_NODES) * 4, "d2h_bytes_per_step": 4 + 4,
                    "ms_per_step": ms_e2e / steps},
            "gpu_launches": launches, "clocks": clocks, "clocks_e2e": clocks_e2e,
            "mean_sampled_cost_per_step": costs, "rollout_steps_T": Ts,
            "allreduce_ms": ar_ms, "grad_allreduce_bytes": grad_bytes if world > 1 else 0}
    peaks, peak_src = measured_peaks()
    # streaming model of the backward: per aug-instance-step the tables K', V, E' are read for the forward recompute
    # and again for the gradients (2 x SURVEY 8d's 161,548 B), and the per-row-step vectors are written and re-read
    alg = 2 * ALG_BYTES_PER_AUG_STEP * (row_steps / POMO) + row_steps * 2 * (104 + 104 + 128) * 4
    ach = alg / (bwd_ms * 1e-3) / 1e9
    line["roofline"] = {"kernel": "elg_reinforce_backward (replay, local/global decode backward, table + encoder backward)",
                        "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                        "peak_source": peak_src, "traffic": None, "algorithmic_bytes_per_step": alg / max(len(events), 1),
                        "ms_per_step": bwd_ms / max(len(events), 1), "share_of_step": bwd_ms / ms_dev,
                        "row_steps_per_step": row_steps / max(len(events), 1),
                        "note": "the instance tables are staged in shared memory once per 4 steps, so HBM is not what binds: "
                                "global_bwd_kernel runs at 60 % of the shared-memory wavefront peak (profiles/r01_train_ncu.md)"}
    if world == 1 and not args.no_cpu_baseline:
        rate, dt, T, cores = cpu_train_rate(args.cpu_train_sample, INSTANCE_SEED)
        line["cpu_baseline"] = {"value": rate, "unit": "instances/s", "cores": cores, "kind": "port",
                                "sample": "%d CVRP100 instances x 100 rollouts, one step, %.1f s, T=%d; oracle port: teacher-forced "
                                          "forward with autograd graph + backward + Adam on pre-sampled tours" % (args.cpu_train_sample, dt, T)}
    return line


def cpu_train_rate(n_inst, seed):
    """The reference's training step on host cores (oracle port): forward with autograd graph, J.backward(), Adam."""
    import torch
    from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_state_dict
    from oracle import elg_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    mp = dict(DEFAULT_MODEL_PARAMS["cvrp"])
    sd = synthetic_state_dict("cvrp", seed=WEIGHT_SEED)
    data = make_instances(n_inst, seed)
    prob = O.load_cvrp(data["depot"], data["loc"], data["demand"], 1)
    perm = O.start_permutation("cvrp", N_NODES, POMO, seed=seed)
    with torch.no_grad():          # sampling pre-pass (not timed): fixes the action sequence
        tours, _, reward = O.rollout(O.Weights(sd, "cvrp", mp), prob, POMO, perm, "sample", generator=torch.Generator().manual_seed(seed))
    W = O.Weights(sd, "cvrp", mp).requires_grad_()
    opt = torch.optim.Adam(list(W.sd.values()), lr=1e-4, weight_decay=1e-6)
    t0 = time.perf_counter()
    J, _ = O.reinforce_loss(W, prob, POMO, tours, reward, True)
    opt.zero_grad()
    J.backward()
    opt.step()
    dt = time.perf_counter() - t0
    return n_inst / dt, dt, int(tours.shape[2]), torch.get_num_threads()


def run_reference_train(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    times, T, cores = [], 0, 1
    for s in range(args.warmup + args.steps):
        rate, dt, T, cores = cpu_train_rate(args.cpu_train_sample, INSTANCE_SEED + s)
        if s >= args.warmup:
            times.append(dt)
    value = args.cpu_train_sample * len(times) / sum(times)
    print(json.dumps({"impl": "reference", "metric": TRAIN_METRIC, "value": value, "unit": "instances/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": train_config(args.cpu_train_sample, 1),
                      "cpu_baseline": {"value": value, "unit": "instances/s", "cores": cores, "kind": "port",
                                       "sample": "%d CVRP100 instances x 100 rollouts per step, T=%d" % (args.cpu_train_sample, T)},
                      "e2e": {"value": value, "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1000, help="instances per step per GPU (10 steps = the 10k-instance config)")
    ap.add_argument("--ref-batch", type=int, default=8, help="instances per step for --impl reference (bounded sample)")
    ap.add_argument("--cpu-sample", type=int, default=12, help="instances in the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the embedded training measurement (config 3) of the inference line")
    ap.add_argument("--workload", default="inference", choices=["inference", "train"],
                    help="inference = BASELINE.json configs[1] (the headline metric); train = configs[2]")
    ap.add_argument("--train-batch", type=int, default=64, help="training instances per step per GPU")
    ap.add_argument("--chunk-steps", type=int, default=128, help="rollout steps per decode-backward launch")
    ap.add_argument("--cpu-train-sample", type=int, default=2, help="instances in the CPU training-step sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's instances) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "inference"):
        ap.error("--dump-outputs applies to the CUDA inference path (--impl ours --workload inference)")
    if args.warmup < 3 and args.impl == "ours" and not os.environ.get("ELG_BENCH_ALLOW_SHORT"):
        args.warmup = 3
    if args.workload == "train":
        run_reference_train(args) if args.impl == "reference" else run_train(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
