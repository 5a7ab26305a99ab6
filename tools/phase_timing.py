#!/usr/bin/env python
"""Per-phase cycle breakdown of the rollout kernel (debug build only).

    python -m elg_b200.build --variant timing                                  # here (libelg_b200_timing.so)
    gpurun -- ELG_B200_LIB=elg_b200/csrc/libelg_b200_timing.so ELG_B200_ATTENTION=tensor python tools/phase_timing.py

Thread 0 of every CTA accumulates clock64() deltas at the phase boundaries; the sum over CTAs is printed as
a share of the total.  The tensor-core kernel also splits its softmax rounds per group: the leader of each group
accumulates five sub-phases, printed as cycles per round and as a share of the step."""
import ctypes as C
import os
import random
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from elg_b200 import _lib
from elg_b200.cvrp import CVRPEnv, CVRPModel
from elg_b200.cvrp.test import solve_batch
from elg_b200.synth import DEFAULT_MODEL_PARAMS, synthetic_cvrp_batch, synthetic_state_dict

TC = os.environ.get("ELG_B200_ATTENTION") == "tensor"
NAMES = (["Q build + list validity + exchange", "bit scan + feature gathers", "local scores + max exchange",
          "local weights -> TMEM, sync, MMA1 issue", "MMA1 wait + ol + sync + MMA2/QK issue", "local finalize (MMA2 wait)",
          "softmax+P (4 rounds)", "O operand + score issue", "score MMA wait", "B3", "select+C", "end barrier", "-", "-", "-", "-"] if TC else
         ["A", "A-barrier", "B1", "copy", "copy-barrier", "B3+C", "end-barrier", "-"] + ["-"] * 8)
dev = "cuda:0"
fn = _lib.lib.elg_debug_phase_clocks_tc if TC else _lib.lib.elg_debug_phase_clocks
model = CVRPModel(**dict(DEFAULT_MODEL_PARAMS["cvrp"]))
model.decoder.add_local_policy(dev)
model.load_state_dict(synthetic_state_dict("cvrp", seed=1234))
model = model.to(dev).eval().requires_grad_(False)
env = CVRPEnv(100, dev)
out = (C.c_ulonglong * (32 if TC else 16))()
for i in range(2):
    random.seed(i)
    data = {k: v.to(dev) for k, v in synthetic_cvrp_batch(400, 100, seed=100 + i).items()}
    solve_batch(model, env, data, 8)
    torch.cuda.synchronize()
    fn(out, 1)
tot = float(sum(out[:16]))
for n, v in zip(NAMES, out[:16]):
    if n != "-":
        print("%-44s %6.2f %%" % (n, 100.0 * v / tot))
if TC:
    # (slot, name) in the order of a round; slot 5 counts the rounds
    SM_NAMES = [(0, "S wait (mbarrier of the group)"), (1, "tcgen05.ld + mask/max"), (2, "pair exchange of the row maximum"),
                (3, "ex2 + hi/lo + tcgen05.st"), (4, "group / CTA barrier + MMA issue")]
    for g in range(2):
        grp = out[16 + 8 * g:24 + 8 * g]
        rounds = max(grp[5], 1)
        total = sum(grp[i] for i, _ in SM_NAMES)
        print("softmax rounds, group %d (%d rounds, %.0f cycles per round):" % (g, rounds, total / rounds))
        for i, n in SM_NAMES:
            print("  %-44s %6.0f cycles  %6.2f %% of the step" % (n, grp[i] / rounds, 100.0 * grp[i] / tot))
