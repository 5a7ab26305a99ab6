"""Host-side engine: owns device buffers (torch tensors) and calls the C ABI.

PyTorch is plumbing here (device memory, streams); all compute on the hot path is in
libelg_b200.so.  Nothing in this module runs the path on the CPU: tensors must live on a
CUDA device and the calls raise otherwise.
"""
import ctypes as C
import os

import torch

from . import _lib
from ._lib import ELG_CVRP, ELG_GREEDY, ELG_SAMPLE, ELG_TSP, check, lib


def _ptr(t):
    return C.c_void_p(0) if t is None else C.c_void_p(t.data_ptr())


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _require_cuda(t, what):
    if not t.is_cuda:
        raise _lib.ElgError("%s must be a CUDA tensor: elg_b200 has no CPU path" % what)


def make_desc(problem, model_params):
    p = model_params
    flags = ((_lib.FLAG_ENSEMBLE if p.get("ensemble", True) else 0) |
             (_lib.FLAG_DISTANCE_PENALTY if p.get("distance_penalty", True) else 0) |
             (_lib.FLAG_POSITIONAL if p.get("positional", True) else 0))
    if p.get("ensemble_size", 1) != 1 or p.get("euclidean", False) or (problem == "cvrp" and not p.get("demand", True)):
        raise _lib.ElgError("only the released configuration is implemented (ensemble_size=1, euclidean=False, demand=True)")
    return _lib.ModelDesc(ELG_CVRP if problem == "cvrp" else ELG_TSP, p["embedding_dim"], p["head_num"], p["qkv_dim"],
                          p["ff_hidden_dim"], p["encoder_layer_num"], p["local_size"][0], p["local_att_hidden_dim"],
                          p["local_att_head_num"], p["local_att_qkv_dim"], float(p["xi"]), float(p["logit_clipping"]), flags)


def weight_slots(problem, desc):
    """state_dict key -> (offset, numel) inside the packed weight buffer (elg_weight_layout)."""
    L = _lib.WeightLayout()
    check(lib.elg_weight_layout(desc, L))
    cv = problem == "cvrp"
    n1, ff, n2 = (("add_n_normalization_1", "feed_forward", "add_n_normalization_2") if cv else
                  ("addAndNormalization1", "feedForward", "addAndNormalization2"))
    m = {}
    if cv:
        m["encoder.embedding_depot.weight"] = L.emb_depot_w
        m["encoder.embedding_depot.bias"] = L.emb_depot_b
        m["encoder.embedding_node.weight"] = L.emb_node_w
        m["encoder.embedding_node.bias"] = L.emb_node_b
    else:
        m["encoder.embedding.weight"] = L.emb_node_w
        m["encoder.embedding.bias"] = L.emb_node_b
    for i in range(desc.layers):
        y, pre = L.layer[i], "encoder.layers.%d." % i
        m.update({pre + "Wq.weight": y.wq, pre + "Wk.weight": y.wk, pre + "Wv.weight": y.wv,
                  pre + "multi_head_combine.weight": y.wo, pre + "multi_head_combine.bias": y.bo,
                  pre + n1 + ".norm.weight": y.n1w, pre + n1 + ".norm.bias": y.n1b,
                  pre + ff + ".W1.weight": y.w1, pre + ff + ".W1.bias": y.b1,
                  pre + ff + ".W2.weight": y.w2, pre + ff + ".W2.bias": y.b2,
                  pre + n2 + ".norm.weight": y.n2w, pre + n2 + ".norm.bias": y.n2b})
    if not cv:
        m["decoder.Wq_first.weight"] = L.dec_wq_first
    m.update({"decoder.Wq_last.weight": L.dec_wq_last, "decoder.Wk.weight": L.dec_wk, "decoder.Wv.weight": L.dec_wv,
              "decoder.multi_head_combine.weight": L.dec_wo, "decoder.multi_head_combine.bias": L.dec_bo})
    lp = "decoder.local_policies.0." if cv else "decoder.local_policy_0."
    m.update({lp + "cur_token_emb": L.loc_token, lp + "init_emb.weight": L.loc_we, lp + "init_emb.bias": L.loc_be,
              lp + "Wq.weight": L.loc_wq, lp + "Wk.weight": L.loc_wk, lp + "Wv.weight": L.loc_wv,
              lp + "multi_head_combine.weight": L.loc_wo, lp + "multi_head_combine.bias": L.loc_bo})
    return m, int(L.total)


class ModelHandle:
    """Packed weights + folded tables of one model on one device."""

    def __init__(self, problem, model_params, state_dict, device, attention=None):
        """attention: None/"auto" (library chooses per shape), "tensor" (tcgen05 attention kernel whenever eligible) or
        "fp32" (fp32-pipe attention kernel); default from the ELG_B200_ATTENTION environment variable.  Diagnostics only:
        both kernels compute the same decode step."""
        self.problem, self.model_params = problem, dict(model_params)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.ElgError("elg_b200 needs a CUDA device (got %s); there is no CPU path" % device)
        self.desc = make_desc(problem, model_params)
        attention = attention or os.environ.get("ELG_B200_ATTENTION", "auto")
        if attention not in ("auto", "tensor", "fp32"):
            raise ValueError("attention must be auto, tensor or fp32")
        self.desc.flags |= {"auto": 0, "tensor": _lib.FLAG_ATTN_TENSOR, "fp32": _lib.FLAG_ATTN_FP32}[attention]
        slots, total = weight_slots(problem, self.desc)
        local_keys = [k for k in slots if ".local_polic" in k]
        self.has_local = bool(self.desc.flags & _lib.FLAG_ENSEMBLE) and all(k in state_dict for k in local_keys)
        if not self.has_local:
            # model_params['ensemble'] False, or the reference's decoder before add_local_policy (CVRP/models.py:294-297,
            # 409): global policy + distance penalty only; the local slots of the packed buffer stay zero
            self.desc.flags &= ~_lib.FLAG_ENSEMBLE
            slots = {k: o for k, o in slots.items() if k not in local_keys}
        missing = [k for k in slots if k not in state_dict]
        if missing:
            raise KeyError("state_dict is missing %s" % missing[:3])
        host = torch.zeros(total, dtype=torch.float32)
        for k, off in slots.items():
            v = state_dict[k].detach().to("cpu", torch.float32).reshape(-1)
            host[off:off + v.numel()] = v
        self.weights = host.to(self.device)
        self.derived = torch.empty(int(lib.elg_derived_floats(self.desc)), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib.elg_prepare_model(self.desc, _ptr(self.weights), _ptr(self.derived), _stream(self.device)))


class EncodedBatch:
    """Device tables of one encoded batch (elg_tables) with the tensors that back them."""

    def __init__(self, handle, xy, demand=None, unscaled=None):
        _require_cuda(xy, "xy")
        self.handle = handle
        self.B, self.N1 = int(xy.shape[0]), int(xy.shape[1])
        dev, f32 = xy.device, torch.float32
        B, N1 = self.B, self.N1
        self.xy = xy.contiguous().to(f32)
        self.demand = None if demand is None else demand.contiguous().to(f32)
        self.unscaled = None if unscaled is None else unscaled.contiguous().to(f32)
        if self.unscaled is not None and self.unscaled.shape[0] != B:
            self.unscaled = self.unscaled.expand(B, -1, -1).contiguous()
        big = torch.empty((4 if handle.problem == "tsp" else 3, B, N1, 128), dtype=f32, device=dev)
        self.enc = torch.empty((B, N1, 128), dtype=f32, device=dev)
        self.k, self.v, self.qtab = big[0], big[1], big[2]
        self.qfirst = big[3] if handle.problem == "tsp" else None
        self.e = torch.empty(int(lib.elg_e_bytes(handle.desc, B, N1)), dtype=torch.uint8, device=dev)
        self.eb = torch.empty((B, N1), dtype=f32, device=dev)
        self.nbr = torch.empty(int(lib.elg_nbr_bytes(handle.desc, B, N1)),
                               dtype=torch.uint8, device=dev)
        self._big = big
        # large instances: the operands once more as tcgen05 tiles for the streamed tensor-core rollout (0 bytes if resident)
        n_et = int(lib.elg_et_bytes(handle.desc, B, N1))
        self.et = torch.empty(n_et, dtype=torch.uint8, device=dev) if n_et else None
        self.ws = None
        self.tables = _lib.Tables(*[_ptr(x).value for x in (self.xy, self.demand, self.unscaled, self.enc, self.k, self.v,
                                                             self.e, self.eb, self.qtab, self.qfirst, self.nbr, self.et, None)])


_workspace = {}


def _get_workspace(device, nbytes):
    ws = _workspace.get(device)
    if ws is None or ws.numel() < nbytes:
        ws = None
        _workspace[device] = None
        ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
        _workspace[device] = ws
    return ws


def load_problems(problem, node_xy, depot_xy=None, node_demand=None, aug=1):
    """x8 augmentation + depot/node concatenation on the device -> (xy (aug*n, N1, 2), demand (aug*n, N1) | None)."""
    _require_cuda(node_xy, "node coordinates")
    if aug not in (1, 8):
        raise NotImplementedError
    cv = problem == "cvrp"
    n, nn = int(node_xy.shape[0]), int(node_xy.shape[1])
    N1 = nn + (1 if cv else 0)
    dev = node_xy.device
    node_xy = node_xy.contiguous().float()
    xy = torch.empty((aug * n, N1, 2), dtype=torch.float32, device=dev)
    dem = torch.empty((aug * n, N1), dtype=torch.float32, device=dev) if cv else None
    if cv:
        depot_xy = depot_xy.reshape(n, 2).contiguous().float()
        node_demand = node_demand.contiguous().float()
    with torch.cuda.device(dev):
        check(lib.elg_load_problems(ELG_CVRP if cv else ELG_TSP, _ptr(depot_xy if cv else None), _ptr(node_xy),
                                    _ptr(node_demand if cv else None), n, nn, aug, _ptr(xy), _ptr(dem), _stream(dev)))
    return xy, dem


def pairwise_dist(xy):
    _require_cuda(xy, "xy")
    B, N1 = int(xy.shape[0]), int(xy.shape[1])
    out = torch.empty((B, N1, N1), dtype=torch.float32, device=xy.device)
    with torch.cuda.device(xy.device):
        check(lib.elg_pairwise_dist(_ptr(xy.contiguous()), B, N1, _ptr(out), _stream(xy.device)))
    return out


def encode(handle, xy, demand=None, unscaled=None):
    batch = EncodedBatch(handle, xy, demand, unscaled)
    dev = batch.xy.device
    nbytes = int(lib.elg_encode_workspace_bytes(handle.desc, batch.B, batch.N1))
    ws = _get_workspace(dev, nbytes)
    with torch.cuda.device(dev):
        check(lib.elg_encode(handle.desc, _ptr(handle.weights), _ptr(handle.derived), batch.tables, batch.B, batch.N1,
                             _ptr(ws), nbytes, _stream(dev)))
    return batch


# when set to a list, rollout() appends (start_event, end_event, n_steps tensor) around the kernel launch
profile_events = None


def rollout(batch, M, start_nodes, mode="greedy", seed=0, sync_tours=True):
    """Whole construction rollout in one launch.

    Returns (tours int16 (B, M, t_max) device buffer, reward (B, M), logp (B, M) | None, n_steps tensor).
    The batch length T is n_steps.max(); tours[:, :, T:] is zero padding.
    """
    h = batch.handle
    dev = batch.xy.device
    B, N1 = batch.B, batch.N1
    t_max = 2 * N1 + 2 if h.problem == "cvrp" else N1
    tiles = int(lib.elg_rollout_tiles(h.desc, B, M, N1))
    if tiles <= 0:
        raise _lib.ElgError("unsupported rollout shape B=%d M=%d N1=%d: %s" % (B, M, N1, lib.elg_last_error().decode()))
    start = torch.as_tensor(start_nodes, dtype=torch.int32).to(dev, non_blocking=True).contiguous()
    if start.numel() != M:
        raise ValueError("start_nodes must have M=%d entries" % M)
    tours = torch.zeros((B, M, t_max), dtype=torch.int16, device=dev)
    reward = torch.empty((B, M), dtype=torch.float32, device=dev)
    n_steps = torch.zeros(B * tiles + 1, dtype=torch.int32, device=dev)      # last slot = work counter
    logp = torch.empty((B, M), dtype=torch.float32, device=dev) if mode == "sample" else None
    n_ws = int(lib.elg_rollout_ws_bytes(h.desc, B, M, N1)) if (batch.et is not None and mode == "greedy") else 0
    if n_ws:
        if batch.ws is None or batch.ws.numel() < n_ws:
            batch.ws = torch.empty(n_ws, dtype=torch.uint8, device=dev)
        batch.tables.ws = batch.ws.data_ptr()
    else:
        batch.tables.ws = None
    with torch.cuda.device(dev):
        if profile_events is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(torch.cuda.current_stream(dev))
        check(lib.elg_rollout(h.desc, _ptr(h.derived), batch.tables, B, M, N1, _ptr(start),
                              ELG_SAMPLE if mode == "sample" else ELG_GREEDY, int(seed) & (2 ** 64 - 1), t_max,
                              _ptr(tours), _ptr(reward), _ptr(n_steps), _ptr(logp),
                              C.c_void_p(n_steps.data_ptr() + 4 * B * tiles), _stream(dev)))
        if profile_events is not None:
            ev1.record(torch.cuda.current_stream(dev))
            profile_events.append((ev0, ev1, n_steps[:B * tiles], tiles))
    return tours, reward, logp, n_steps[:B * tiles]


def mask_words(N1):
    return (int(N1) + 31) // 32


def pack_mask_bits(ninf_mask):
    """(B, M, N1) fp32 {0,-inf} (or bool, True = masked) -> (B, M, ceil(N1/32)) int32 bit words."""
    m = ninf_mask if ninf_mask.dtype == torch.bool else torch.isinf(ninf_mask)
    B, M, N1 = m.shape
    W = mask_words(N1)
    pad = torch.zeros((B, M, W * 32), dtype=torch.int64, device=m.device)
    pad[:, :, :N1] = m
    w = (pad.view(B, M, W, 32) << torch.arange(32, device=m.device, dtype=torch.int64)).sum(-1)
    return torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32).contiguous()


def decode_step(batch, M, cur, mask_bits, load=None, first=None, mode="greedy", seed=0, step=0, want_logits=False):
    h = batch.handle
    dev = batch.xy.device
    B, N1 = batch.B, batch.N1
    cur = cur.to(torch.int32).contiguous()
    load = None if load is None else load.float().contiguous()
    first = None if first is None else first.to(torch.int32).contiguous()
    sel = torch.empty((B, M), dtype=torch.int32, device=dev)
    prob = torch.empty((B, M), dtype=torch.float32, device=dev) if mode == "sample" else None
    logits = torch.empty((B, M, N1), dtype=torch.float32, device=dev) if want_logits else None
    with torch.cuda.device(dev):
        check(lib.elg_decode_step(h.desc, _ptr(h.derived), batch.tables, B, M, N1, _ptr(cur), _ptr(load), _ptr(first),
                                  _ptr(mask_bits), ELG_SAMPLE if mode == "sample" else ELG_GREEDY,
                                  int(seed) & (2 ** 64 - 1), int(step), _ptr(sel), _ptr(prob), _ptr(logits), _stream(dev)))
    return sel.long(), prob, logits


def env_step(problem, demand, selected, load, visited_bits, mask_bits, finished, ninf_mask=None, counter=None):
    dev = selected.device
    B, M = selected.shape
    N1 = int(demand.shape[1]) if demand is not None else int(ninf_mask.shape[2])
    with torch.cuda.device(dev):
        check(lib.elg_env_step(ELG_CVRP if problem == "cvrp" else ELG_TSP, _ptr(demand), B, M, N1,
                               _ptr(selected), _ptr(load), _ptr(visited_bits), _ptr(mask_bits), _ptr(finished),
                               _ptr(ninf_mask), _ptr(counter), _stream(dev)))


def cur_feature(xy, cur, demand=None, load=None):
    dev = xy.device
    B, N1 = int(xy.shape[0]), int(xy.shape[1])
    M = int(cur.shape[1])
    f32 = torch.float32
    cur_dist = torch.empty((B, M, N1), dtype=f32, device=dev)
    theta = torch.empty((B, M, N1), dtype=f32, device=dev)
    rel = torch.empty((B, M, N1, 2), dtype=f32, device=dev)
    nd = torch.empty((B, M, N1), dtype=f32, device=dev) if demand is not None else None
    cur32 = cur.to(torch.int32).contiguous()
    with torch.cuda.device(dev):
        check(lib.elg_cur_feature(_ptr(xy), _ptr(demand), _ptr(load), _ptr(cur32), B, M, N1, _ptr(cur_dist), _ptr(theta),
                                  _ptr(rel), _ptr(nd), _stream(dev)))
    return cur_dist, theta, rel, nd


def tour_length(xy, tours, rounding=False):
    _require_cuda(xy, "xy")
    B, M, T = tours.shape
    out = torch.empty((B, M), dtype=torch.float32, device=tours.device)
    t64 = tours.to(torch.int64).contiguous()
    xy = xy.contiguous().float()
    with torch.cuda.device(tours.device):
        check(lib.elg_tour_length(_ptr(xy), int(xy.shape[0]), _ptr(t64), B, M, T, int(xy.shape[1]), 1 if rounding else 0,
                                  _ptr(out), _stream(tours.device)))
    return out


def two_opt(problem, xy, tours, inst=None, max_iterations=1000, rounding=False):
    """Best-improvement 2-opt local search (elg_two_opt; semantics in include/elg_b200.h), one launch for all tours.

    xy (Bxy, N1, 2) coordinates; tours (R, L) int16 (the rollout's rows) or int64 node ids: tsp a permutation in positions
    0..N1-1 that keeps its start node, cvrp a depot-delimited row whose moves stay inside one route; inst (R,) picks the xy
    instance of every tour (default: tour r uses xy[r], or xy[0] when Bxy == 1); rounding rint()s every edge (library
    metric).  Returns (tours int64 (R, L), length (R,) as tour_length measures it, iterations (R,) moves applied)."""
    _require_cuda(xy, "xy")
    _require_cuda(tours, "tours")
    if tours.dim() != 2 or xy.dim() != 3 or xy.shape[2] != 2:
        raise ValueError("tours must be (R, L) and xy (Bxy, N1, 2)")
    if max_iterations < 0:
        raise ValueError("max_iterations must be >= 0")
    dev = tours.device
    R, L = tours.shape
    Bxy, N1 = int(xy.shape[0]), int(xy.shape[1])
    n = L if problem == "cvrp" else min(N1, L)
    if R and n:
        lo, hi = torch.aminmax(tours[:, :n])
        if int(lo) < 0 or int(hi) >= N1:
            raise ValueError("tour node ids must lie in [0, %d)" % N1)
    if inst is not None:
        inst = torch.as_tensor(inst, device=dev).to(torch.int32).contiguous()
        if inst.shape != (R,) or (R and (int(inst.min()) < 0 or int(inst.max()) >= Bxy)):
            raise ValueError("inst must be (R,) indices into the %d xy instances" % Bxy)
    t16 = tours.to(torch.int16, copy=True).contiguous()
    length = torch.empty(R, dtype=torch.float32, device=dev)
    iters = torch.empty(R, dtype=torch.int32, device=dev)
    xy = xy.contiguous().float()
    with torch.cuda.device(dev):
        check(lib.elg_two_opt(ELG_CVRP if problem == "cvrp" else ELG_TSP, _ptr(xy), Bxy, N1, _ptr(inst), _ptr(t16), R, L,
                              1 if rounding else 0, int(max_iterations), _ptr(iters), _ptr(length), _stream(dev)))
    return t16.long(), length, iters


def tsp_local_search(xy, tours, inst=None, max_iterations=1000, max_segment=3, rounding=False):
    """Best-improvement TSP local search with 2-opt and Or-opt moves (elg_tsp_local_search; semantics in
    include/elg_b200.h), one launch for all tours.

    xy (Bxy, N1, 2) coordinates; tours (R, L) int16 or int64 with a permutation of 0..N1-1 in positions 0..N1-1 (L >= N1;
    the rest is left as it is); inst (R,) picks the xy instance of every tour (default: tour r uses xy[r], or xy[0] when
    Bxy == 1); max_segment (0..3) the longest Or-opt segment, 0 being plain 2-opt; rounding rint()s every edge (library
    metric).  Position 0 never moves.  Returns (tours int64 (R, L), length (R,) as tour_length measures it,
    iterations (R,) moves applied)."""
    if tours.dim() != 2 or xy.dim() != 3 or xy.shape[2] != 2:
        raise ValueError("tours must be (R, L) and xy (Bxy, N1, 2)")
    R, L = tours.shape
    Bxy, N1 = int(xy.shape[0]), int(xy.shape[1])
    if L < N1:
        raise ValueError("tours need at least N1 = %d positions (got %d)" % (N1, L))
    if max_iterations < 0:
        raise ValueError("max_iterations must be >= 0")
    if max_segment not in (0, 1, 2, 3):
        raise ValueError("max_segment must be 0, 1, 2 or 3 (got %r)" % (max_segment,))
    dev = tours.device
    if inst is not None:
        inst = torch.as_tensor(inst, device=dev).to(torch.int32).contiguous()
        if inst.shape != (R,) or (R and (int(inst.min()) < 0 or int(inst.max()) >= Bxy)):
            raise ValueError("inst must be (R,) indices into the %d xy instances" % Bxy)
    elif Bxy not in (1, R):
        raise ValueError("without inst, xy must hold 1 or R instances (got %d for %d rows)" % (Bxy, R))
    if R and N1:
        t = tours[:, :N1].long()
        if int(t.min()) < 0 or int(t.max()) >= N1:
            raise ValueError("tour node ids must lie in [0, %d)" % N1)
        if not torch.equal(t.sort(1)[0], torch.arange(N1, device=dev).expand(R, -1)):
            raise ValueError("positions 0..%d of every tour must hold a permutation of the nodes" % (N1 - 1))
    _require_cuda(xy, "xy")
    _require_cuda(tours, "tours")
    t16 = tours.to(torch.int16, copy=True).contiguous()
    length = torch.empty(R, dtype=torch.float32, device=dev)
    iters = torch.empty(R, dtype=torch.int32, device=dev)
    xy = xy.contiguous().float()
    with torch.cuda.device(dev):
        check(lib.elg_tsp_local_search(_ptr(xy), Bxy, N1, _ptr(inst), _ptr(t16), R, L, int(max_segment),
                                       1 if rounding else 0, int(max_iterations), _ptr(iters), _ptr(length), _stream(dev)))
    return t16.long(), length, iters


def cvrp_local_search(xy, tours, demand, capacity, inst=None, max_iterations=1000, rounding=False):
    """Capacity-aware best-improvement CVRP local search (elg_cvrp_local_search; semantics in include/elg_b200.h): 2-opt
    inside a route, relocate, swap and 2-opt* between routes, one launch for all rows.

    xy (Bxy, N1, 2) coordinates; tours (R, L) rollout rows, int16 or int64, with every customer exactly once, position 0
    the depot and every route within capacity; demand (Bxy, N1) normalised demands as CVRPEnv holds them (depot 0);
    capacity the integer vehicle capacity: demands in units are rint(demand * capacity) and must lie within 1e-3 of it.
    inst (R,) picks the xy / demand instance of every row (default: row r uses instance r, or 0 when Bxy == 1); rounding
    rint()s every edge (library metric).  Returns (canonical tours int64 (R, L), length (R,) as tour_length measures it,
    iterations (R,) moves applied)."""
    if tours.dim() != 2 or xy.dim() != 3 or xy.shape[2] != 2 or demand.shape != xy.shape[:2]:
        raise ValueError("tours must be (R, L), xy (Bxy, N1, 2) and demand (Bxy, N1)")
    if max_iterations < 0:
        raise ValueError("max_iterations must be >= 0")
    if int(capacity) != capacity or capacity <= 0:
        raise ValueError("capacity must be a positive integer (got %r)" % (capacity,))
    capacity = int(capacity)
    dev = tours.device
    R, L = tours.shape
    Bxy, N1 = int(xy.shape[0]), int(xy.shape[1])
    scaled = demand.double() * capacity
    units = torch.round(scaled)
    if bool(((scaled - units).abs() > 1e-3).any()):
        raise ValueError("demand * capacity must be integral (within 1e-3): demands are whole units of the capacity")
    units = units.to(torch.int32).contiguous()
    if inst is not None:
        inst = torch.as_tensor(inst, device=dev).to(torch.int32).contiguous()
        if inst.shape != (R,) or (R and (int(inst.min()) < 0 or int(inst.max()) >= Bxy)):
            raise ValueError("inst must be (R,) indices into the %d xy instances" % Bxy)
    elif Bxy not in (1, R):
        raise ValueError("without inst, xy must hold 1 or R instances (got %d for %d rows)" % (Bxy, R))
    if R:
        t = tours.long()
        if int(t.min()) < 0 or int(t.max()) >= N1 or bool((t[:, 0] != 0).any()):
            raise ValueError("rows must hold node ids in [0, %d) with the depot at position 0" % N1)
        counts = torch.zeros(R, N1, dtype=torch.int32, device=dev).scatter_add_(1, t, torch.ones_like(t, dtype=torch.int32))
        if not bool((counts[:, 1:] == 1).all()):
            raise ValueError("every row must visit each customer 1..%d exactly once" % (N1 - 1))
        which = inst.long() if inst is not None else (torch.arange(R, device=dev) if Bxy > 1 else torch.zeros(R, dtype=torch.long, device=dev))
        d = units[which].gather(1, t)
        route = (t == 0).long().cumsum(1)
        loads = torch.zeros(R, L + 1, dtype=torch.int64, device=dev).scatter_add_(1, route, d.long())
        if int(loads.max()) > capacity:
            raise ValueError("an input route exceeds the capacity %d" % capacity)
    _require_cuda(xy, "xy")
    _require_cuda(tours, "tours")
    _require_cuda(units, "demand")
    t16 = tours.to(torch.int16, copy=True).contiguous()
    length = torch.empty(R, dtype=torch.float32, device=dev)
    iters = torch.empty(R, dtype=torch.int32, device=dev)
    xy = xy.contiguous().float()
    with torch.cuda.device(dev):
        check(lib.elg_cvrp_local_search(_ptr(xy), Bxy, N1, _ptr(units), capacity, _ptr(inst), _ptr(t16), R, L,
                                        1 if rounding else 0, int(max_iterations), _ptr(iters), _ptr(length), _stream(dev)))
    return t16.long(), length, iters


# ---------------------------------------------------------------------------------------------- training path
def encode_train(handle, xy, demand=None):
    """model.pre_forward for a training step: elg_encode that also keeps every layer's activations.
    Returns (EncodedBatch, saved-activation buffer)."""
    batch = EncodedBatch(handle, xy, demand, None)
    dev = batch.xy.device
    nbytes = int(lib.elg_train_saved_bytes(handle.desc, batch.B, batch.N1))
    saved = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(lib.elg_encode_train(handle.desc, _ptr(handle.weights), _ptr(handle.derived), batch.tables, batch.B, batch.N1,
                                   _ptr(saved), nbytes, _stream(dev)))
    return batch, saved


_train_ws = {}
# when set to a list, reinforce_backward() appends (start_event, end_event, row-steps differentiated)
train_profile_events = None


def reinforce_backward(batch, saved, M, tours, T, reward, logp=None, scale_norm=True, chunk_steps=16, grads=None):
    """J.backward() of the reference's training step (CVRP/train.py:112-124) for the recorded rollout.
    Returns (grads packed like handle.weights, loss (1,) tensor, workspace tensor)."""
    h = batch.handle
    dev = batch.xy.device
    B, N1 = batch.B, batch.N1
    t_max = int(tours.shape[2])
    nbytes = int(lib.elg_train_workspace_bytes(h.desc, B, M, N1, t_max, int(chunk_steps)))
    if nbytes == 0:
        raise _lib.ElgError("unsupported training shape: %s" % lib.elg_last_error().decode())
    ws = _train_ws.get(dev)
    if ws is None or ws.numel() < nbytes:
        _train_ws[dev] = None
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _train_ws[dev] = ws
    if grads is None:
        grads = torch.empty_like(h.weights)
    loss = torch.zeros(1, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        if train_profile_events is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(torch.cuda.current_stream(dev))
        check(lib.elg_reinforce_backward(h.desc, _ptr(h.weights), _ptr(h.derived), batch.tables, _ptr(saved), B, M, N1,
                                         _ptr(tours), t_max, int(T), _ptr(reward.contiguous()), _ptr(logp), 1 if scale_norm else 0,
                                         _ptr(grads), _ptr(loss), _ptr(ws), ws.numel(), _stream(dev)))
        if train_profile_events is not None:
            ev1.record(torch.cuda.current_stream(dev))
            train_profile_events.append((ev0, ev1, B * M * max(int(T) - (2 if h.problem == "cvrp" else 1), 0)))
    return grads, loss, ws


def train_workspace_layout(handle, B, M, N1, t_max):
    out = (C.c_int64 * 8)()
    check(lib.elg_train_workspace_layout(handle.desc, B, M, N1, t_max, out))
    names = ("dEp", "dK", "dV", "dqtab", "dqfirst", "deb", "dwl", "lg")
    return dict(zip(names, [int(x) for x in out]))


def adam_step(params, grads, exp_avg, exp_avg_sq, step, lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=1e-6,
              grad_scale=1.0):
    dev = params.device
    with torch.cuda.device(dev):
        check(lib.elg_adam_step(_ptr(params), _ptr(grads), _ptr(exp_avg), _ptr(exp_avg_sq), params.numel(), int(step),
                                lr, beta1, beta2, eps, weight_decay, grad_scale, _stream(dev)))


def prepare_model(handle):
    """Re-fold the decoder / local-policy tables after the packed weights changed (optimizer step)."""
    with torch.cuda.device(handle.device):
        check(lib.elg_prepare_model(handle.desc, _ptr(handle.weights), _ptr(handle.derived), _stream(handle.device)))
