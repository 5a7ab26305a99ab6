"""Drop-in for the reference's CVRPEnv (CVRP/CVRPEnv.py:34-318) on bit-mask device state.

Public surface kept: CVRPEnv(multi_width, device), load_random_problems, load_vrplib_problem,
reset, reset_width, pre_step, step, get_cur_feature, compute_unscaled_reward, and the attributes
callers read (batch_size, problem_size, multi_width, depot_node_xy, depot_node_demand,
selected_node_list, reset_state, step_state).  `capacity` additionally keeps the vehicle capacity of a library
instance (None for random problems, whose demands arrive already normalised); the drivers' local search needs it.  fp32 {0,-inf} masks are produced for API
compatibility; the kernels work on 128-bit visited/mask words per row.
"""
import torch

from .. import engine


class Reset_State:
    """depot_xy (B,1,2), node_xy (B,N,2), node_demand (B,N), dist (B,N+1,N+1) -- CVRP/CVRPEnv.py:9-18.
    `dist` is computed on first access only (the encoder never reads it)."""

    def __init__(self):
        self.depot_xy = None
        self.node_xy = None
        self.node_demand = None
        self._dist = None
        self._depot_node_xy = None
        self._depot_node_demand = None

    @property
    def dist(self):
        if self._dist is None and self._depot_node_xy is not None:
            self._dist = engine.pairwise_dist(self._depot_node_xy)
        return self._dist

    @dist.setter
    def dist(self, v):
        self._dist = v


class Step_State:
    """selected_count, load (B,M), current_node (B,M), ninf_mask (B,M,N+1), finished (B,M) -- CVRP/CVRPEnv.py:21-31."""

    def __init__(self):
        self.selected_count = None
        self.load = None
        self.current_node = None
        self.ninf_mask = None
        self.finished = None
        self._mask_bits = None


class CVRPEnv:
    _elg_fused = True

    def __init__(self, multi_width, device):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise engine._lib.ElgError("elg_b200.CVRPEnv needs a CUDA device; there is no CPU path")
        self.vrplib = False
        self.problem_size = None
        self.multi_width = multi_width
        self.batch_size = None
        self.depot_node_xy = None          # (batch, problem+1, 2)
        self.depot_node_demand = None      # (batch, problem+1)
        self.unscaled_depot_node_xy = None
        self.capacity = None
        self.input_mask = None
        self.dist = None
        self.selected_count = None
        self.current_node = None
        self.load = None
        self.finished = None
        self.ninf_mask = None
        self.reset_state = Reset_State()
        self.step_state = Step_State()
        self._actions = []
        self._solutions = None

    # ---- problem loading ------------------------------------------------------------------------
    def _publish(self):
        rs = self.reset_state = Reset_State()
        rs._depot_node_xy, rs._depot_node_demand = self.depot_node_xy, self.depot_node_demand
        rs.depot_xy = self.depot_node_xy[:, :1, :]
        rs.node_xy = self.depot_node_xy[:, 1:, :]
        rs.node_demand = self.depot_node_demand[:, 1:]
        self.problem_size = self.depot_node_xy.shape[1] - 1
        self.batch_size = self.depot_node_xy.shape[0]
        self.dist = None

    def load_random_problems(self, batch, aug_factor=1):
        """batch: dict with 'loc' (n,N,2), 'demand' (n,N), 'depot' (n,2)|(n,1,2) -- CVRP/CVRPEnv.py:125-150."""
        if aug_factor not in (1, 8):
            raise NotImplementedError
        self.vrplib = False
        self.capacity = None
        loc = batch['loc'].to(self.device, non_blocking=True)
        demand = batch['demand'].to(self.device, non_blocking=True)
        depot = batch['depot'].to(self.device, non_blocking=True)
        self.depot_node_xy, self.depot_node_demand = engine.load_problems("cvrp", loc, depot, demand, aug=aug_factor)
        self._publish()

    def load_vrplib_problem(self, instance, aug_factor=1):
        """instance: dict with node_coord (N+1,2), demand (N+1,), capacity, depot -- CVRP/CVRPEnv.py:84-123.
        Per-axis min-max scaling; node 0 must be the depot."""
        if aug_factor not in (1, 8):
            raise NotImplementedError
        self.vrplib = True
        self.capacity = instance['capacity']
        coord = torch.FloatTensor(instance['node_coord']).unsqueeze(0).to(self.device)
        demand = torch.FloatTensor(instance['demand']).unsqueeze(0).to(self.device) / instance['capacity']
        lo, hi = coord.min(dim=1, keepdim=True)[0], coord.max(dim=1, keepdim=True)[0]
        scaled = (coord - lo) / (hi - lo)
        n = coord.shape[1] - 1
        self.depot_node_xy, self.depot_node_demand = engine.load_problems(
            "cvrp", scaled[:, 1:, :], scaled[:, :1, :], demand[:, 1:], aug=aug_factor)
        self.unscaled_depot_node_xy, _ = engine.load_problems(
            "cvrp", coord[:, 1:, :], coord[:, :1, :], demand[:, 1:], aug=aug_factor)
        self._publish()
        assert self.problem_size == n

    # ---- episode state ----------------------------------------------------------------------------
    def reset(self):
        B, M, N1 = self.batch_size, self.multi_width, self.problem_size + 1
        dev = self.device
        self.selected_count = 0
        self.current_node = None
        self._actions, self._solutions = [], None
        self.load = torch.ones((B, M), device=dev)
        self.finished = torch.zeros((B, M), dtype=torch.bool, device=dev)
        self._finished_u8 = torch.zeros((B, M), dtype=torch.uint8, device=dev)
        self._visited_bits = torch.zeros((B, M, engine.mask_words(N1)), dtype=torch.int32, device=dev)
        self._mask_bits = torch.zeros((B, M, engine.mask_words(N1)), dtype=torch.int32, device=dev)
        self._counter = torch.zeros(1, dtype=torch.int32, device=dev)
        self.ninf_mask = None
        self._ninf_shape = (B, M, N1)
        return self.reset_state, None, False

    def reset_width(self, new_width):
        self.multi_width = new_width

    def _sync_step_state(self):
        s = self.step_state
        s.selected_count = self.selected_count
        s.load = self.load
        s.current_node = self.current_node
        if self.ninf_mask is None:
            self.ninf_mask = torch.zeros(self._ninf_shape, device=self.device)
        s.ninf_mask = self.ninf_mask
        s.finished = self.finished
        s._mask_bits = self._mask_bits

    def pre_step(self):
        self._sync_step_state()
        return self.step_state, None, False

    def step(self, selected):
        """selected (B, M) int64 -> (Step_State, reward | None, done) -- CVRP/CVRPEnv.py:190-249."""
        if self.ninf_mask is None:
            self.ninf_mask = torch.zeros(self._ninf_shape, device=self.device)
        self.selected_count += 1
        self.current_node = selected
        self._actions.append(selected)
        self._counter.zero_()
        engine.env_step("cvrp", self.depot_node_demand, selected.to(torch.int32).contiguous(), self.load,
                        self._visited_bits, self._mask_bits, self._finished_u8, self.ninf_mask, self._counter)
        self.finished = self._finished_u8.bool()
        self._sync_step_state()
        done = int(self._counter.item()) == 0
        reward = None
        if done:
            reward = self.compute_unscaled_reward() if self.vrplib else self._get_reward()
        return self.step_state, reward, done

    @property
    def selected_node_list(self):
        if self._solutions is not None:
            return self._solutions
        if not self._actions:
            return torch.zeros((self.batch_size, self.multi_width, 0), dtype=torch.long, device=self.device)
        return torch.stack(self._actions, dim=2)

    def _finish_fused(self, solutions, reward):
        """State after a fused rollout (elg_b200.cvrp.utils.rollout)."""
        self._solutions = solutions
        self.selected_count = solutions.shape[2]
        self.current_node = solutions[:, :, -1]
        self.finished = torch.ones_like(self.finished)

    def _get_reward(self):
        return -engine.tour_length(self.depot_node_xy, self.selected_node_list)

    def compute_unscaled_reward(self, solutions=None, rounding=True):
        if solutions is None:
            solutions = self.selected_node_list
        return -engine.tour_length(self.unscaled_depot_node_xy, solutions, rounding=rounding)

    def get_cur_feature(self):
        """(cur_dist, cur_theta, relative_xy, norm_demand) -- CVRP/CVRPEnv.py:291-318."""
        if self.current_node is None:
            return None, None, None, None
        return engine.cur_feature(self.depot_node_xy, self.current_node, self.depot_node_demand, self.load)
