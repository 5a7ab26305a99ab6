from .CVRPEnv import CVRPEnv, Reset_State, Step_State
from .CVRPModel import CVRPModel
from .utils import augment_xy_data_by_8_fold, batched_two_opt_torch, check_feasible, cvrp_local_search, rollout, seed_everything
