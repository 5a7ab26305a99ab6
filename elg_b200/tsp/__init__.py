from .TSPEnv import TSPEnv, Reset_State, Step_State
from .TSPModel import TSPModel
from .utils import augment_xy_data_by_8_fold, batched_two_opt_torch, check_feasible, rollout, seed_everything, tsp_local_search
