"""ctypes binding of libelg_b200.so (the C ABI declared in include/elg_b200.h).

There is no CPU or PyTorch fallback: if the CUDA library has not been built, importing
this module raises.  Build it with `python -m elg_b200.build` (or `__graft_entry__.build()`).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ELG_B200_LIB: a diagnostic build of the same sources (tools/phase_timing.py: `python -m elg_b200.build --variant timing`)
LIB_PATH = os.environ.get("ELG_B200_LIB") or os.path.join(_HERE, "csrc", "libelg_b200.so")

ELG_TSP, ELG_CVRP = 0, 1
ELG_GREEDY, ELG_SAMPLE = 0, 1
FLAG_ENSEMBLE, FLAG_DISTANCE_PENALTY, FLAG_POSITIONAL = 1, 2, 4
FLAG_ATTN_FP32, FLAG_ATTN_TENSOR = 8, 16
MAX_LAYERS = 16
NBR_STRIDE = 128
ABI_VERSION = 4


class ModelDesc(C.Structure):
    _fields_ = [("problem", C.c_int32), ("emb", C.c_int32), ("heads", C.c_int32), ("qkv", C.c_int32),
                ("ff", C.c_int32), ("layers", C.c_int32), ("local_k", C.c_int32), ("local_emb", C.c_int32),
                ("local_heads", C.c_int32), ("local_qkv", C.c_int32), ("xi", C.c_float), ("clip", C.c_float),
                ("flags", C.c_int32)]


class _LayerLayout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("wq", "wk", "wv", "wo", "bo", "n1w", "n1b", "w1", "b1", "w2", "b2", "n2w", "n2b")]


class WeightLayout(C.Structure):
    _fields_ = ([("total", C.c_int64), ("emb_depot_w", C.c_int64), ("emb_depot_b", C.c_int64),
                 ("emb_node_w", C.c_int64), ("emb_node_b", C.c_int64), ("layer", _LayerLayout * MAX_LAYERS)] +
                [(n, C.c_int64) for n in ("dec_wq_first", "dec_wq_last", "dec_wk", "dec_wv", "dec_wo", "dec_bo",
                                          "loc_token", "loc_we", "loc_be", "loc_wq", "loc_wk", "loc_wv", "loc_wo",
                                          "loc_bo")])


class Tables(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("xy", "demand", "unscaled", "enc", "k", "v", "e", "eb", "qtab", "qfirst", "nbr", "et", "ws")]


# name -> (restype, argtypes); every symbol include/elg_b200.h declares
_P, _I, _U64, _SZ = C.c_void_p, C.c_int, C.c_uint64, C.c_size_t
SYMBOLS = {
    "elg_abi_version": (_I, []),
    "elg_last_error": (C.c_char_p, []),
    "elg_launch_count": (_U64, []),
    "elg_weight_layout": (_I, [C.POINTER(ModelDesc), C.POINTER(WeightLayout)]),
    "elg_derived_floats": (C.c_int64, [C.POINTER(ModelDesc)]),
    "elg_prepare_model": (_I, [C.POINTER(ModelDesc), _P, _P, _P]),
    "elg_load_problems": (_I, [_I, _P, _P, _P, _I, _I, _I, _P, _P, _P]),
    "elg_pairwise_dist": (_I, [_P, _I, _I, _P, _P]),
    "elg_encode_workspace_bytes": (_SZ, [C.POINTER(ModelDesc), _I, _I]),
    "elg_encode": (_I, [C.POINTER(ModelDesc), _P, _P, C.POINTER(Tables), _I, _I, _P, _SZ, _P]),
    "elg_rollout_tiles": (_I, [C.POINTER(ModelDesc), _I, _I, _I]),
    "elg_rollout_resident": (_I, [C.POINTER(ModelDesc), _I]),
    "elg_nbr_bytes": (_SZ, [C.POINTER(ModelDesc), _I, _I]),
    "elg_e_bytes": (_SZ, [C.POINTER(ModelDesc), _I, _I]),
    "elg_et_bytes": (_SZ, [C.POINTER(ModelDesc), _I, _I]),
    "elg_rollout_ws_bytes": (_SZ, [C.POINTER(ModelDesc), _I, _I, _I]),
    "elg_rollout": (_I, [C.POINTER(ModelDesc), _P, C.POINTER(Tables), _I, _I, _I, _P, _I, _U64, _I, _P, _P, _P, _P, _P, _P]),
    "elg_decode_step": (_I, [C.POINTER(ModelDesc), _P, C.POINTER(Tables), _I, _I, _I, _P, _P, _P, _P, _I, _U64, _U64,
                             _P, _P, _P, _P]),
    "elg_env_step": (_I, [_I, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "elg_cur_feature": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P]),
    "elg_tour_length": (_I, [_P, _I, _P, _I, _I, _I, _I, _I, _P, _P]),
    "elg_two_opt": (_I, [_I, _P, _I, _I, _P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "elg_cvrp_local_search": (_I, [_P, _I, _I, _P, _I, _P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "elg_tsp_local_search": (_I, [_P, _I, _I, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "elg_train_saved_bytes": (_SZ, [C.POINTER(ModelDesc), _I, _I]),
    "elg_encode_train": (_I, [C.POINTER(ModelDesc), _P, _P, C.POINTER(Tables), _I, _I, _P, _SZ, _P]),
    "elg_train_workspace_bytes": (_SZ, [C.POINTER(ModelDesc), _I, _I, _I, _I, _I]),
    "elg_train_workspace_layout": (_I, [C.POINTER(ModelDesc), _I, _I, _I, _I, C.POINTER(C.c_int64)]),
    "elg_reinforce_backward": (_I, [C.POINTER(ModelDesc), _P, _P, C.POINTER(Tables), _P, _I, _I, _I, _P, _I, _I, _P, _P,
                                    _I, _P, _P, _P, _SZ, _P]),
    "elg_adam_step": (_I, [_P, _P, _P, _P, C.c_int64, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                           C.c_float, _P]),
    "elg_generate_problems": (_I, [_I, _I, _I, _I, _I, C.c_float, C.c_float, C.c_float, C.c_float, _U64, _P, _P, _P, _P]),
    "elg_selftest_umma": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
}


class ElgError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ElgError("libelg_b200.so is not built (%s). Run `python -m elg_b200.build`; there is no CPU fallback."
                       % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError here means the .so is stale
        fn.restype, fn.argtypes = res, args
    if lib.elg_abi_version() != ABI_VERSION:
        raise ElgError("libelg_b200.so ABI %d != binding ABI %d; rebuild" % (lib.elg_abi_version(), ABI_VERSION))
    return lib


lib = _load()


def check(rc):
    if rc != 0:
        raise ElgError("elg_b200 call failed (code %d): %s" % (rc, lib.elg_last_error().decode()))


def launch_count():
    return int(lib.elg_launch_count())
