"""ctypes binding of include/kge_b200.h.  There is no fallback: if libkge_b200.so is missing or a call
fails, this raises."""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KGE_LIB") or os.path.join(HERE, "csrc", "libkge_b200.so")   # KGE_LIB: an A/B build (build.py)

TRANSE, DISTMULT, COMPLEX, ROTATE, PROTATE = range(5)
MODEL_IDS = {"TransE": TRANSE, "DistMult": DISTMULT, "ComplEx": COMPLEX, "RotatE": ROTATE, "pRotatE": PROTATE}
SINGLE, HEAD_BATCH, TAIL_BATCH = range(3)
MODE_IDS = {"single": SINGLE, "head-batch": HEAD_BATCH, "tail-batch": TAIL_BATCH}
LOSS_NEG_ADVERSARIAL, LOSS_NEG_UNIFORM, LOSS_POSITIVE = range(3)
ERR_INVALID, ERR_CUDA, ERR_DEVICE = -1, -2, -3
SIM_IDS = {"dot": 0, "cosine": 1, "l2": 2, "l1": 3}
TABLE_ENTITY, TABLE_RELATION = range(2)


class KgeModelStruct(Structure):
    _fields_ = [("model", c_int32), ("device", c_int32), ("nentity", c_int64), ("nrelation", c_int64),
                ("hidden_dim", c_int64), ("entity_dim", c_int64), ("relation_dim", c_int64),
                ("gamma", c_float), ("embedding_range", c_float),
                ("entity", c_void_p), ("relation", c_void_p), ("modulus", c_void_p)]


class KgeAdamTensor(Structure):
    _fields_ = [("param", c_void_p), ("grad", c_void_p), ("exp_avg", c_void_p), ("exp_avg_sq", c_void_p),
                ("numel", c_int64), ("step", c_int32), ("l3", c_int32)]


class KgeEntityAdam(Structure):
    _fields_ = [("exp_avg", c_void_p), ("exp_avg_sq", c_void_p), ("step", c_int32), ("reserved", c_int32),
                ("lr", c_double), ("beta1", c_double), ("beta2", c_double), ("eps", c_double),
                ("l3_coefficient", c_double), ("reg_partials", c_void_p), ("n_reg_partials", c_int64)]


PLAN_SINGLE_READ, PLAN_ENTITY_ADAM = 1, 2
PEER_MAX_RANKS, PEER_HANDLE_BYTES = 16, 64


class KgePeerGroup(Structure):
    _fields_ = [("world", c_int32), ("rank", c_int32), ("grad", c_void_p * PEER_MAX_RANKS),
                ("flags", c_void_p * PEER_MAX_RANKS), ("multicast", c_void_p)]


class KgeShard(Structure):
    _fields_ = [("world", c_int32), ("rank", c_int32), ("block", c_void_p * PEER_MAX_RANKS), ("multicast", c_void_p),
                ("block_bytes", c_int64),
                ("gather_offset", c_int64), ("rows_max", c_int64), ("rows_of", c_int32 * PEER_MAX_RANKS)]


# name -> (restype, argtypes): exactly the prototypes of include/kge_b200.h
_M = POINTER(KgeModelStruct)
PROTOTYPES = {
    "kge_abi_version": (c_int, []),
    "kge_last_error": (c_char_p, []),
    "kge_device_check": (c_int, [c_int, POINTER(c_int), POINTER(c_int64)]),
    "kge_score_forward": (c_int, [_M, c_int, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "kge_score_backward": (c_int, [_M, c_int, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "kge_train_rows": (c_int, [_M, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                               c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_int64, c_void_p, c_void_p]),
    "kge_train_workspace_bytes": (c_int64, [_M, c_int64, c_int64]),
    "kge_train_plan": (c_int, [_M, c_int64, c_int64]),
    "kge_debug_row_phase_cycles": (c_int, [POINTER(ctypes.c_uint64), c_int]),
    "kge_train_rows_adam": (c_int, [_M, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                    c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                    POINTER(KgeEntityAdam), c_void_p]),
    "kge_train_rows_begin": (c_int, [_M, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                     c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                     c_void_p, POINTER(c_int32), c_void_p]),
    "kge_train_entity_pass": (c_int, [_M, c_int, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p,
                                      c_void_p]),
    "kge_zero": (c_int, [c_void_p, c_int64, c_void_p]),
    "kge_copy_h2d": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "kge_copy_d2h_sync": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "kge_weight_sum": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "kge_loss_finalize": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_void_p, c_int64,
                                  c_void_p, c_void_p]),
    "kge_adam_step": (c_int, [POINTER(KgeAdamTensor), c_int, c_double, c_double, c_double, c_double, c_double,
                              c_void_p, c_int64, c_void_p, c_void_p]),
    "kge_eval_query_vectors": (c_int, [_M, c_int, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "kge_eval_phase_table": (c_int, [_M, c_void_p, c_void_p]),
    "kge_eval_positive_scores": (c_int, [_M, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "kge_eval_count_ranks": (c_int, [_M, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64,
                                     c_int64, c_void_p, c_void_p, c_void_p]),
    "kge_eval_count_ranks_two_stage": (c_int, [_M, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                               c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "kge_eval_count_ranks_two_stage_approx": (c_int, [_M, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                                      c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                                      c_void_p, c_void_p]),
    "kge_eval_two_stage_band": (c_int, [c_int, c_int64, c_float, POINTER(c_float)]),
    "kge_eval_gemm_supported": (c_int, [_M]),
    "kge_eval_gemm_split": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "kge_eval_gemm_count_ranks": (c_int, [_M, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p,
                                          c_int64, c_void_p, c_void_p, c_void_p]),
    "kge_eval_gemm_band": (c_float, [c_int64]),
    "kge_eval_count_rank_stats": (c_int, [_M, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                          c_int64, c_int64, c_void_p, c_void_p]),
    "kge_eval_count_rank_stats_two_stage": (c_int, [_M, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                                    c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                                    c_void_p]),
    "kge_eval_gemm_count_rank_stats": (c_int, [_M, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                               c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "kge_eval_candidate_rank_stats": (c_int, [_M, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                              c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                              c_void_p]),
    "kge_eval_path_query_vectors": (c_int, [_M, c_int, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p,
                                            c_void_p]),
    "kge_eval_path_bits_dense": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                         c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "kge_eval_path_bits": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64,
                                   c_void_p, c_void_p, c_int64, c_int64, c_int, c_int64, c_int64, c_void_p, c_void_p,
                                   c_void_p, c_void_p]),
    "kge_eval_topk_scratch_bytes": (c_int64, [_M, c_int64, c_int64, c_int64, c_int]),
    "kge_eval_topk": (c_int, [_M, c_int, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p,
                              c_void_p, c_int64, c_void_p]),
    "kge_eval_topk_merge": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "kge_similarity_rows": (c_int, [_M, c_int, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "kge_similarity_norms": (c_int, [_M, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "kge_similarity_topk_scratch_bytes": (c_int64, [_M, c_int, c_int64, c_int64, c_int64, c_int]),
    "kge_similarity_topk": (c_int, [_M, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                    c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "kge_eval_relation_table": (c_int, [_M, c_void_p, c_void_p]),
    "kge_eval_relation_count_ranks": (c_int, [_M, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                              c_int64, c_void_p, c_void_p, c_void_p]),
    "kge_eval_relation_topk_scratch_bytes": (c_int64, [_M, c_int64, c_int64, c_int64, c_int]),
    "kge_eval_relation_topk": (c_int, [_M, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int,
                                       c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "kge_eval_relation_filter_bits": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64,
                                              c_void_p, c_void_p]),
    "kge_sample_negatives":(c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, ctypes.c_uint64,
                                     ctypes.c_uint64, c_void_p, c_void_p]),
    "kge_eval_filter_bits": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "kge_eval_filter_index_scratch_bytes": (c_int64, [c_int64, c_int64]),
    "kge_eval_filter_index_build": (c_int, [c_void_p, c_int64, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                                            c_int64, c_void_p, c_void_p]),
    "kge_eval_filter_bits_lookup_dense": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int64, c_int64,
                                                  c_void_p, c_void_p]),
    "kge_peer_alloc": (c_int, [c_int, c_int64, POINTER(c_void_p)]),
    "kge_peer_free": (c_int, [c_void_p]),
    "kge_peer_export": (c_int, [c_void_p, c_void_p]),
    "kge_peer_open": (c_int, [c_int, c_void_p, POINTER(c_void_p)]),
    "kge_peer_close": (c_int, [c_void_p]),
    "kge_peer_reduce_adam": (c_int, [POINTER(KgePeerGroup), ctypes.c_uint32, POINTER(KgeAdamTensor), c_int, c_int64,
                                     c_int64, c_int64, c_int64, c_int64, c_int64, c_int64, c_void_p, c_double, c_double,
                                     c_double, c_double, c_double, c_void_p, c_void_p]),
    "kge_train_gather_bytes": (c_int64, [_M, c_int, c_int64, c_int64]),
    "kge_train_shard_workspace_bytes": (c_int64, [_M, c_int, c_int64, c_int64]),
    "kge_train_rows_sharded": (c_int, [_M, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                       c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, POINTER(KgeShard),
                                       c_void_p, c_void_p, c_void_p]),
    "kge_train_entity_sharded": (c_int, [_M, c_int, c_int64, POINTER(KgeShard), c_void_p, c_int64,
                                         POINTER(KgeEntityAdam), c_void_p, c_void_p]),
    "kge_peer_barrier": (c_int, [POINTER(KgePeerGroup), c_int, ctypes.c_uint32, c_int, c_int, c_void_p, c_void_p]),
    "kge_l3_partials": (c_int, [POINTER(KgeAdamTensor), c_int, c_void_p, c_int64, c_void_p]),
    "kge_eval_filter_bits_lookup": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int64,
                                            c_int64, c_void_p, c_void_p]),
}

_lib = None


class KgeError(RuntimeError):
    pass


def load():
    """dlopen libkge_b200.so (built in-tree by build.py / __graft_entry__.build()) and type its symbols."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise KgeError(f"{LIB_PATH} is missing: run `python __graft_entry__.py` (or knowledgegraphembedding_b200/build.py)"
                       " to compile the sm_100a kernels; this package has no CPU or eager-PyTorch fallback")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype, fn.argtypes = res, args
    if lib.kge_abi_version() != 2:
        raise KgeError("libkge_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc):
    """Map a C-ABI return code to the exception the reference would raise at the same place."""
    if rc == 0:
        return
    msg = load().kge_last_error().decode("utf-8", "replace")
    if rc == ERR_INVALID:
        raise ValueError(msg)
    raise KgeError(msg)


def call(name, *args):
    check(getattr(load(), name)(*args))


_checked_devices = set()


def require_device(index):
    """Loud failure on anything that is not a B200-class (sm_100) GPU."""
    if index in _checked_devices:
        return
    sm, l2 = c_int(0), c_int64(0)
    check(load().kge_device_check(int(index), ctypes.byref(sm), ctypes.byref(l2)))
    _checked_devices.add(index)
