"""ctypes binding of libbrk_b200.so (the C ABI declared in include/brk_b200.h).

PyTorch is only the plumbing here: it owns device memory and streams; every compute call goes
through the C ABI with raw device pointers.  There is no CPU fallback: if the library is missing,
or no sm_100 device is present, the calls raise.
"""
import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbrk_b200.so")


class BrkError(RuntimeError):
    pass


class brk_table(C.Structure):
    _fields_ = [("w", C.c_void_p), ("g", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p),
                ("touched", C.c_void_p), ("rows", C.c_int64), ("d", C.c_int32), ("_pad", C.c_int32)]


class brk_adam_hyper(C.Structure):
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float)]


class brk_neumf_model(C.Structure):
    _fields_ = [("uMLP", brk_table), ("iMLP", brk_table), ("uMF", brk_table), ("iMF", brk_table),
                ("dense", brk_table), ("bn_moving", C.c_void_p), ("E", C.c_int32), ("H1", C.c_int32),
                ("H2", C.c_int32), ("H3", C.c_int32), ("act", C.c_int32), ("loss", C.c_int32),
                ("dropout", C.c_int32), ("tensor_cores", C.c_int32),
                # ABI 2: He et al. variant (all zero = the reference class graph)
                ("EMF", C.c_int32), ("mf_mode", C.c_int32), ("no_batch_norm", C.c_int32), ("_pad", C.c_int32)]


class brk_neumf_workspace(C.Structure):
    _fields_ = [("h1", C.c_void_p), ("h2", C.c_void_p), ("dy1", C.c_void_p), ("dy2", C.c_void_p),
                ("acc", C.c_void_p)]


BRK_MAX_PEERS = 8


class brk_shards(C.Structure):
    _fields_ = [("w", C.c_void_p * BRK_MAX_PEERS), ("g", C.c_void_p * BRK_MAX_PEERS),
                ("touched", C.c_void_p * BRK_MAX_PEERS), ("world", C.c_int32), ("rank", C.c_int32)]


class brk_neumf_shards(C.Structure):
    _fields_ = [("uMLP", brk_shards), ("iMLP", brk_shards), ("uMF", brk_shards), ("iMF", brk_shards)]


class brk_dp_peer(C.Structure):
    _fields_ = [("peer_w", C.c_void_p), ("peer_g", C.c_void_p), ("peer_flags", C.c_void_p), ("m", C.c_void_p),
                ("v", C.c_void_p), ("local_sync", C.c_void_p), ("n", C.c_int64), ("rank", C.c_int32),
                ("world", C.c_int32)]


class brk_tower(C.Structure):
    _fields_ = [("emb", brk_table), ("dense", brk_table), ("E", C.c_int32), ("S", C.c_int32)]


class brk_twotower_workspace(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("eu", "ei", "q", "c", "dq", "dc", "scores", "ones", "acc", "deu", "dei")]


class brk_tt_retrieval(C.Structure):
    _fields_ = [("cand_prob", C.c_void_p), ("row_weight", C.c_void_p), ("last", C.c_void_p), ("gap", C.c_void_p),
                ("step", C.c_void_p), ("rows", C.c_int64), ("inv_temperature", C.c_float), ("alpha", C.c_float)]


class brk_twotower_shards(C.Structure):
    _fields_ = [("user", brk_shards), ("item", brk_shards)]


class brk_tt_estimator_sharded(C.Structure):
    _fields_ = [("last", C.c_void_p * BRK_MAX_PEERS), ("gap", C.c_void_p * BRK_MAX_PEERS), ("rows", C.c_int64),
                ("world", C.c_int32), ("rank", C.c_int32)]


class brk_tt_retrieval_sharded(C.Structure):
    _fields_ = [("cand_prob", C.c_void_p), ("row_weight", C.c_void_p), ("est", C.POINTER(brk_tt_estimator_sharded)),
                ("inv_temperature", C.c_float)]


class brk_tt_sampled(C.Structure):
    _fields_ = [("ids", C.c_void_p), ("step", C.c_void_p), ("count", C.c_int64), ("lo", C.c_int64), ("hi", C.c_int64),
                ("rows", C.c_int64), ("seed", C.c_uint32), ("replica", C.c_uint32)]


class brk_twotower_global(C.Structure):
    _fields_ = [("cand", C.c_void_p * BRK_MAX_PEERS), ("ids", C.c_void_p * BRK_MAX_PEERS),
                ("slot", C.c_void_p * BRK_MAX_PEERS), ("offset", C.c_int64 * BRK_MAX_PEERS),
                ("count", C.c_int64 * BRK_MAX_PEERS), ("cap", C.c_int64), ("n_cap", C.c_int64), ("c_all", C.c_void_p),
                ("ids_all", C.c_void_p), ("err", C.c_void_p), ("world", C.c_int32), ("rank", C.c_int32)]


_P, _I32, _I64, _U32, _F32, _F64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_float, C.c_double

# name -> (restype, argtypes); mirrors include/brk_b200.h one to one.
SIGNATURES = {
    "brk_abi_version": (C.c_int, []),
    "brk_last_error": (C.c_char_p, []),
    "brk_create": (C.c_int, [C.POINTER(_P), C.c_int]),
    "brk_destroy": (C.c_int, [_P]),
    "brk_sm_count": (C.c_int, [_P]),
    "brk_gather_rows": (C.c_int, [_P, _P, _I64, _I32, _P, _I64, _P, _P]),
    "brk_scatter_add_rows": (C.c_int, [_P, _P, _I64, _I32, _P, _I64, _P, _P, _I32, _P]),
    "brk_philox_bpr_negatives": (C.c_int, [_P, _P, _I64, _I64, _U32, _U32, _I32, _P, _P, _P, _P]),
    "brk_philox_neumf_negatives": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _U32, _U32, _P, _P, _P]),
    "brk_philox4x32_10": (C.c_int, [_P, _P, _I64, _U32, _U32, _P, _P]),
    "brk_bpr_fwd_bwd": (C.c_int, [_P, C.POINTER(brk_table), C.POINTER(brk_table), _P, _P, _P, _I64, _I64, _P, _P]),
    "brk_bpr_train_steps": (C.c_int, [_P, C.POINTER(brk_table), C.POINTER(brk_table), _P, _P, _P, _I64, _I64,
                                      C.POINTER(C.c_int64), _I32, brk_adam_hyper, _I32, _P, _P, _P]),
    "brk_bpr_train_steps_host": (C.c_int, [_P, C.POINTER(brk_table), C.POINTER(brk_table), _P, _P, _I64, _I64, _I64,
                                           C.POINTER(C.c_int64), _I32, _U32, _U32, _I32, _P, _P, brk_adam_hyper, _I32,
                                           _P, _P, _P, _P, _P, _P]),
    "brk_bpr_host_stage_ints": (C.c_int64, [_I64]),
    "brk_bpr_train_steps_mapped": (C.c_int, [_P, C.POINTER(brk_table), C.POINTER(brk_table), _P, _P, _I64, _I64,
                                             C.POINTER(C.c_int64), _I32, _U32, _U32, _I32, _P, _P, brk_adam_hyper,
                                             _P, _P, _P]),
    "brk_bpr_scores": (C.c_int, [_P, _P, _P, _I32, _P, _P, _P, _I64, _P, _P]),
    "brk_adam_dense_keras": (C.c_int, [_P, C.POINTER(brk_table), _I32, brk_adam_hyper, _P, _I32, _P]),
    "brk_adam_rows": (C.c_int, [_P, C.POINTER(brk_table), _I32, brk_adam_hyper, _P, _I32, _P]),
    "brk_adagrad_rows": (C.c_int, [_P, C.POINTER(brk_table), _I32, _F32, _F32, _P]),
    "brk_adagrad_dense": (C.c_int, [_P, C.POINTER(brk_table), _I32, _F32, _F32, _P]),
    "brk_neumf_dense_floats": (C.c_int64, [_I32, _I32, _I32, _I32]),
    "brk_neumf_dense_floats_ex": (C.c_int64, [_I32, _I32, _I32, _I32, _I32]),
    "brk_neumf_acc_doubles": (C.c_int64, [_I32, _I32]),
    "brk_neumf_step": (C.c_int, [_P, C.POINTER(brk_neumf_model), _P, _P, _P, _I64, _I64, _I64, _I32, _U32, _U32,
                                 C.POINTER(brk_neumf_workspace), _P, _P, _P]),
    "brk_neumf_train_step": (C.c_int, [_P, C.POINTER(brk_neumf_model), _P, _P, _P, _I64, _I64, _U32, _U32, brk_adam_hyper, _P,
                                       _I32, C.POINTER(brk_neumf_workspace), _P, _P, _P]),
    "brk_neumf_host_stage_ints": (C.c_int64, [_I64]),
    "brk_neumf_train_steps_host": (C.c_int, [_P, C.POINTER(brk_neumf_model), _P, _I64, _I64, C.POINTER(C.c_int64), _I32, _U32,
                                             _U32, brk_adam_hyper, _P, _I32, C.POINTER(brk_neumf_workspace), _P, _P, _P, _P, _P]),
    "brk_neumf_train_steps": (C.c_int, [_P, C.POINTER(brk_neumf_model), _P, _P, _P, _I64, _I64, C.POINTER(C.c_int64), _I32,
                                        _U32, _U32, brk_adam_hyper, _P, _I32, C.POINTER(brk_neumf_workspace), _P, _P, _P]),
    "brk_neumf_step_sharded": (C.c_int, [_P, C.POINTER(brk_neumf_model), C.POINTER(brk_neumf_shards), _P, _P, _P, _I64,
                                         _I64, _I64, _I32, _U32, _U32, C.POINTER(brk_neumf_workspace), _P, _P, _P]),
    "brk_bpr_fwd_bwd_sharded": (C.c_int, [_P, C.POINTER(brk_shards), C.POINTER(brk_shards), _I32, _P, _P, _P, _I64, _I64, _P, _P]),
    "brk_peer_barrier": (C.c_int, [_P, _P, _P, _I32, _I32, _P]),
    "brk_allreduce_dense_peer": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _I32, _P]),
    "brk_gather_rows_sharded": (C.c_int, [_P, C.POINTER(brk_shards), _I32, _P, _I64, _P, _P]),
    "brk_scatter_add_rows_sharded": (C.c_int, [_P, C.POINTER(brk_shards), _I32, _P, _I64, _P, _P]),
    "brk_tc_selftest": (C.c_int, [_P, _I32, _I32, _I32, _I32, _P, _I32, _I32, _P, _I32, _I32, _P, _P]),
    "brk_dp_adam_peer": (C.c_int, [_P, C.POINTER(brk_dp_peer), brk_adam_hyper, _P, _P]),
    "brk_bpr_train_steps_dp": (C.c_int, [_P, C.POINTER(brk_table), C.POINTER(brk_table), _P, _P, _P, _I64, _I64,
                                         C.POINTER(C.c_int64), _I32, brk_adam_hyper, C.POINTER(brk_dp_peer), _P, _P, _P]),
    "brk_sgemm": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _F32, _I32, _P]),
    "brk_gemm_tf32": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _F32, _I32, _P]),
    "brk_gemm_tf32_trace": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _F32, _I32, _P, _P]),
    "brk_tower_forward": (C.c_int, [_P, C.POINTER(brk_tower), _P, _I64, _P, _P, _P]),
    "brk_twotower_step": (C.c_int, [_P, C.POINTER(brk_tower), C.POINTER(brk_tower), _P, _P, _P, _P, _I64, _I32, _I32,
                                    C.POINTER(brk_twotower_workspace), _P, _P]),
    "brk_twotower_train_step": (C.c_int, [_P, C.POINTER(brk_tower), C.POINTER(brk_tower), _P, _P, _P, _P, _I64, _I32,
                                          C.POINTER(brk_twotower_workspace), _F32, _F32, _I64, _P, _P]),
    "brk_twotower_step_retrieval": (C.c_int, [_P, C.POINTER(brk_tower), C.POINTER(brk_tower), _P, _P, _P, _P, _I64, _I32,
                                              _I32, C.POINTER(brk_twotower_workspace), _P, _P, C.POINTER(brk_tt_retrieval)]),
    "brk_twotower_train_step_retrieval": (C.c_int, [_P, C.POINTER(brk_tower), C.POINTER(brk_tower), _P, _P, _P, _P, _I64, _I32,
                                                    C.POINTER(brk_twotower_workspace), _F32, _F32, _I64, _P, _P,
                                                    C.POINTER(brk_tt_retrieval)]),
    "brk_twotower_step_sharded": (C.c_int, [_P, C.POINTER(brk_tower), C.POINTER(brk_tower), C.POINTER(brk_twotower_shards), _P,
                                            _P, _P, _P, _I64, _I32, C.POINTER(brk_twotower_workspace), _P, _P]),
    "brk_tower_forward_sharded": (C.c_int, [_P, C.POINTER(brk_tower), C.POINTER(brk_shards), _P, _I64, _P, _P, _P]),
    "brk_tt_estimator_update_sharded": (C.c_int, [_P, C.POINTER(brk_tt_estimator_sharded), _P, _I64, _F32, _P, _P]),
    "brk_twotower_step_sharded_retrieval": (C.c_int, [_P, C.POINTER(brk_tower), C.POINTER(brk_tower),
                                                      C.POINTER(brk_twotower_shards), _P, _P, _P, _P, _I64, _I32,
                                                      C.POINTER(brk_twotower_workspace), _P, _P,
                                                      C.POINTER(brk_tt_retrieval_sharded)]),
    "brk_twotower_step_sampled": (C.c_int, [_P, C.POINTER(brk_tower), C.POINTER(brk_tower), _P, _P, _I64, _I32,
                                            C.POINTER(brk_twotower_workspace), _P, _P, C.POINTER(brk_tt_sampled),
                                            C.POINTER(brk_tt_retrieval)]),
    "brk_twotower_train_step_sampled": (C.c_int, [_P, C.POINTER(brk_tower), C.POINTER(brk_tower), _P, _P, _I64, _I32,
                                                  C.POINTER(brk_twotower_workspace), _F32, _F32, _I64, _P, _P,
                                                  C.POINTER(brk_tt_sampled), C.POINTER(brk_tt_retrieval)]),
    "brk_twotower_step_sharded_sampled": (C.c_int, [_P, C.POINTER(brk_tower), C.POINTER(brk_tower),
                                                    C.POINTER(brk_twotower_shards), _P, _P, _I64, _I32,
                                                    C.POINTER(brk_twotower_workspace), _P, _P, C.POINTER(brk_tt_sampled),
                                                    C.POINTER(brk_tt_retrieval_sharded)]),
    "brk_twotower_step_global": (C.c_int, [_P, _I32, C.POINTER(brk_tower), C.POINTER(brk_tower), C.POINTER(brk_twotower_shards),
                                           C.POINTER(brk_twotower_global), _P, _P, _I32, C.POINTER(brk_twotower_workspace), _P,
                                           _P]),
    "brk_bf16_padded_dim": (C.c_int32, [_I32]),
    "brk_rows_to_bf16": (C.c_int, [_P, _P, _I64, _I32, _P, _I32, _P]),
    "brk_score_topk_workspace_bytes": (C.c_int64, [_P, _I64, _I64, _I32]),
    "brk_score_topk_bf16": (C.c_int, [_P, _P, _I64, _P, _I64, _I32, _I32, _I32, _P, _P, _P, _I64, _P]),
    "brk_score_topk_bf16_excl": (C.c_int, [_P, _P, _I64, _P, _I64, _I32, _I32, _I32, _P, _P, _P, _P, _P, _I64, _P]),
    "brk_mask_excluded": (C.c_int, [_P, _P, _I64, _I64, _I32, _P, _P, _P]),
    "brk_topk_metrics": (C.c_int, [_P, _P, _I64, _I32, _P, _P, _P, _I64, _P, _P, _P]),
    "brk_rank_eval_rows": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _P, _I32, _P, _P, _P, _P]),
    "brk_topk_rows": (C.c_int, [_P, _P, _I64, _I64, _I32, _P, _P, _P]),
    "brk_topk_merge": (C.c_int, [_P, _P, _P, _I32, _I64, _I32, _P, _P, _P]),
    "brk_topk_merge_peer": (C.c_int, [_P, _P, _P, _P, _I32, _I64, _I32, _P, _P, _P, _P]),
    "brk_neumf_topk_workspace_bytes": (C.c_int64, [_P, _I64, _I64, _I32]),
    "brk_neumf_score_topk": (C.c_int, [_P, C.POINTER(brk_neumf_model), _P, _P, _I64, _P, _P, _I64, _I32, _I32, _P, _P, _P,
                                       _I64, _P]),
    "brk_neumf_score_topk_excl": (C.c_int, [_P, C.POINTER(brk_neumf_model), _P, _P, _I64, _P, _P, _I64, _I32, _I32, _P, _P,
                                            _P, _P, _P, _I64, _P]),
    "brk_neumf_topk_fp32_workspace_bytes": (C.c_int64, [_P, C.POINTER(brk_neumf_model), _I64, _I64, _I32]),
    "brk_neumf_score_topk_fp32": (C.c_int, [_P, C.POINTER(brk_neumf_model), _P, _P, _I64, _P, _P, _I64, _I32, _I32, _P, _P,
                                            _P, _I64, _P]),
    "brk_neumf_score_topk_fp32_excl": (C.c_int, [_P, C.POINTER(brk_neumf_model), _P, _P, _I64, _P, _P, _I64, _I32, _I32,
                                                 _P, _P, _P, _P, _P, _I64, _P]),
    "brk_epoch_permutation":(C.c_int, [_P, _I64, _I64, _I64, _U32, _U32, _U32, _P, _P]),
    "brk_epoch_permutation_host": (C.c_int, [_I64, _I64, _I64, _U32, _U32, _U32, _P]),
    "brk_neumf_epoch_build": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _I64, _U32, _U32, _I32, _P, _P, _P, _P, _P, _P]),
    "brk_vocab_capacity": (C.c_int64, [_I64]),
    "brk_vocab_workspace_bytes": (C.c_int64, [_I64]),
    "brk_vocab_build_u64": (C.c_int, [_P, _P, _I64, _I32, _P, _P, _I64, _P, _P, _P, _P, _P]),
    "brk_vocab_lookup_u64": (C.c_int, [_P, _P, _I64, _P, _P, _I64, _I32, _P, _P]),
    "brk_svd_schedule_workspace_bytes": (C.c_int64, [_I64, _I64, _I64]),
    "brk_svd_schedule": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _P, _P, _P, _I64, _P]),
    "brk_svd_fit_epoch": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _P, _I64, _I64, _I32, _F64, _F64, _F64, _F64, _P,
                                    _I64, _I32, _P]),
    "brk_svd_fit_workspace_bytes": (C.c_int64, [_I64, _I64, _I32]),
    "brk_svd_predict": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _P, _I32, _F64, _P, _P]),
    "brk_svd_reduce_workspace_bytes": (C.c_int64, [_P]),
    "brk_svd_errors": (C.c_int, [_P, _P, _P, _P, _I64, _P, _P, _P, _P, _I32, _F64, _P, _P, _P]),
    "brk_svd_mean": (C.c_int, [_P, _P, _I64, _P, _P, _P]),
    "brk_svd_quintile_ratings": (C.c_int, [_P, _P, _P, _I64, _F64, _F64, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                           _P, _P]),
    "brk_svd_recommend": (C.c_int, [_P, _P, _P, _I32, _P, _I64, _I32, _I32, _P, _P, _P, _P]),
}

_lib = None
_lock = threading.Lock()
_ctx = {}


def lib():
    """Loads the shared library (no GPU needed for this step)."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise BrkError(
                        f"{LIB_PATH} is missing: build it with binary-recommendation_b200/csrc/build.sh "
                        "(or __graft_entry__.build()); there is no CPU fallback")
                l = C.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(l, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = l
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().brk_last_error().decode(errors="replace")
        raise BrkError(f"{what} failed (rc={rc}): {msg}")


def ctx(device=None):
    """Per-device library context (created on first use)."""
    if not torch.cuda.is_available():
        raise BrkError("no CUDA device: the brk_b200 hot path is sm_100a CUDA only (no CPU fallback)")
    dev = torch.cuda.current_device() if device is None else torch.device(device).index
    if dev is None:
        dev = torch.cuda.current_device()
    h = _ctx.get(dev)
    if h is None:
        with _lock:
            h = _ctx.get(dev)
            if h is None:
                torch.cuda.init()
                out = _P()
                check(lib().brk_create(C.byref(out), dev), "brk_create")
                h = out
                _ctx[dev] = h
                from . import _torchext
                _torchext.share_ctx(dev, h.value)            # the torch-extension ops use the same context
    return h


def stream_ptr():
    return _P(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (or None)."""
    if t is None:
        return _P(0)
    if not t.is_cuda:
        raise BrkError("expected a CUDA tensor")
    if not t.is_contiguous():
        raise BrkError("expected a contiguous tensor")
    return _P(t.data_ptr())
