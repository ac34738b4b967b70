"""ctypes binding of libhals_b200.so (the C ABI declared in include/hals_b200.h).

The library is the product's only compute path.  There is no CPU or PyTorch fallback:
if the shared object is missing, or a compute entry point is called without a CUDA
device, this module raises.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HALS_LIB_PATH") or os.path.join(_HERE, "libhals_b200.so")   # env override: A/B builds
CSRC = os.path.join(_HERE, "csrc")

c_i32, c_i64, c_f32, c_vp, c_sz = ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t


class NativeError(RuntimeError):
    pass


class AlsPlan(ctypes.Structure):
    """struct hals_als_plan (include/hals_b200.h)."""
    _fields_ = [
        ("n_items", c_i64), ("n_long_rows", c_i64), ("n_slots", c_i64),
        ("seg_len", c_i32), ("max_nseg", c_i32),
        ("item_row", c_vp), ("item_begin", c_vp), ("item_len", c_vp), ("item_slot", c_vp),
        ("long_row", c_vp), ("long_slot0", c_vp), ("long_nseg", c_vp),
        ("n_long_gt16", c_i64), ("n_long_gt256", c_i64),
        ("n_chunks", c_i64), ("item_chunk0", c_vp), ("item_cost0", c_vp), ("chunk_pos", c_vp), ("chunk_cnt", c_vp),
        ("vals_hl", c_vp), ("vals_scale", c_vp), ("item_npos", c_vp), ("packed_alpha", c_f32),
    ]


class TowerWeights(ctypes.Structure):
    """struct hals_tower_weights (include/hals_b200.h)."""
    _fields_ = [
        ("embedding_size", c_i32), ("manu_dim", c_i32), ("cat_dim", c_i32), ("num_hidden", c_i32),
        ("user_emb", c_vp), ("item_emb", c_vp), ("manu_emb", c_vp), ("cat_emb", c_vp),
        ("num_w", c_vp), ("num_b", c_vp), ("out_w", c_vp), ("out_b", c_vp),
        ("user_ln_g", c_vp), ("user_ln_b", c_vp), ("item_ln_g", c_vp), ("item_ln_b", c_vp),
        ("ln_eps", c_f32), ("num_scale", c_f32 * 2), ("num_offset", c_f32 * 2),
        ("num_users", c_i32), ("num_items", c_i32), ("num_manufacturers", c_i32), ("num_categories", c_i32),
    ]


class TowerParams(ctypes.Structure):
    """struct hals_tower_params (include/hals_b200.h): the tower tensors the training step mutates."""
    _fields_ = [
        ("embedding_size", c_i32), ("manu_dim", c_i32), ("cat_dim", c_i32), ("num_hidden", c_i32),
        ("user_emb", c_vp), ("item_emb", c_vp), ("manu_emb", c_vp), ("cat_emb", c_vp),
        ("num_w", c_vp), ("num_b", c_vp), ("out_w", c_vp), ("out_b", c_vp),
        ("user_ln_g", c_vp), ("user_ln_b", c_vp), ("item_ln_g", c_vp), ("item_ln_b", c_vp),
        ("ln_eps", c_f32),
        ("num_users", c_i32), ("num_items", c_i32), ("num_manufacturers", c_i32), ("num_categories", c_i32),
    ]


class TowerBatch(ctypes.Structure):
    """struct hals_tower_batch (include/hals_b200.h)."""
    _fields_ = [
        ("n", c_i64), ("user_ids", c_vp), ("item_ids", c_vp), ("manufacturer_ids", c_vp), ("category_ids", c_vp),
        ("numeric", c_vp), ("labels", c_vp),
        ("order_user", c_vp), ("order_item", c_vp), ("order_manufacturer", c_vp), ("order_category", c_vp),
    ]


# name -> (restype, argtypes); kept in one table so tests can check it against the header
SIGNATURES = {
    "hals_abi_version": (ctypes.c_int, []),
    "hals_last_error": (ctypes.c_char_p, []),
    "hals_launch_count": (c_i64, []),
    "hals_max_rank": (ctypes.c_int, []),
    "hals_als_plan_count_host": (ctypes.c_int, [c_vp, c_i64, c_i32, c_vp, c_vp, c_vp]),
    "hals_als_plan_fill_host": (ctypes.c_int, [c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "hals_als_plan_chunk_count_host": (c_i64, [c_vp, c_i64]),
    "hals_als_plan_chunks_host": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, ctypes.c_int, c_vp, c_vp, c_vp, c_vp]),
    "hals_als_workspace_bytes": (c_sz, [c_i64, ctypes.c_int, c_i64]),
    "hals_als_default_seg_len": (c_i32, [ctypes.c_int]),
    "hals_als_pack_ratings": (ctypes.c_int, [c_vp, c_i64, c_vp, c_vp]),
    "hals_als_pack_ratings_implicit": (ctypes.c_int, [c_vp, c_i64, c_f32, c_vp, c_vp, c_vp]),
    "hals_als_plan_count_positive": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "hals_als_half_step": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, ctypes.c_int, c_f32,
                                          ctypes.c_int, c_f32, c_vp, ctypes.POINTER(AlsPlan), c_vp, c_sz, c_vp]),
    "hals_als_half_step_nonnegative": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, ctypes.c_int, c_f32,
                                                      ctypes.c_int, c_f32, c_vp, ctypes.POINTER(AlsPlan), c_vp, c_sz,
                                                      c_vp, c_vp]),
    "hals_als_split_factors": (ctypes.c_int, [c_vp, c_i64, ctypes.c_int, c_vp, c_vp]),
    "hals_als_half_step_split": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, ctypes.c_int, c_f32, ctypes.POINTER(AlsPlan), c_vp,
                                                  c_sz, c_vp]),
    "hals_gram_workspace_bytes": (c_sz, [ctypes.c_int]),
    "hals_gram": (ctypes.c_int, [c_vp, c_i64, ctypes.c_int, c_vp, c_vp, c_sz, c_vp]),
    "hals_als_predict": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "hals_als_sse_workspace_bytes": (c_sz, []),
    "hals_als_sse": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "hals_f1_at_k": (ctypes.c_int, [c_vp, c_i64, ctypes.c_int, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "hals_ranking_metrics": (ctypes.c_int, [c_vp, c_i64, ctypes.c_int, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "hals_similar_items": (ctypes.c_int, [c_vp, ctypes.c_int, c_vp, c_i64, c_vp, c_i64, ctypes.c_double, c_vp, c_vp, c_vp]),
    "hals_tower_user": (ctypes.c_int, [ctypes.POINTER(TowerWeights), c_vp, c_i64, c_vp, c_i64, c_vp]),
    "hals_tower_item": (ctypes.c_int, [ctypes.POINTER(TowerWeights), c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "hals_tower_train_workspace_bytes": (c_sz, [ctypes.POINTER(TowerParams), c_i64]),
    "hals_tower_train_step": (ctypes.c_int, [ctypes.POINTER(TowerParams), ctypes.POINTER(TowerBatch), c_i64, c_vp, c_sz,
                                             c_vp, c_vp]),
    "hals_tower_adam_step": (ctypes.c_int, [ctypes.POINTER(TowerParams), ctypes.POINTER(TowerParams),
                                            ctypes.POINTER(TowerParams), ctypes.POINTER(TowerBatch), c_i64, c_vp, c_sz,
                                            ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, c_vp]),
    "hals_score_extrema": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, ctypes.c_int, c_vp, c_i64, c_vp, c_i64,
                                          ctypes.c_int, c_i64, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "hals_score_workspace_bytes": (c_sz, [c_i64, c_i64, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "hals_score_flag_counter_offset": (c_i64, [c_i64, c_i64, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "hals_score_blend_topk": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, ctypes.c_int, c_vp, c_i64, c_vp, c_i64,
                                             ctypes.c_int, c_i64, c_i64, c_vp, c_f32, c_f32, ctypes.c_int, c_i32,
                                             c_vp, c_vp, c_vp, c_sz, c_vp]),
    "hals_score_blend_topk_excluding": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, ctypes.c_int, c_vp, c_i64, c_vp, c_i64,
                                                       ctypes.c_int, c_i64, c_i64, c_vp, c_f32, c_f32, ctypes.c_int, c_i32,
                                                       c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "hals_score_topk": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, ctypes.c_int, c_i64, c_i64, ctypes.c_int, c_i32, c_vp,
                                       c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "hals_score_lists_workspace_bytes": (c_sz, [c_i64, ctypes.c_int]),
    "hals_score_blend_topk_lists": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, ctypes.c_int, c_vp, c_i64, c_vp, c_i64,
                                                   ctypes.c_int, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_f32,
                                                   c_f32, ctypes.c_int, ctypes.c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "hals_topk_merge": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, c_i64, ctypes.c_int, c_vp, c_vp, c_vp]),
    "hals_score_one_user": (ctypes.c_int, [c_vp, c_vp, c_i64, ctypes.c_int, c_vp, c_i64, c_vp, c_vp]),
    "hals_fuse_lists": (ctypes.c_int, [c_vp, c_vp, c_i64, c_f32, c_f32, c_vp, c_vp, c_vp]),
    "hals_debug_umma_probe": (ctypes.c_int, [c_vp, ctypes.c_int] + [ctypes.c_uint32] * 8 +
                              [ctypes.c_int, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, ctypes.c_int, c_vp, c_vp]),
}

_lib = None


def build(force: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into libhals_b200.so (nvcc cross-compiles without a GPU)."""
    args = ["make", "-s", "-j8", "-C", CSRC]
    if force:
        args.append("-B")
    subprocess.check_call(args)
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C csrc`); there is no CPU fallback for this path")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)   # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if L.hals_abi_version() != 1:
            raise NativeError("libhals_b200.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().hals_last_error().decode(errors="replace")
        raise NativeError(f"{what or 'hals call'} failed (status {rc}): {msg}")


def launch_count() -> int:
    return int(lib().hals_launch_count())


def ptr(t):
    """Device (or host) pointer of a torch tensor / numpy array, None -> NULL."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return ctypes.c_void_p(t.data_ptr())
    return t.ctypes.data_as(ctypes.c_void_p)


def current_stream():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise NativeError("no CUDA device: the hals_b200 kernels have no CPU fallback")
