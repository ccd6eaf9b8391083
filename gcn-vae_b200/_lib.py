"""ctypes binding of libkgvae_b200.so (the C ABI declared in include/kgvae_b200.h).

There is no CPU fallback: every op raises if the library is missing or the tensors are not
CUDA tensors.
"""
import ctypes
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libkgvae_b200.so")

_P, _I, _F, _L, _Z = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_longlong, ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/kgvae_b200.h one to one
_SIGNATURES = {
    "kg_last_error": (ctypes.c_char_p, []),
    "kg_version": (_I, []),
    "kg_device_info": (_I, [_P, _P, _P]),
    "kg_peer_alloc": (_I, [_Z, _P, _P]),
    "kg_peer_open": (_I, [_P, _P]),
    "kg_peer_close": (_I, [_P]),
    "kg_peer_free": (_I, [_P]),
    "kg_graph_build_workspace_bytes": (_Z, [_I]),
    "kg_graph_build": (_I, [_P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "kg_sample_relabel_workspace_bytes": (_Z, [_I]),
    "kg_sample_relabel": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "kg_neighbor_sample_plan": (_I, [_I, _I, _I, _P, _P]),
    "kg_neighbor_sample": (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "kg_graph_index_workspace_bytes": (_Z, [_I]),
    "kg_graph_index": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "kg_embedding_fwd": (_I, [_P, _P, _I, _I, _P, _P]),
    "kg_embedding_bwd": (_I, [_P, _P, _I, _I, _P, _P]),
    "kg_bdd_weight_layouts": (_I, [_P, _I, _I, _I, _I, _P, _P, _P]),
    "kg_bdd_rel_fwd": (_I, [_P, _P, _I, _P, _I, _P, _P, _I, _I, _I, _P, _I, _P]),
    "kg_bdd_rel_bwd": (_I, [_P, _P, _I, _P, _P, _I, _P, _P, _I, _I, _I, _P, _P, _I, _P]),
    "kg_bdd_rel_fwd_cols": (_I, [_P, _P, _I, _P, _I, _I, _I, _I, _I, _P, _I, _P]),
    "kg_bdd_rel_bwd_cols": (_I, [_P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P]),
    "kg_bdd_layouts_needed": (_I, [_I, _I, _I]),
    "kg_graph_rel_tiled_workspace_bytes": (_Z, [_I]),
    "kg_graph_rel_tiled": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _Z, _P]),
    "kg_basis_id_fwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P]),
    "kg_basis_id_bwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "kg_basis_id_src_eligible": (_I, [_I, _I, _I]),
    "kg_basis_id_src_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P, _P]),
    "kg_basis_id_src_bwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "kg_basis_dense_fwd": (_I, [_P, _P, _I, _P, _I, _I, _I, _P, _P]),
    "kg_basis_dense_bwd": (_I, [_P, _P, _P, _I, _P, _I, _I, _I, _P, _P, _P]),
    "kg_act_dropout_bwd": (_I, [_P, _P, _P, _I, _L, _P, _P]),
    "kg_act_dropout_bwd_colsum": (_I, [_P, _P, _P, _I, _I, _I, _P, _P, _P, _Z, _P]),
    "kg_colsum_workspace_bytes": (_Z, [_I, _I]),
    "kg_colsum": (_I, [_P, _I, _I, _P, _P, _Z, _P]),
    "kg_gemm_f32_workspace_bytes": (_Z, [_I, _I, _I]),
    "kg_gemm_f32": (_I, [_P, _I, _I, _P, _I, _I, _P, _I, _I, _I, _I, _P, _P, _I, _P, _I, _P, _Z, _P]),
    "kg_gemm_f32_uses_tensor_cores": (_I, [_I, _I, _I]),
    "kg_gemm_prep_bytes": (_Z, [_I, _I]),
    "kg_gemm_prepare": (_I, [_P, _I, _I, _I, _P, _Z, _P]),
    "kg_gemm_f32_prepared_workspace_bytes": (_Z, [_I, _I, _I]),
    "kg_gemm_f32_prepared": (_I, [_P, _I, _P, _I, _P, _I, _I, _I, _I, _P, _P, _I, _P, _I, _P, _Z, _P]),
    "kg_reparam_fwd": (_I, [_P, _P, _I, _I, _P, _P, _P, _P]),
    "kg_reparam_bwd": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _P, _P]),
    "kg_kl_mog_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P]),
    "kg_kl_mog_bwd": (_I, [_P, _P, _P, _P, _P, _P, _F, _I, _I, _I, _P, _P, _P, _P, _P]),
    "kg_kl_mog_bwd_fused": (_I, [_P, _P, _P, _P, _P, _P, _F, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "kg_kl_mog_fwd_rows": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P]),
    "kg_kl_mog_bwd_fused_rows": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "kg_iaf_update_fwd": (_I, [_P, _P, _P, _P, _I, _I, _P, _P, _P]),
    "kg_iaf_update_bwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P]),
    "kg_reverse_columns": (_I, [_P, _I, _I, _P, _P]),
    "kg_distmult_score": (_I, [_P, _P, _P, _I, _I, _P, _P, _P]),
    "kg_reduce_workspace_bytes": (_Z, [_L]),
    "kg_bce_logits_fwd": (_I, [_P, _P, _I, _P, _P, _P, _Z, _P]),
    "kg_sum_squares": (_I, [_P, _L, _P, _P, _Z, _P]),
    "kg_sum": (_I, [_P, _L, _P, _P, _Z, _P]),
    "kg_sum_squares_rows": (_I, [_P, _I, _I, _P, _P, _P, _Z, _P]),
    "kg_triplet_index_workspace_bytes": (_Z, [_I]),
    "kg_triplet_index": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "kg_distmult_bce_workspace_bytes": (_Z, [_I]),
    "kg_distmult_bce_fwd": (_I, [_P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "kg_distmult_bwd_dz": (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _P]),
    "kg_triplet_index_trailing": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "kg_distmult_bce_fwd_lead": (_I, [_P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "kg_distmult_bwd_dz_trailing": (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _P]),
    "kg_distmult_bwd_dw": (_I, [_P, _P, _P, _I, _I, _P, _P]),
    "kg_distmult_rank_workspace_bytes": (_Z, [_I, _I, _I]),
    "kg_distmult_rank": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _I, _I, _P, _P, _P, _Z, _P, _P, _P]),
    "kg_probe_l2": (_I, [_P, _P, _I, _I, _L, _I, _P, _P]),
    "kg_set_tc_terms": (_I, [_I]),
    "kg_distmult_topk_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "kg_distmult_topk": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _I, _P, _Z, _P, _P, _P]),
    "kg_distmult_topk_filtered": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _I, _P, _P, _P, _Z, _P, _P, _P]),
    "kg_distmult_topk_shard": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _I, _I, _I, _P, _P, _P, _Z, _P, _P, _P]),
    "kg_filter_table_workspace_bytes": (_Z, [_I]),
    "kg_filter_table": (_I, [_P, _I, _I, _I, _I, _P, _P, _P, _Z, _P]),
    "kg_filter_count_workspace_bytes": (_Z, [_I]),
    "kg_filter_count": (_I, [_P, _P, _I, _I, _P, _P, _I, _P, _P, _P, _Z, _P]),
    "kg_filter_gather": (_I, [_P, _P, _I, _I, _P, _P, _I, _P, _P, _P]),
}

_lib = None


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"kgvae_b200: {LIB_PATH} is missing - build it with "
                "`python -c 'import __graft_entry__ as g; g.build()'` (there is no CPU fallback)")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


# kernels launched per entry point (bench.py's gpu_launches; CUB sorts/scans counted as 2 each)
KERNELS_PER_CALL = {
    "kg_graph_build": 14, "kg_graph_index": 10, "kg_graph_rel_tiled": 5, "kg_triplet_index": 13, "kg_triplet_index_trailing": 18, "kg_distmult_bce_fwd": 5, "kg_distmult_bce_fwd_lead": 5, "kg_colsum": 2, "kg_act_dropout_bwd_colsum": 1,
    "kg_gemm_f32": 5,        # two operand preparations (2 kernels each) + the product (+ split-K finish): a lower bound
    "kg_gemm_prepare": 2,
    "kg_sample_relabel": 7, "kg_kl_mog_fwd_rows": 2, "kg_sum_squares_rows": 2,
    "kg_neighbor_sample_plan": 0, "kg_neighbor_sample": 1,
    "kg_kl_mog_fwd": 2, "kg_bce_logits_fwd": 2, "kg_sum_squares": 2, "kg_sum": 2, "kg_distmult_rank": 3, "kg_distmult_topk": 5,
    "kg_distmult_topk_filtered": 5, "kg_distmult_topk_shard": 5, "kg_filter_table": 5, "kg_filter_count": 4,
}
launches = 0          # running count of kernels launched through this binding
profile = None        # when a dict: name -> [(start_event, end_event), ...] per call


_seen_dev = None      # device index of the tensors whose pointers were taken since the last call()


def call(name, *args, tag=None):
    """Invoke an int-returning entry point; raise RuntimeError with kg_last_error() on failure.  The kernels launch
    on the CURRENT device's stream: tensors that live on another device would be dereferenced in the wrong context,
    so the device of the pointers taken for this call (ptr()) is checked against it - one query per call."""
    global launches, _seen_dev
    handle = lib()
    if _seen_dev is not None:
        dev, _seen_dev = _seen_dev, None
        if dev != torch.cuda.current_device():
            raise RuntimeError(f"kgvae_b200: {name} was given tensors on cuda:{dev} while the current device is "
                               f"cuda:{torch.cuda.current_device()} (use torch.cuda.set_device / torch.cuda.device)")
    if profile is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    rc = getattr(handle, name)(*args)
    if rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {handle.kg_last_error().decode()}")
    launches += KERNELS_PER_CALL.get(name, 1)
    if profile is not None:
        ev1.record()
        profile.setdefault(tag or name, []).append((ev0, ev1))


def ptr(t, dtype=None):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("kgvae_b200 ops need CUDA tensors (no CPU fallback)")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"kgvae_b200: expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise RuntimeError("kgvae_b200: tensor must be contiguous")
    global _seen_dev
    idx = t.device.index
    if _seen_dev is not None and _seen_dev != idx:
        _seen_dev = None
        raise RuntimeError("kgvae_b200: the tensors of one call live on different devices")
    _seen_dev = idx
    return t.data_ptr()


def f32(t):
    return ptr(t, torch.float32)


def i32(t):
    return ptr(t, torch.int32)


def stream():
    return torch.cuda.current_stream().cuda_stream


def workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def device_info():
    a, b, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    call("kg_device_info", ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
    return {"sm_count": a.value, "cc": (b.value, c.value)}
