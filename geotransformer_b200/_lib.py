"""ctypes binding of the C-ABI library ``libgeob200.so`` (declared in ``include/geob200.h``).

The product path has NO fallback: if the library is missing or a call fails, a RuntimeError is raised
(the reference raises RuntimeError through TORCH_CHECK, ``extensions/common/torch_helper.h:6-35``).
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libgeob200.so')
_lib = None

c_void_p, c_int64, c_int32, c_float, c_size_t, c_int = (
    ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_float, ctypes.c_size_t, ctypes.c_int)

# name -> (restype, argtypes); kept in one table so tests can check it against include/geob200.h
SIGNATURES = {}


def _sig(name, restype, *argtypes):
    SIGNATURES[name] = (restype, list(argtypes))


P, I64, I32, F, SZ = c_void_p, c_int64, c_int32, c_float, c_size_t
_sig('geob200_last_error', ctypes.c_char_p)
_sig('geob200_launch_count', ctypes.c_uint64)
_sig('geob200_grid_subsample_workspace_bytes', SZ, I64, I64)
_sig('geob200_grid_subsample', c_int, P, I64, P, I64, F, P, P, P, SZ, P)
_sig('geob200_radius_search_workspace_bytes', SZ, I64, I64, I64)
_sig('geob200_radius_search', c_int, P, I64, P, I64, P, P, I64, F, I64, P, P, P, P, SZ, P)

_sig('geob200_neighbor_histogram', c_int, P, I64, I64, I64, I64, P, P)
_sig('geob200_kpconv_workspace_bytes', SZ, I64)
_sig('geob200_kpconv', c_int, P, P, P, P, I64, I64, I64, P, I64, P, P, I64, I64, F, P, P, SZ, P)
_sig('geob200_kpconv_tc_workspace_bytes', SZ, I64, I64, I64)
_sig('geob200_kpconv_tc', c_int, P, P, P, P, I64, I64, I64, P, I64, P, P, I64, I64, F, P, P, SZ, P)
_sig('geob200_set_linear_mode', None, c_int)
_sig('geob200_linear', c_int, P, I64, P, P, P, I64, I64, I64, I64, c_int, P)
_sig('geob200_linear_batched', c_int, P, I64, I64, P, I64, I64, P, I64, P, I64, I64, I64, I64, I64, I64, c_int, P)
_sig('geob200_group_norm_workspace_bytes', SZ, I64, I64, I64, I64)
_sig('geob200_group_norm', c_int, P, I64, I64, I64, P, P, F, P, c_int, F, P, P, SZ, P)
_sig('geob200_linear_group_norm', c_int, P, I64, P, P, I64, I64, I64, I64, P, P, F, P, c_int, F, P, P, P, SZ, P)
_sig('geob200_kpconv_group_norm', c_int, P, P, P, P, I64, I64, I64, P, I64, P, P, I64, I64, F, I64, P, P, F, c_int, F, P, P, P, SZ,
     P, SZ, P)
_sig('geob200_group_norm_batched', c_int, P, I64, I64, I64, P, P, F, P, c_int, F, P, P, SZ, P, I64, P)
_sig('geob200_linear_group_norm_batched', c_int, P, I64, P, P, I64, I64, I64, I64, P, P, F, P, c_int, F, P, P, P, SZ, P, I64, P)
_sig('geob200_maxpool', c_int, P, P, I64, I64, I64, I64, P, P)
_sig('geob200_upsample_concat', c_int, P, P, I64, I64, P, I64, I64, I64, P, P)
_sig('geob200_point_to_node_partition', c_int, P, I64, P, I64, I64, P, P, P, P, P, P, P)
_sig('geob200_gather_rows', c_int, P, I64, I64, P, I64, P, P)
_sig('geob200_knn_partition', c_int, P, I64, P, I64, I64, P, P, P)
_sig('geob200_pairwise_distance', c_int, P, I64, P, I64, I64, c_int, P, P)
_sig('geob200_point_to_node_indices', c_int, P, I64, P, I64, P, P, P)
_sig('geob200_apply_transform', c_int, P, I64, P, P, P)
_sig('geob200_gse_indices', c_int, P, I64, F, F, I64, P, P, P)
_sig('geob200_gse_indices_batched', c_int, P, I64, P, F, F, I64, P, P, P)
_sig('geob200_gse_embed_workspace_bytes', SZ, I64, I64)
_sig('geob200_gse_table_bytes', SZ, I64, I64, F, F)
_sig('geob200_gse_table_build', c_int, P, P, P, P, P, I64, I64, F, F, P, SZ, P)
_sig('geob200_gse_embed_table', c_int, P, P, I64, I64, P, SZ, I64, F, F, P, P, P, P, P, P, P)
_sig('geob200_gse_embed', c_int, P, P, I64, I64, P, P, P, P, P, P, P, P, c_int, P, SZ, P)
_sig('geob200_gse_embed_pairs', c_int, P, P, I64, I64, P, P, P, P, P, P, P, P, c_int, P, SZ, P)
_sig('geob200_attention_workspace_bytes', SZ, I64, I64, I64)
_sig('geob200_attention', c_int, P, I64, P, I64, P, I64, P, P, P, I64, I64, I64, I64, P, I64, P, SZ, P)
_sig('geob200_set_attention_tma', c_int, c_int)
_sig('geob200_head_bias', c_int, P, I64, P, I64, I64, I64, P, P)
_sig('geob200_add_layernorm', c_int, P, P, P, P, I64, I64, F, P, P)
_sig('geob200_l2_normalize', c_int, P, I64, I64, P, P)
_sig('geob200_superpoint_matching_workspace_bytes', SZ, I64, I64)
_sig('geob200_superpoint_matching', c_int, P, P, I64, I64, I64, P, P, I64, c_int, P, P, P, P, P, SZ, P)
_sig('geob200_gather_patches', c_int, P, I64, P, P, I64, P, I64, P, P, P, P)
_sig('geob200_patch_scores', c_int, P, I64, P, I64, I64, P, P, I64, I64, P, P)
_sig('geob200_sinkhorn', c_int, P, P, P, P, I64, I64, I64, F, P, P)
_sig('geob200_lgr_workspace_bytes', SZ, I64, I64, I64)
_sig('geob200_local_global_registration', c_int, P, P, P, P, P, I64, I64, I64, I64, F, c_int, F, I64, I64, P, P, P, P, P,
     P, P, P, P, P, SZ, P)
_sig('geob200_weighted_procrustes', c_int, P, P, P, I64, I64, F, F, P, P)

_sig('geob200_node_correspondences_workspace_bytes', SZ, I64, I64, I64)
_sig('geob200_node_correspondences', c_int, P, P, P, P, P, P, P, P, I64, I64, I64, P, F, P, P, P, P, SZ, P)
_sig('geob200_evaluate', c_int, P, P, I64, F, P, P, I64, P, P, I64, F, P, P, P, I64, c_int, F, F, F, P, P)
_sig('geob200_evaluate_counts', c_int, P, P, I64, P, F, P, P, I64, P, P, P, I64, P, F, P, P, P, I64, c_int, F, F, F, P, P)

_sig('geob200_linear_profile_enable', c_int, c_int)
_sig('geob200_set_split_k', c_int, c_int)
_sig('geob200_set_linear_persistent', c_int, c_int)
_sig('geob200_linear_profile_read', I64, I64, P, P)
_sig('geob200_backbone_workspace_bytes', SZ, P, P)
_sig('geob200_backbone_forward', c_int, P, P, P, P, P, P, P, P, P, P, P, P, SZ, P, SZ, P)
_sig('geob200_transformer_workspace_bytes', SZ, I64, I64, I64, I64, I64)
_sig('geob200_transformer_forward', c_int, P, I64, I64, I64, P, I64, I64, P, P, P, P, SZ, P)
_sig('geob200_backbone_gn_workspace_bytes', SZ, P, P, I64)
_sig('geob200_backbone_forward_batched', c_int, P, P, P, P, P, P, P, P, P, P, P, P, SZ, P, SZ, P, I64, P, P)
_sig('geob200_cloud_max_count', c_int, P, I64, I64, I64, I64, P, P, P)
_sig('geob200_maxpool_batched', c_int, P, P, I64, I64, I64, I64, P, I64, P, P, P)
_sig('geob200_transformer_batched_workspace_bytes', SZ, I64, P, I64, I64, I64)
_sig('geob200_transformer_forward_batched', c_int, P, I64, I64, I64, P, I64, P, P, P, P, SZ, P)
_sig('geob200_attention_batched_workspace_bytes', SZ, P, I64, I64)
_sig('geob200_attention_batched', c_int, P, I64, I64, I64, I64, I64, I64, I64, P, SZ, P)


def lib():
    """Load (once) and return the C-ABI library; raises RuntimeError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                '(there is no CPU fallback for the geotransformer_b200 ops)')
        handle = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().geob200_last_error().decode(errors='replace')
        raise RuntimeError(f'{what} failed ({rc}): {msg}')


_tls = threading.local()


def stream_ptr():
    """cudaStream_t of the current torch stream.  Inside a ``stream_scope`` the pointer is served from a thread-local
    (querying torch costs ~2 us, and every op of the forward asks for it)."""
    p = getattr(_tls, 'stream', None)
    if p is not None:
        return p
    return torch.cuda.current_stream().cuda_stream


class stream_scope:
    """``with torch.cuda.stream(s), stream_scope(s.cuda_stream): ...`` -- pins the stream pointer for this thread."""

    def __init__(self, ptr):
        self.ptr = ptr

    def __enter__(self):
        self.prev = getattr(_tls, 'stream', None)
        _tls.stream = self.ptr
        return self

    def __exit__(self, *a):
        _tls.stream = self.prev
        return False


def require_cuda(t, name, dtype=None):
    if not t.is_cuda:
        raise RuntimeError(f'{name} must be a CUDA tensor (geotransformer_b200 has no CPU path)')
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f'{name} must be {dtype}, got {t.dtype}')
    if not t.is_contiguous():
        raise RuntimeError(f'{name} must be contiguous')


_WS = {}


def workspace(nbytes, device, tag='default'):
    """Grow-only scratch buffer per (device, current stream, tag): ops on one stream reuse it serially, concurrent streams
    (RegistrationEngine runs several pairs at once) never share scratch."""
    key = (device.index if device.index is not None else torch.cuda.current_device(), stream_ptr(), tag)
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        # 30% headroom: pair sizes vary by a few percent and regrowing a large scratch means a cudaMalloc in the hot loop
        buf = torch.empty(max(int(nbytes * 1.3), 1 << 20), dtype=torch.uint8, device=device)
        _WS[key] = buf
    return buf


def ptr(t):
    return None if t is None else t.data_ptr()
