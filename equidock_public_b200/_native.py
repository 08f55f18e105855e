"""ctypes binding of ``libeqd_iegmn.so`` (the C ABI declared in ``include/eqd_iegmn.h``).

There is NO fallback: if the CUDA library is missing or a call fails, this raises.  The library is
built in-tree by ``equidock_public_b200/csrc/build.sh`` (``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# EQD_LIB_PATH: load another build of the same ABI instead (A/B runs of kernel variants, scripts/forward_ab.py)
LIB_PATH = os.environ.get('EQD_LIB_PATH') or os.path.join(_HERE, 'libeqd_iegmn.so')

ABI_VERSION = 9
EDGE_FEATS, N_RBF, HID, H0, H0_PAD, N_RES_TYPES, HEADS, TILE_ROWS = 27, 15, 64, 69, 72, 21, 50, 128
STATUS_SVD_DEGENERATE, STATUS_NAN, STATUS_DEGREE_OVERFLOW, STATUS_BAD_RESIDUE = 1, 2, 4, 8

_vp, _i32, _f32 = C.c_void_p, C.c_int32, C.c_float


class EqdGraph(C.Structure):
    _fields_ = [('n_pairs', _i32), ('n_nodes', _i32), ('n_lig_nodes', _i32), ('n_edges', _i32),
                ('n_lig_edges', _i32), ('max_in_degree', _i32),
                ('seg_ptr', _vp), ('row_ptr', _vp), ('col_src', _vp), ('edge_dst', _vp),
                ('he_lig', _vp), ('he_rec', _vp),
                ('n_node_tiles', _i32), ('node_tiles', _vp)]


class EqdLayerParams(C.Structure):
    _fields_ = [('dh', _i32), ('dhp', _i32),
                ('w_proj', _vp), ('b_proj', _vp), ('w_edge1', _vp), ('edge_ln_g', _vp), ('edge_ln_b', _vp),
                ('w_edge2', _vp), ('b_edge2', _vp), ('w_coor1', _vp), ('b_coor1', _vp), ('w_coor2', _vp),
                ('b_coor2', _f32), ('w_edge_tc', _vp), ('w_node_tc', _vp), ('w_proj_tc', _vp),
                ('w_node1', _vp), ('b_node1', _vp), ('node_ln_g', _vp), ('node_ln_b', _vp),
                ('w_node2', _vp), ('b_node2', _vp),
                ('skip_weight_h', _f32), ('x_connection_init', _f32), ('leaky_slope', _f32)]


class EqdLayerConsts(C.Structure):
    """eqd_layer_consts: launch-time constants of the tensor-core kernels, host VALUES (not pointers)."""
    _fields_ = [('edge', _f32 * 64 * 5), ('node', _f32 * 304), ('proj_bias', _f32 * 320)]


class EqdLayer(C.Structure):
    """eqd_layer: what the entry points take -- `dev` (device pointers + scalars, passed to kernels by value) + `consts`."""
    _fields_ = [('dev', EqdLayerParams), ('consts', EqdLayerConsts)]


class EqdForwardIO(C.Structure):
    _fields_ = [(n, _vp) for n in ('emb', 'res_lig', 'res_rec', 'mu_lig', 'mu_rec', 'x_lig', 'x_rec', 'rot', 'trans',
                                   'ligand_out', 'sing', 'status', 'h_out', 'x_out', 'keypts', 'cov', 'ymean', 'stage_events')] + \
               [('layer0_fp32', _i32), ('train_stash', _vp), ('train_stash_bytes', C.c_size_t)]


class EqdHeadParams(C.Structure):
    _fields_ = [('w_mean', _vp), ('b_mean', _vp), ('w_key', _vp), ('w_query', _vp), ('m_qk', _vp), ('leaky_slope', _f32)]


class EqdDropout(C.Structure):
    """eqd_dropout: counter-based dropout masks of a training forward / backward (key in DEVICE memory)."""
    _fields_ = [('key', _vp), ('threshold', C.c_uint32), ('scale', _f32), ('rank', C.c_uint32)]


# symbol -> (restype, argtypes); every symbol include/eqd_iegmn.h declares must be listed here
_G, _L, _H, _D = C.POINTER(EqdGraph), C.POINTER(EqdLayer), C.POINTER(EqdHeadParams), C.POINTER(EqdDropout)
PROTOTYPES = {
    'eqd_abi_version': (C.c_int, []),
    'eqd_workspace_bytes': (C.c_size_t, [_i32, _i32, _i32]),
    'eqd_embed': (C.c_int, [_G, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_embed_checked': (C.c_int, [_G, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_project': (C.c_int, [_G, _L, _vp, _i32, _vp, _vp]),
    'eqd_edge_stage': (C.c_int, [_G, _L, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_edge_stage_ffma': (C.c_int, [_G, _L, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_node_stage': (C.c_int, [_G, _L, _L, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_kv_blocks_bytes': (C.c_size_t, [_i32]),
    'eqd_project_tc': (C.c_int, [_G, _L, _vp, _vp, _vp, _vp]),
    'eqd_project_tc0': (C.c_int, [_G, _L, _vp, _vp, _vp, _vp, _vp]),
    'eqd_attention_tc0': (C.c_int, [_G, _vp, _vp, _vp, _vp, _vp]),
    'eqd_node_mlp_tc0': (C.c_int, [_G, _L, _vp, _vp, _vp, _vp, _vp]),
    'eqd_node_stage_tc0': (C.c_int, [_G, _L, _L, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_kv_blocks': (C.c_int, [_G, _vp, _i32, _i32, _i32, _vp, _vp]),
    'eqd_attention_tc': (C.c_int, [_G, _vp, _vp, _vp, _vp]),
    'eqd_node_mlp_tc': (C.c_int, [_G, _L, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_node_stage_tc': (C.c_int, [_G, _L, _L, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_iegmn_layer_forward': (C.c_int, [_G, _L, _L, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_head_fold': (C.c_int, [_H, _vp, _vp]),
    'eqd_forward_workspace_bytes': (C.c_size_t, [_G]),
    'eqd_iegmn_forward': (C.c_int, [_G, C.POINTER(_L), _i32, _H, C.POINTER(EqdForwardIO), _vp, C.c_size_t, _vp]),
    'eqd_iegmn_forward_dropout': (C.c_int, [_G, C.POINTER(_L), _i32, _H, C.POINTER(EqdForwardIO), _D, _vp, C.c_size_t, _vp]),
    'eqd_dropout_mask': (C.c_int, [_D, _i32, _i32, _i32, _i32, _vp, _vp]),
    'eqd_forward_stash_bytes': (C.c_size_t, [_G, _i32]),
    'eqd_forward_stash_offsets': (C.c_int, [_G, _i32, C.POINTER(C.c_size_t)]),
    'eqd_tn_partial_floats': (C.c_size_t, [C.c_int64, _i32, _i32, C.POINTER(_i32), C.POINTER(_i32)]),
    'eqd_tn_gemm': (C.c_int, [_vp, _i32, _i32, _vp, _i32, _i32, C.c_int64, _f32, _vp, _vp, C.POINTER(_i32), _vp]),
    'eqd_grad_reduce': (C.c_int, [_vp, _i32, C.c_int64, _vp, _vp, _i32, _vp, _vp]),
    'eqd_bwd_node_mlp': (C.c_int, [_G, _L] + [_vp] * 3 + [_i32, _vp, _vp, _i32] + [_vp] * 9 + [C.POINTER(_i32), _vp]),
    'eqd_bwd_node_mlp_dropout': (C.c_int, [_G, _L] + [_vp] * 3 + [_i32, _vp, _vp, _i32] + [_vp] * 9 +
                                 [C.POINTER(_i32), _D, _i32, _vp]),
    'eqd_bwd_attention': (C.c_int, [_G, _L, _vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    'eqd_bwd_edge': (C.c_int, [_G, _L] + [_vp] * 14 + [C.POINTER(_i32), _vp]),
    'eqd_bwd_edge_dropout': (C.c_int, [_G, _L] + [_vp] * 14 + [C.POINTER(_i32), _D, _i32, _vp]),
    'eqd_bwd_edge_gather': (C.c_int, [_G, _vp, _vp, _vp, _vp, _vp, _f32, _vp, _i32, _vp, _vp]),
    'eqd_bwd_project': (C.c_int, [_G, _L, _vp, _vp, _vp, _vp]),
    'eqd_bwd_embed': (C.c_int, [_G, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_bwd_head_workspace_bytes': (C.c_size_t, [_i32, _i32, _i32]),
    'eqd_bwd_head': (C.c_int, [_G, _H] + [_vp] * 9 + [C.c_size_t] + [_vp] * 6),
    'eqd_bwd_head_dropout': (C.c_int, [_G, _H] + [_vp] * 9 + [C.c_size_t] + [_vp] * 5 + [_D, _i32, _vp]),
    'eqd_losses_workspace_bytes': (C.c_size_t, [_i32, _i32]),
    'eqd_losses': (C.c_int, [_G] + [_vp] * 7 + [_i32, _i32, _f32, _f32, _f32, _f32, _vp, C.c_size_t] + [_vp] * 6),
    'eqd_graph_build_workspace_bytes': (C.c_size_t, [_i32]),
    'eqd_graph_build_knn': (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _i32, _vp, C.c_size_t, _vp, _vp, _vp, _vp]),
    'eqd_graph_build_edges': (C.c_int, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_rmsd_meter': (C.c_int, [_G, _vp, _vp, _vp, _vp, _vp, _vp]),
    'eqd_sqnorm_partials': (C.c_int, [_vp, C.c_int64, _vp, _i32, _vp]),
    'eqd_clip_adam': (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64, _vp, _i32, _f32, _f32, _f32, _f32, _f32, _f32, _i32, _f32, _vp, _vp]),
    'eqd_event_create': (_vp, []),
    'eqd_event_destroy': (None, [_vp]),
    'eqd_event_elapsed_ms': (C.c_float, [_vp, _vp]),
    'eqd_keypoints': (C.c_int, [_G, _H, _vp, _vp, _vp, C.c_size_t, _vp, _vp, _vp, _vp]),
    'eqd_kabsch_apply': (C.c_int, [_G, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
}

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def load():
    """Loads the shared library once; raises NativeLibraryError if it is absent (no CPU fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise NativeLibraryError(
            f'{LIB_PATH} not found: build it with equidock_public_b200/csrc/build.sh '
            '(python -c "import __graft_entry__ as g; g.build()"). This engine has no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype, fn.argtypes = res, args
    if lib.eqd_abi_version() != ABI_VERSION:
        raise NativeLibraryError(f'ABI mismatch: library {lib.eqd_abi_version()} vs binding {ABI_VERSION}')
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc == 0:
        return
    if rc <= -1000:
        raise NativeLibraryError(f'{what}: CUDA error {-(rc + 1000)} at kernel launch')
    names = {-1: 'EQD_ERR_BAD_ARG', -2: 'EQD_ERR_UNSUPPORTED', -3: 'EQD_ERR_WORKSPACE'}
    raise NativeLibraryError(f'{what}: {names.get(rc, rc)}')


def ptr(t):
    """Device (or host) pointer of a torch tensor as c_void_p; None -> NULL."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def dropout_threshold(p: float) -> int:
    """Keep iff the Philox word >= this: min(round(p 2^32), 2^32 - 1) (include/eqd_iegmn.h, eqd_dropout)."""
    return min(int(round(float(p) * 2.0 ** 32)), 2 ** 32 - 1)


def dropout_scale(p: float) -> float:
    """fp32(1 / (1 - p)), the factor of a kept element (torch.nn.Dropout's)."""
    return float(C.c_float(1.0 / (1.0 - float(p))).value)


class Dropout:
    """The dropout state of ONE forward: probability, the 64-bit key (a one-element int64 DEVICE tensor drawn from torch's CUDA
    generator on the device: no host sync, reproducible under ``torch.manual_seed``, the CPU generator untouched) and the
    data-parallel rank.  ``struct`` is the eqd_dropout descriptor the entry points take; the backward passes the same one."""

    def __init__(self, p: float, device, rank: int = 0, key=None):
        p = float(p)
        if not 0.0 < p < 1.0:
            raise ValueError(f'dropout probability {p} outside (0, 1)')
        self.p, self.rank = p, int(rank)
        if key is None:
            import torch
            key = torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64, device=device)
        self.key = key
        self.struct = EqdDropout(key.data_ptr(), dropout_threshold(p), dropout_scale(p), self.rank)
