"""ctypes binding of libmpntrack_b200.so (the C ABI declared in include/mpntrack_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, the caller gets
an exception.  PyTorch is used by the callers only to own device memory and streams.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libmpntrack_b200.so')

ABI_VERSION = 2

c_i64, c_i32, c_f32, c_vp = C.c_int64, C.c_int32, C.c_float, C.c_void_p
c_i64p = C.POINTER(C.c_int64)


class CoreWeights(C.Structure):
    """mpn_core_weights"""
    _fields_ = [('dn', c_i32), ('de', c_i32), ('edge_h', c_i32), ('flow_h', c_i32), ('cls_h', c_i32)] + \
               [(n, c_vp) for n in (
                   'edge_w0', 'edge_b0', 'edge_w1', 'edge_b1', 'fin_w0', 'fin_b0', 'fin_w1', 'fin_b1',
                   'fout_w0', 'fout_b0', 'fout_w1', 'fout_b1', 'node_w', 'node_b',
                   'cls_w0', 'cls_b0', 'cls_w1', 'cls_b1')] + [('node_agg', c_i32)]


class EdgeLayout(C.Structure):
    """mpn_edge_layout"""
    _fields_ = [('num_nodes', c_i64), ('num_edges', c_i64), ('num_out', c_i64),
                ('slot_row', c_vp), ('slot_col', c_vp), ('slot_edge', c_vp),
                ('out_ptr', c_vp), ('in_ptr', c_vp)]


# name -> (restype, argtypes); must list every symbol include/mpntrack_b200.h declares
SIGNATURES = {
    'mpn_last_error': (C.c_char_p, []),
    'mpn_abi_version': (C.c_int, []),
    'mpn_device_arch': (C.c_int, []),
    'mpn_launch_count': (C.c_longlong, []),
    'mpn_profile_begin': (C.c_int, []),
    'mpn_profile_end': (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    'mpn_time_valid_pairs_count': (C.c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64p, c_vp]),
    'mpn_time_valid_pairs_fill': (C.c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    'mpn_pair_reid_dist': (C.c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp]),
    'mpn_knn_mask_workspace': (c_i64, [c_i64]),
    'mpn_knn_mask': (C.c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, C.c_int, C.c_int, c_vp, c_vp, c_vp]),
    'mpn_assign_edge_labels': (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, C.c_int, c_vp, c_vp, c_vp]),
    'mpn_compact_pairs': (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64p, c_vp]),
    'mpn_edge_feats_assemble': (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_f32,
                                          c_vp, c_i64, c_vp, c_vp, c_vp]),
    'mpn_knn_graph_workspace': (c_i64, [c_i64, c_i64, c_i64]),
    'mpn_knn_graph_pairs': (C.c_int, [c_vp, c_vp, c_i64p, c_i64, c_vp, c_i64, c_i64, C.c_int, c_i64, C.c_int, c_vp, c_i64,
                                      c_vp, c_vp, c_vp, c_vp, c_i64p, c_i64p, c_vp]),
    'mpn_edge_layout_workspace': (c_i64, [c_i64, c_i64]),
    'mpn_edge_layout_build': (C.c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64p, c_vp]),
    'mpn_avgpool': (C.c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_vp]),
    'mpn_linear': (C.c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_i64, C.c_int, c_vp, c_vp]),
    'mpn_node_encoder_tc_workspace': (c_i64, [c_i64]),
    'mpn_node_encoder_tc': (C.c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    'mpn_gather_rows': (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp]),
    'mpn_edge_encoder': (C.c_int, [c_vp, c_vp, c_i64, C.POINTER(c_i32), c_i32, C.POINTER(c_vp),
                                   C.POINTER(c_vp), c_vp, c_vp]),
    'mpn_mp_workspace': (c_i64, [c_i64, c_i64]),
    'mpn_mp_step': (C.c_int, [C.POINTER(CoreWeights), C.POINTER(EdgeLayout), c_vp, c_vp, c_vp, c_vp, c_i32,
                              c_vp, c_vp, c_vp, c_vp, c_vp]),
    'mpn_mp_forward': (C.c_int, [C.POINTER(CoreWeights), C.POINTER(EdgeLayout), c_vp, c_vp, c_i32, c_i32,
                                 c_vp, c_vp, c_vp, c_vp, c_vp]),
    'mpn_gemm': (C.c_int, [c_vp, c_i64, C.c_int, c_vp, c_i64, c_vp, c_i64, C.c_int, c_vp, C.c_int, C.c_int, c_vp, c_i64,
                           c_i64, c_i64, c_i64, c_vp]),
    'mpn_colsum': (C.c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, C.c_int, c_vp, c_vp]),
    'mpn_gather_cols': (C.c_int, [c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_vp]),
    'mpn_segment_sum': (C.c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_i64, C.c_int, c_vp, c_i64, c_i64, c_vp]),
    'mpn_segment_reduce': (C.c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_i64, C.c_int, c_vp, c_i64, c_i64, C.c_int,
                                     c_vp, c_vp]),
    'mpn_segment_grad': (C.c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, C.c_int, c_vp, c_i64, c_vp]),
    'mpn_batchnorm_forward': (C.c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp, c_f32,
                                        C.c_uint64, c_vp, C.c_int, c_vp, c_i64, c_vp, c_vp]),
    'mpn_batchnorm_backward': (C.c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_f32, c_vp, c_vp,
                                         c_vp, c_i64, c_vp]),
    'mpn_dropout_forward': (C.c_int, [c_vp, c_i64, c_i64, c_i64, c_f32, C.c_uint64, c_vp, C.c_int, c_vp, c_vp]),
    'mpn_dropout_backward': (C.c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_f32, c_vp, c_i64, c_vp]),
    'mpn_relu_mask': (C.c_int, [c_vp, c_vp, c_i64, c_vp]),
    'mpn_adam_step': (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_f32, c_f32, c_f32, c_i64, c_f32, c_vp]),
    'mpn_adam_step_dev': (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_f32, c_f32, c_f32, c_vp, c_f32, c_vp]),
    'mpn_weighted_bce_workspace': (c_i64, []),
    'mpn_weighted_bce': (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'mpn_attn_aggregate': (C.c_int, [c_vp, c_i64, c_i64, C.POINTER(EdgeLayout), c_vp, c_vp, c_vp, c_vp]),
    'mpn_attn_aggregate_backward': (C.c_int, [c_vp, c_i64, c_i64, C.POINTER(EdgeLayout), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'mpn_mp_tc_workspace': (c_i64, [c_i64, c_i64]),
    'mpn_rounding_workspace': (c_i64, [c_i64]),
    'mpn_constr_satisfaction': (C.c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, C.c_int, c_vp, c_vp, c_vp, c_i64p, c_vp]),
    'mpn_greedy_project': (C.c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_i64p, c_vp]),
    'mpn_connected_components_workspace': (c_i64, [c_i64]),
    'mpn_connected_components': (C.c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_i64p, c_vp]),
    'mpn_mp_tc_read_schedule': (C.c_int, [c_vp, c_i64, c_i64, c_i32, C.POINTER(c_i32), C.POINTER(c_f32), C.POINTER(c_f32), c_vp]),
    'mpn_mp_forward_tc': (C.c_int, [C.POINTER(CoreWeights), C.POINTER(EdgeLayout), c_vp, c_vp, c_i32, c_i32,
                                    c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
}

_lib = None


class MpnError(RuntimeError):
    pass


def lib():
    """The loaded shared library; raises if it has not been built (``python -c 'import
    __graft_entry__ as g; g.build()'`` or ``make -C mpntrackseg_b200/csrc``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MpnError(f'{LIB_PATH} is missing: build it with `make -C mpntrackseg_b200/csrc` '
                           '(there is no CPU fallback for the message-passing path)')
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)          # AttributeError if the .so is stale
            fn.restype, fn.argtypes = res, args
        if handle.mpn_abi_version() != ABI_VERSION:
            raise MpnError(f'libmpntrack_b200.so has ABI {handle.mpn_abi_version()}, binding expects {ABI_VERSION}')
        _lib = handle
    return _lib


def check(rc, what=''):
    if rc != 0:
        msg = lib().mpn_last_error().decode('utf-8', 'replace')
        if rc == -1:
            raise ValueError(f'{what}: {msg}')
        raise MpnError(f'{what}: rc={rc}: {msg}')


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
