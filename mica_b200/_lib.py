"""ctypes binding of libmica_b200.so (the C ABI in include/mica_b200.h).

There is no CPU fallback: importing this module raises if the library has not
been built (``python -m mica_b200.build``), and every op raises if the CUDA
driver / a GPU is missing."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libmica_b200.so')

MICA_OK = 0
ERR_NAMES = {-1: 'MICA_ERR_INVALID', -2: 'MICA_ERR_CUDA', -3: 'MICA_ERR_WORKSPACE', -4: 'MICA_ERR_NO_DEVICE'}
NORM_OK, NORM_NO_POSITIVE, NORM_ZERO_PCTL, NORM_PENDING, NORM_PEER_TIMEOUT = 0, 1, 2, 3, 4
DTYPE_I8, DTYPE_I16, DTYPE_F32, DTYPE_U16 = 0, 1, 2, 6      # MICA_DTYPE_*: the MRC modes of these sample types
INT_STATS_RESULT_BYTES = 32
SELECT_HIST_WORDS = 4096
SELECT_PASSES = 7


class MicaError(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f'{LIB_PATH} is missing: build it with `python -m mica_b200.build` '
        '(or __graft_entry__.build()). mica_b200 has no CPU fallback.')

lib = C.CDLL(LIB_PATH)

_p, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t
_I3 = C.c_int * 3
_F3 = C.c_float * 3

#: every symbol include/mica_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    'mica_version': (_i, []),
    'mica_last_error': (C.c_char_p, []),
    'mica_device_count': (_i, []),
    'mica_launch_count': (_i64, []),
    'mica_zoom_output_shape': (_i, [C.POINTER(_i), C.POINTER(_f), C.POINTER(_i)]),
    'mica_resample_workspace_bytes': (_sz, [_i] * 7),
    'mica_resample_force_generic': (_i, [_i]),
    'mica_resample_slab_source_planes': (_i, [_i, _i, _i, _i, _p, _p]),
    'mica_resample_slab_source_planes_general': (_i, [_i, _i, _i, _i, _p, _p]),
    'mica_bspline_resample_f32': (_i, [_p, _i, _i, _i, _i, _i, _p, _i, _i, _i, _i, _i, _p, _sz, _i, _p]),
    'mica_resample': (_i, [_p, _i, _i, _i, _i, _i, _i, _p, _i, _i, _i, _i, _i, _i, _p, _sz, _i, _p]),
    'mica_last_resample_path': (_i, [_i]),
    'mica_select_workspace_bytes': (_sz, []),
    'mica_select_workspace_bytes_for': (_sz, [_i64]),
    'mica_select_set_compact': (_i, [_p, _sz, _p]),
    'mica_select_compact_info': (_i, [_p, C.POINTER(_i64), _p]),
    'mica_select_init': (_i, [_p, _i64, _p]),
    'mica_select_hist': (_i, [_p, _i64, _p, _i, _p]),
    'mica_select_hist_ptr': (_p, [_p]),
    'mica_select_pick': (_i, [_p, _i, _p]),
    'mica_select_force_fallback': (_i, [_i]),
    'mica_order_stats_f32': (_i, [_p, _i64, _p, _p]),
    'mica_select_result': (_i, [_p, C.POINTER(_f), C.POINTER(_f), C.POINTER(_i64), C.POINTER(_i), _p]),
    'mica_select_result_async': (_i, [_p, _p, _p]),
    'mica_normalize_apply_f32': (_i, [_p, _p, _i64, _p, _p]),
    'mica_int_stats_workspace_bytes': (_sz, []),
    'mica_int_order_stats': (_i, [_p, _i, _i64, _p, _p]),
    'mica_int_stats_init': (_i, [_p, _i, _i64, _p]),
    'mica_int_stats_hist': (_i, [_p, _i, _i64, _p, _p]),
    'mica_int_stats_hist_ptr': (_p, [_p]),
    'mica_int_stats_pick': (_i, [_p, _i, _p]),
    'mica_int_peer_buffer_bytes': (_sz, []),
    'mica_int_stats_peer_publish': (_i, [_p, _i, _p, _i, _i, _i, _i, _p]),
    'mica_int_stats_peer_sum': (_i, [_p, _i, _p, _i, _i, _i, _i, _p]),
    'mica_int_stats_result': (_i, [_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(_i64), C.POINTER(_i),
                                   _p]),
    'mica_int_stats_result_async': (_i, [_p, _p, _p]),
    'mica_normalize_apply_int': (_i, [_p, _i, _p, _i64, _p, _p]),
    'mica_normalize_force_reference_arith': (_i, [_i]),
    'mica_select_set_thresholds': (_i, [_p, _f, _f, _p]),
    'mica_peer_buffer_bytes': (_sz, []),
    'mica_peer_alloc': (_i, [C.POINTER(_p), _p]),
    'mica_peer_open': (_i, [_p, C.POINTER(_p)]),
    'mica_peer_close': (_i, [_p]),
    'mica_peer_free': (_i, [_p]),
    'mica_peer_enable': (_i, [_i, _i]),
    'mica_select_peer_reduce': (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    'mica_halo_buffer_bytes': (_sz, [_i64]),
    'mica_ipc_alloc': (_i, [_sz, C.POINTER(_p), _p]),
    'mica_halo_publish': (_i, [_p, _i64, _i64, _i64, _i64, _p, _i, _i, _i, _i, _i64, _p]),
    'mica_halo_pull': (_i, [_p, _i64, _p, _i64, _p, _i, _i, _i, _i, _i64, _p, _p]),
    'mica_halo_publish_bytes': (_i, [_p, _i64, _i64, _i64, _i64, _p, _i, _i, _i, _i, _i64, _p]),
    'mica_halo_pull_bytes': (_i, [_p, _i64, _p, _i64, _p, _i, _i, _i, _i, _i64, _p, _p]),
    'mica_af3_encode': (_i, [_p, _p, _p, _i64, _f, _f, _f, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p]),
    'mica_af3_bins_workspace_bytes': (_sz, [_i64, _i, _i, _i, C.POINTER(_i), _i, _i]),
    'mica_af3_bin_atoms': (_i, [_p, _p, _p, _i64, _f, _f, _f, _i, _i, _i, _i, _i, _i, C.POINTER(_i), _i, _i,
                                _p, _sz, _p, _p]),
    'mica_af3_fill_cubes': (_i, [_p, _i64, _i, _i, _i, C.POINTER(_i), _i, _i, _p, _i, _p, _i, _p, _i64, _p, _p]),
    'mica_extract_cubes': (_i, [_p, _i64, _i, _i, _i, _i, _i, _i, C.POINTER(_i), _i, _i, _p, _i, _p, _i64,
                                _p, _p, _p]),
    'mica_last_extract_path': (_i, []),
    'mica_postproc_stitch': (_i, [_p, _p, _p, _p, _i, _i, _i, _i, C.POINTER(_i), C.POINTER(_i), _i, _i,
                                  _p, _p, _p, _p, _p]),
    'mica_stitch_cubes': (_i, [_p, _i, _p, _i, _i, _i, _i, C.POINTER(_i), C.POINTER(_i), _i, _i, _p, _p]),
    'mica_postproc_stitch_peer': (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, C.POINTER(_i), _i, _p]),
    'mica_overlap_accumulate_fixed': (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, C.POINTER(_f), _p, _p, _p]),
    'mica_overlap_accumulate_fixed_peer': (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, C.POINTER(_f), _p, _p, _i,
                                                C.POINTER(_i), _i, _p]),
    'mica_overlap_finalize_fixed': (_i, [_p, _i64, _p]),
    'mica_peer_atomics_supported': (_i, [_i, _i]),
    'mica_parse_pdb': (_i64, [C.c_char_p, _i64, _i, _i64, _p, _p, _p, _p, _p, _p, _p]),
    # SURVEY 8(f) N1: candidates
    'mica_cand_threshold_workspace_bytes': (_sz, [_i64]),
    'mica_cand_threshold_count': (_i, [_p, _i64, _f, _p, _sz, _p, _p]),
    'mica_cand_threshold_write': (_i, [_p, _i, _i, _i, _f, _p, _p, _p, _i64, _p]),
    'mica_gather_f32': (_i, [_p, _p, _i64, _p, _p]),
    'mica_dbscan_workspace_bytes': (_sz, [_i, _i, _i, _i64]),
    'mica_dbscan_lattice': (_i, [_p, _i64, _i, _i, _i, _i, _i, _p, _sz, _p, _p, _p]),
    'mica_cand_cluster_scores': (_i, [_p, _p, _i64, _i, _p, _p, _p]),
    'mica_cand_valid_points': (_i, [_p, _p, _i64, _i, _p, _p]),
    'mica_cand_clustered_volume': (_i, [_p, _i64, _p, _p, _i64, _p, _p]),
    'mica_cand_nms': (_i, [_p, _i, _i, _i, _p, _p, _i64, _i, _p, _p, C.POINTER(_i), _p]),
    'mica_cand_picks_workspace_bytes': (_sz, [_i64]),
    'mica_cand_nms_picks': (_i, [_p, _i, _i, _p, _p, _i64, _i64, _p, _sz, _p, _p, _p, _p]),
    'mica_cand_refine': (_i, [_p, _p, _p, _i, _i, _i, _p, _i64, _p, _p, _p, _p, _p]),
    'mica_cand_neighbor_graph': (_i, [_p, _i64, _p, _i, _i, _i, _p, _p, _p]),
    'mica_cand_best_neighbors': (_i, [_p, _i64, _p, _p]),
    'mica_cand_neighbor_lists': (_i, [_p, _i64, C.c_double, _i, _p, _p, _p]),
    # N3: label masks, N4: docking masks
    'mica_label_class_mask': (_i, [_p, _p, _i64, _f, _f, _f, _i, _i, _i, _i, _i, _i, _p, _p, _p]),
    'mica_label_aa_mask_workspace_bytes': (_sz, [_i, _i, _i]),
    'mica_label_aa_mask': (_i, [_p, _p, _i64, _f, _f, _f, _i, _i, _i, _i, _i, _i, _p, _sz, _p, _p, _p]),
    'mica_contour_threshold_f32': (_i, [_p, _p, _i64, _f, _p]),
    'mica_zero_around_atoms': (_i, [_p, _i64, C.POINTER(_f), C.POINTER(_f), C.c_double, _i, _i, _i, _p, _p, _p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)          # AttributeError here == header / library mismatch
    _fn.restype, _fn.argtypes = _res, _args


def last_error() -> str:
    return lib.mica_last_error().decode('utf-8', 'replace')


def check(rc: int, what: str = ''):
    if rc != MICA_OK:
        raise MicaError(f'{what or "mica call"} failed: {ERR_NAMES.get(rc, rc)}: {last_error()}')


def int3(v):
    return _I3(int(v[0]), int(v[1]), int(v[2]))


def float3(v):
    return _F3(float(v[0]), float(v[1]), float(v[2]))
