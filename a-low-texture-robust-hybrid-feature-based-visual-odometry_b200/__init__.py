"""hvo-front: B200-native (sm_100a) feature front-end of the hybrid point/line/plane VO.

This package is a thin ctypes binding over the C ABI in include/hvo_capi.h (libhvofront.so, hand-written
CUDA).  The classes mirror the reference's C++ interfaces (names, argument meaning, error behaviour) so the
parity tests read like calls into the reference:

    ORBextractor(nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST)   reference include/ORBextractor.h:51
    ORBextractor.__call__(image, mask) -> (keypoints, descriptors)        reference include/ORBextractor.h:59

There is no CPU fallback: importing works without a GPU (so the ABI can be inspected), but every compute call
raises HvoError when the CUDA library or device is missing.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('HVO_LIB_PATH') or os.path.join(_HERE, 'libhvofront.so')  # HVO_LIB_PATH: tuning aid (a differently built library)

HVO_OK, HVO_ERR_ARG, HVO_ERR_CUDA, HVO_ERR_STATE, HVO_ERR_OVERFLOW = 0, 1, 2, 3, 4

KP_DTYPE = np.dtype([('x', '<f4'), ('y', '<f4'), ('size', '<f4'), ('angle', '<f4'), ('response', '<f4'),
                     ('octave', '<i4'), ('class_id', '<i4')])


class HvoError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f'hvo status {status}: {msg}')
        self.status = status


class _OrbParams(C.Structure):
    _fields_ = [('nfeatures', C.c_int), ('scale_factor', C.c_float), ('nlevels', C.c_int),
                ('ini_th_fast', C.c_int), ('min_th_fast', C.c_int)]


class _RgbdParams(C.Structure):
    _fields_ = [('depth_factor', C.c_float), ('bf', C.c_float), ('distorted', C.c_int)]


class _Camera(C.Structure):
    _fields_ = [(n, C.c_float) for n in ('fx', 'fy', 'cx', 'cy', 'k1', 'k2', 'p1', 'p2', 'k3')]


def _dist5(dist):
    """mDistCoef (4 entries, or 5 when Camera.k3 != 0) -> k1, k2, p1, p2, k3 as float32."""
    d = np.asarray(dist, np.float32).ravel()
    if len(d) not in (4, 5):
        raise HvoError(HVO_ERR_ARG, f'dist must hold k1, k2, p1, p2 [, k3] (got {len(d)} values)')
    return np.concatenate([d, np.zeros(5 - len(d), np.float32)])


def _camera(K, dist):
    """hvo_camera of mK (3x3) and mDistCoef, both narrowed to float32 as the reference stores them."""
    K = np.asarray(K, np.float32).reshape(3, 3)
    return _Camera(K[0, 0], K[1, 1], K[0, 2], K[1, 2], *_dist5(dist))


_lib = None
_vp = C.c_void_p

# name -> (restype, argtypes); every symbol include/hvo_capi.h declares
ABI = {
    'hvo_last_error': (C.c_char_p, []),
    'hvo_version': (C.c_char_p, []),
    'hvo_device_count': (C.c_int, [C.POINTER(C.c_int)]),
    'hvo_orb_create': (C.c_int, [C.POINTER(_OrbParams), C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    'hvo_orb_destroy': (None, [_vp]),
    'hvo_orb_capacity': (C.c_int, [_vp]),
    'hvo_orb_get_tables': (C.c_int, [_vp] * 6),
    'hvo_orb_extract': (C.c_int, [_vp, _vp, C.c_size_t, _vp, _vp, C.c_int, C.POINTER(C.c_int)]),
    'hvo_orb_extract_batch': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp, C.POINTER(_RgbdParams), _vp, _vp]),
    'hvo_orb_extract_batch_device': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp, C.POINTER(_RgbdParams), _vp, _vp]),
    'hvo_orb_sync': (C.c_int, [_vp]),
    'hvo_orb_timer_start': (C.c_int, [_vp]),
    'hvo_orb_timer_stop': (C.c_int, [_vp, C.POINTER(C.c_float)]),
    'hvo_orb_set_profiling': (C.c_int, [_vp, C.c_int]),
    'hvo_orb_stage_times': (C.c_int, [_vp, C.POINTER(C.c_float)]),
    'hvo_orb_last_launches': (C.c_int, [_vp]),
    'hvo_stereo_uright_from_depth': (C.c_int, [_vp, _vp, C.c_int, C.c_float, _vp]),
    'hvo_undistort_points': (C.c_int, [C.POINTER(_Camera), _vp, C.c_int, _vp]),
    'hvo_image_bounds': (C.c_int, [C.POINTER(_Camera), C.c_int, C.c_int] + [C.POINTER(C.c_float)] * 4),
    'hvo_orb_undistort_batch_device': (C.c_int, [_vp, C.POINTER(_Camera), _vp, _vp, C.c_int, _vp, C.c_float, _vp, _vp]),
    'hvo_membership4_expand': (C.c_int, [_vp, C.c_int, _vp]),
    'hvo_seq_create': (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int, C.c_int, _vp]),
    'hvo_seq_destroy': (None, [_vp]),
    'hvo_seq_devices': (C.c_int, [_vp]),
    'hvo_seq_capacities': (C.c_int, [_vp, _vp, _vp, _vp]),
    'hvo_seq_shard': (None, [C.c_int, C.c_int, C.c_int, _vp, _vp]),
    'hvo_seq_extract': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp]),
    'hvo_seq_set_vocabulary': (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int]),
    'hvo_seq_extract_bow': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp]),
    'hvo_seq_extract_grid': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp]),
    'hvo_seq_image_bounds': (C.c_int, [_vp] + [C.POINTER(C.c_float)] * 4),
    'hvo_seq_line_grid_capacity': (C.c_int, [_vp]),
    'hvo_seq_extract_lpvo': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    'hvo_seq_lpvo_capacity': (C.c_int, [_vp]),
    'hvo_seq_last_ms': (C.c_float, [_vp]),
    'hvo_normals3_expand': (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _vp]),
    'hvo_orb_level_size': (C.c_int, [_vp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'hvo_orb_get_pyramid_level': (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_size_t]),
    'hvo_orb_get_candidates': (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int, C.POINTER(C.c_int)]),
    'hvo_matcher_create': (C.c_int, [C.c_int, C.POINTER(_vp)]),
    'hvo_matcher_destroy': (None, [_vp]),
    'hvo_hamming_distance': (C.c_int, [_vp, _vp]),
    'hvo_match_knn2': (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, _vp, _vp]),
    'hvo_match_knn2_device': (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, _vp, _vp]),
    'hvo_match_distinctive': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp]),
    'hvo_match_lines_epipolar': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp, C.c_int, _vp, C.c_float, C.c_float, _vp]),
    'hvo_matcher_sync': (C.c_int, [_vp]),
    'hvo_matcher_timer_start': (C.c_int, [_vp]),
    'hvo_matcher_timer_stop': (C.c_int, [_vp, C.POINTER(C.c_float)]),
    'hvo_lbd_create': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    'hvo_lbd_destroy': (None, [_vp]),
    'hvo_lbd_compute': (C.c_int, [_vp, _vp, C.c_size_t, _vp, C.c_int, _vp]),
    'hvo_lbd_compute_batch': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    'hvo_lbd_compute_batch_device': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp]),
    'hvo_lbd_get_gradients': (C.c_int, [_vp, C.c_int, _vp, _vp]),
    'hvo_lbd_sync': (C.c_int, [_vp]),
    'hvo_lbd_timer_start': (C.c_int, [_vp]),
    'hvo_lbd_timer_stop': (C.c_int, [_vp, C.POINTER(C.c_float)]),
    'hvo_bow_create': (C.c_int, [C.c_int, C.POINTER(_vp)]),
    'hvo_bow_destroy': (None, [_vp]),
    'hvo_bow_set_vocabulary': (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_int]),
    'hvo_bow_transform': (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'hvo_bow_last_launches': (C.c_int, [_vp]),
    'hvo_proj_create': (C.c_int, [C.c_int, C.POINTER(_vp)]),
    'hvo_proj_destroy': (None, [_vp]),
    'hvo_proj_set_frame': (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float]),
    'hvo_proj_get_grid': (C.c_int, [_vp, _vp, _vp]),
    'hvo_proj_features_in_area': (C.c_int, [_vp, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int, _vp, C.c_int, C.POINTER(C.c_int)]),
    'hvo_proj_search': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, C.c_int, C.c_int, C.c_float, _vp, _vp, C.POINTER(C.c_int)]),
    'hvo_proj_set_level_sigma': (C.c_int, [_vp, _vp, C.c_int]),
    'hvo_proj_set_window_origin': (C.c_int, [_vp, C.c_float, C.c_float]),
    'hvo_proj_last_rounds': (C.c_int, [_vp]),
    'hvo_proj_last_launches': (C.c_int, [_vp]),
    'hvo_proj_match_candidates': (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, _vp, _vp, _vp]),
    'hvo_proj_search_candidates': (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, _vp, _vp, C.c_int, C.c_float, _vp, _vp, C.POINTER(C.c_int)]),
    'hvo_proj_search_triangulation': (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, C.c_float, C.c_float, _vp, _vp,
                                               C.c_int, C.c_int, C.c_int, _vp, _vp, C.POINTER(C.c_int)]),
    'hvo_predict_scale_thresholds': (C.c_int, [C.c_float, C.c_int, C.c_int, _vp]),
    'hvo_proj_frustum_points': (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_float, _vp]),
    'hvo_proj_search_local_map': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_float, C.c_float, _vp, _vp, C.c_int, C.c_float, _vp, _vp, _vp,
                                           C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'hvo_proj_search_initialization': (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_float, _vp, _vp, C.POINTER(C.c_int)]),
    'hvo_proj_timer_start': (C.c_int, [_vp]),
    'hvo_proj_timer_stop': (C.c_int, [_vp, C.POINTER(C.c_float)]),
    'hvo_line_create': (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    'hvo_line_destroy': (None, [_vp]),
    'hvo_line_max_lines': (C.c_int, [_vp]),
    'hvo_line_segment_capacity': (C.c_int, [_vp]),
    'hvo_line_scaled_size': (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'hvo_line_extract': (C.c_int, [_vp, _vp, C.c_size_t, _vp, _vp, _vp, C.c_int, C.POINTER(C.c_int)]),
    'hvo_line_extract_batch': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    'hvo_line_extract_batch_device': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    'hvo_line_detect_batch': (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, _vp]),
    'hvo_line_set_culling': (C.c_int, [_vp, C.c_int]),
    'hvo_line_cull': (C.c_int, [_vp, _vp, C.c_size_t, _vp, _vp, C.c_int, _vp, C.POINTER(C.c_int)]),
    'hvo_line_cull_batch_device': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    'hvo_line_get_scaled': (C.c_int, [_vp, C.c_int, _vp]),
    'hvo_line_get_seed_order': (C.c_int, [_vp, C.c_int, _vp, C.c_int, C.POINTER(C.c_int)]),
    'hvo_line_set_profiling': (C.c_int, [_vp, C.c_int]),
    'hvo_line_stage_times': (C.c_int, [_vp, C.POINTER(C.c_float)]),
    'hvo_line_last_launches': (C.c_int, [_vp]),
    'hvo_line_sync': (C.c_int, [_vp]),
    'hvo_line_timer_start': (C.c_int, [_vp]),
    'hvo_line_timer_stop': (C.c_int, [_vp, C.POINTER(C.c_float)]),
    'hvo_plane_create': (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    'hvo_plane_destroy': (None, [_vp]),
    'hvo_plane_detect': (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, _vp]),
    'hvo_plane_detect_batch': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_int, _vp]),
    'hvo_plane_detect_batch_device': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_int, _vp]),
    'hvo_plane_detect_batch_device_u8': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_int, _vp, _vp]),
    'hvo_plane_last_launches': (C.c_int, [_vp]),
    'hvo_plane_get_phase_cycles': (C.c_int, [_vp, C.c_int, _vp]),
    'hvo_plane_blocks_device': (C.c_int, [_vp, _vp, C.c_int]),
    'hvo_plane_get_blocks': (C.c_int, [_vp, C.c_int, _vp]),
    'hvo_plane_sync': (C.c_int, [_vp]),
    'hvo_plane_timer_start': (C.c_int, [_vp]),
    'hvo_plane_timer_stop': (C.c_int, [_vp, C.POINTER(C.c_float)]),
    'hvo_normals_create': (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    'hvo_normals_destroy': (None, [_vp]),
    'hvo_normals_count': (C.c_int, [_vp]),
    'hvo_normals_compute_batch': (C.c_int, [_vp, _vp, C.c_int, _vp]),
    'hvo_normals_compute_batch_device': (C.c_int, [_vp, _vp, C.c_int, _vp]),
    'hvo_normals_get_distance_map': (C.c_int, [_vp, C.c_int, _vp]),
    'hvo_normals_sync': (C.c_int, [_vp]),
    'hvo_normals_timer_start': (C.c_int, [_vp]),
    'hvo_normals_timer_stop': (C.c_int, [_vp, C.POINTER(C.c_float)]),
    'hvo_lproj_create': (C.c_int, [C.c_int, C.POINTER(_vp)]),
    'hvo_lproj_destroy': (None, [_vp]),
    'hvo_lproj_set_frame': (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float]),
    'hvo_lproj_get_grid': (C.c_int, [_vp, _vp, _vp, C.c_int, C.POINTER(C.c_int)]),
    'hvo_lproj_features_in_area': (C.c_int, [_vp, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _vp, C.c_int, C.POINTER(C.c_int)]),
    'hvo_lproj_search': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, C.c_int, C.c_float, _vp, _vp, C.POINTER(C.c_int)]),
    'hvo_lproj_frustum_lines': (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_float, _vp]),
    'hvo_lproj_search_local_map': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_float, C.c_float, _vp, C.c_float, _vp, _vp, _vp,
                                            C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'hvo_lproj_last_rounds': (C.c_int, [_vp]),
    'hvo_lproj_last_launches': (C.c_int, [_vp]),
    'hvo_lpvo_create': (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    'hvo_lpvo_destroy': (None, [_vp]),
    'hvo_lpvo_capacity': (C.c_int, [_vp]),
    'hvo_lpvo_compute_batch': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    'hvo_lpvo_compute_batch_device': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    'hvo_lpvo_sync': (C.c_int, [_vp]),
    'hvo_lpvo_timer_start': (C.c_int, [_vp]),
    'hvo_lpvo_timer_stop': (C.c_int, [_vp, C.POINTER(C.c_float)]),
    'hvo_timeline_enable': (C.c_int, [C.c_int]),
    'hvo_timeline_dump': (C.c_int, [C.c_char_p, C.c_int]),
    'hvo_frame_create': (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    'hvo_frame_destroy': (None, [_vp]),
    'hvo_frame_capacities': (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'hvo_frame_lanes': (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'hvo_frame_extract_batch': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp]),
    'hvo_frame_extract_batch_async': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp]),
    'hvo_frame_extract_batch_device': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp]),
    'hvo_frame_set_vocabulary': (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int]),
    'hvo_frame_extract_batch_bow': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp]),
    'hvo_frame_extract_batch_async_bow': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp]),
    'hvo_frame_extract_batch_device_bow': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp]),
    'hvo_frame_extract_batch_grid': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp]),
    'hvo_frame_extract_batch_async_grid': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp]),
    'hvo_frame_extract_batch_device_grid': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp]),
    'hvo_frame_image_bounds': (C.c_int, [_vp] + [C.POINTER(C.c_float)] * 4),
    'hvo_frame_line_grid_capacity': (C.c_int, [_vp]),
    'hvo_frame_extract_batch_lpvo': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    'hvo_frame_extract_batch_async_lpvo': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    'hvo_frame_extract_batch_device_lpvo': (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    'hvo_frame_lpvo_capacity': (C.c_int, [_vp]),
    'hvo_frame_last_launches': (C.c_int, [_vp]),
    'hvo_frame_sync': (C.c_int, [_vp]),
    'hvo_frame_timer_start': (C.c_int, [_vp]),
    'hvo_frame_timer_stop': (C.c_int, [_vp, C.POINTER(C.c_float)]),
}


def timeline(on):
    """profiling aid: start (True) or stop (False) recording one timed event per kernel launch site."""
    _check(lib().hvo_timeline_enable(int(bool(on))))


def timeline_dump():
    """-> list of (ms since the first mark, stream id, name); call after the work has been synchronised."""
    buf = C.create_string_buffer(1 << 20)
    _check(lib().hvo_timeline_dump(buf, len(buf)))
    return [(float(a), int(b), c) for a, b, c in (ln.split() for ln in buf.value.decode().splitlines())]


def lib():
    """Load libhvofront.so.  Fails loudly when it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HvoError(HVO_ERR_STATE, f'{LIB_PATH} is missing: run __graft_entry__.build() (nvcc, sm_100a)')
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in ABI.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def _check(st):
    if st != HVO_OK:
        raise HvoError(st, lib().hvo_last_error().decode())


def _np_ptr(a):
    return a.ctypes.data_as(_vp)


def device_count():
    n = C.c_int(0)
    _check(lib().hvo_device_count(C.byref(n)))
    return n.value


# hvo_frustum_cam / hvo_map_point / hvo_track_point / hvo_map_line / hvo_track_line (include/hvo_capi.h)
FRUSTUM_CAM_DTYPE = np.dtype([('Rcw', '<f4', (9,)), ('tcw', '<f4', (3,)), ('Ow', '<f4', (3,)), ('fx', '<f4'), ('fy', '<f4'), ('cx', '<f4'),
                              ('cy', '<f4'), ('bf', '<f4'), ('min_x', '<f4'), ('min_y', '<f4'), ('max_x', '<f4'), ('max_y', '<f4'),
                              ('log_scale_factor', '<f4'), ('n_levels', '<i4')])
MAP_POINT_DTYPE = np.dtype([('pos', '<f4', (3,)), ('normal', '<f4', (3,)), ('min_distance', '<f4'), ('max_distance', '<f4')])
TRACK_POINT_DTYPE = np.dtype([('u', '<f4'), ('v', '<f4'), ('ur', '<f4'), ('level', '<i4'), ('view_cos', '<f4'), ('in_view', '<i4')])
MAP_LINE_DTYPE = np.dtype([('pos', '<f8', (6,)), ('normal', '<f8', (3,)), ('dir', '<f8', (3,)), ('min_distance', '<f4'), ('max_distance', '<f4')])
TRACK_LINE_DTYPE = np.dtype([('x1', '<f4'), ('y1', '<f4'), ('x2', '<f4'), ('y2', '<f4'), ('level', '<i4'), ('view_cos', '<f4'), ('in_view', '<i4')])
assert FRUSTUM_CAM_DTYPE.itemsize == 104 and MAP_POINT_DTYPE.itemsize == 32 and TRACK_POINT_DTYPE.itemsize == 24
assert MAP_LINE_DTYPE.itemsize == 104 and TRACK_LINE_DTYPE.itemsize == 28


def frustum_cam(Rcw, tcw, fx, fy, cx, cy, bf, bounds, scale_factor=1.2, n_levels=8):
    """hvo_frustum_cam of a frame pose: mOw = -Rcw^T * tcw as Frame::UpdatePoseMatrices computes it (cv::gemm on CV_32F: float products
    summed in k order), mfLogScaleFactor = log(scaleFactor) narrowed to float (src/Frame.cc:105)."""
    c = np.zeros((), FRUSTUM_CAM_DTYPE)
    R = np.asarray(Rcw, np.float32).reshape(3, 3); t = np.asarray(tcw, np.float32).reshape(3)
    Ow = np.zeros(3, np.float32)
    for i in range(3):
        acc = np.float32(0)
        for k in range(3):
            acc = np.float32(acc + np.float32(np.float32(-R[k, i]) * t[k]))   # -mRcw.t() * mtcw
        Ow[i] = acc
    c['Rcw'] = R.reshape(9); c['tcw'] = t; c['Ow'] = Ow
    c['fx'], c['fy'], c['cx'], c['cy'], c['bf'] = fx, fy, cx, cy, bf
    c['min_x'], c['min_y'], c['max_x'], c['max_y'] = bounds
    c['log_scale_factor'] = np.float32(np.log(np.float64(np.float32(scale_factor))))
    c['n_levels'] = n_levels
    return c


def undistort_points(pts, K, dist):
    """cv2.undistortPoints(pts, K, dist, None, K) bit for bit (hvo_undistort_points, host): pts [n,2] -> float32 [n,2]; K 3x3,
    dist = k1, k2, p1, p2 [, k3], narrowed to float32 as the reference's mK / mDistCoef.  No k1 == 0 shortcut."""
    p = np.ascontiguousarray(np.asarray(pts, np.float32).reshape(-1, 2))
    out = np.empty_like(p)
    _check(lib().hvo_undistort_points(C.byref(_camera(K, dist)), _np_ptr(p), len(p), _np_ptr(out)))
    return out


def image_bounds(K, dist, width, height):
    """Frame::ComputeImageBounds (reference src/Frame.cc:1733-1760) -> (mnMinX, mnMaxX, mnMinY, mnMaxY) as float32."""
    v = [C.c_float(0) for _ in range(4)]
    _check(lib().hvo_image_bounds(C.byref(_camera(K, dist)), int(width), int(height), *[C.byref(a) for a in v]))
    return tuple(np.float32(a.value) for a in v)


def predict_scale_thresholds(log_scale_factor, lo, n):
    thr = np.empty(max(n, 1), np.float32)
    _check(lib().hvo_predict_scale_thresholds(float(log_scale_factor), int(lo), int(n), _np_ptr(thr)))
    return thr[:n]


class ORBextractor:
    """Mirror of ORB_SLAM2::ORBextractor (reference include/ORBextractor.h:46-110).

    Extra constructor arguments (image size, max_batch, device) size the device buffers; when omitted the
    handle is created lazily from the first image, as the C++ shim does.
    """

    def __init__(self, nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST, width=None, height=None, max_batch=1,
                 device=0):
        self.nfeatures, self.scaleFactor, self.nlevels = int(nfeatures), float(scaleFactor), int(nlevels)
        self.iniThFAST, self.minThFAST = int(iniThFAST), int(minThFAST)
        self.max_batch, self.device = int(max_batch), int(device)
        self._h = None
        self._size = None
        if width is not None and height is not None:
            self._create(int(width), int(height))

    # -- lifecycle ------------------------------------------------------------------------------------
    def _create(self, w, h):
        self.close()
        p = _OrbParams(self.nfeatures, self.scaleFactor, self.nlevels, self.iniThFAST, self.minThFAST)
        out = _vp()
        _check(lib().hvo_orb_create(C.byref(p), w, h, self.max_batch, self.device, C.byref(out)))
        self._h = out
        self._size = (w, h)
        self.capacity = lib().hvo_orb_capacity(self._h)

    def close(self):
        if getattr(self, '_h', None):
            lib().hvo_orb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ensure(self, w, h):
        if self._h is None or self._size != (w, h):
            self._create(w, h)

    # -- getters (ORBextractor.h:63-83) -----------------------------------------------------------------
    def GetLevels(self):
        return self.nlevels

    def GetScaleFactor(self):
        return self.scaleFactor

    def _tables(self):
        if self._h is None:
            raise HvoError(HVO_ERR_STATE, 'extractor has no device handle yet (no image size known)')
        n = self.nlevels
        t = [np.empty(n, np.float32) for _ in range(4)] + [np.empty(n, np.int32)]
        _check(lib().hvo_orb_get_tables(self._h, *[_np_ptr(a) for a in t]))
        return t

    def GetScaleFactors(self):
        return self._tables()[0]

    def GetInverseScaleFactors(self):
        return self._tables()[1]

    def GetScaleSigmaSquares(self):
        return self._tables()[2]

    def GetInverseScaleSigmaSquares(self):
        return self._tables()[3]

    def GetFeaturesPerLevel(self):
        return self._tables()[4]

    # -- operator() ---------------------------------------------------------------------------------
    def __call__(self, image, mask=None):
        """(keypoints[KP_DTYPE], descriptors[n,32] uint8).  The mask is ignored (ORBextractor.h:57)."""
        if image is None or image.size == 0:
            return np.empty(0, KP_DTYPE), np.empty((0, 32), np.uint8)  # silent return, .cc:1044-1045
        if image.dtype != np.uint8 or image.ndim != 2:
            raise HvoError(HVO_ERR_ARG, 'image must be 8-bit single channel (assert at ORBextractor.cc:1048)')
        if image.strides[1] != 1:
            image = np.ascontiguousarray(image)
        h, w = image.shape
        self._ensure(w, h)
        kps = np.empty(self.capacity, KP_DTYPE)
        desc = np.empty((self.capacity, 32), np.uint8)
        n = C.c_int(0)
        _check(lib().hvo_orb_extract(self._h, _vp(image.ctypes.data), image.strides[0], _np_ptr(kps), _np_ptr(desc),
                                     self.capacity, C.byref(n)))
        return kps[:n.value].copy(), desc[:n.value].copy()

    # -- batched host path ----------------------------------------------------------------------------
    def extract_batch(self, frames, depth16=None, depth_factor=None, bf=None, out=None, distorted=False, camera=None):
        """frames [n,h,w] uint8 (host; pinned memory makes the copies asynchronous).  Returns
        dict(counts, kps [n,cap], desc [n,cap,32], depth, uright).  distorted: the camera has k1 != 0, so mvuRight needs the
        undistorted keypoints (Frame.cc:1944): uright comes back as -1, form it with stereo_uright_from_depth().
        camera = (K, dist): Frame::UndistortKeyPoints on the device as well (hvo_orb_undistort_batch_device): the result gains
        kps_un [n,cap] (mvKeysUn) and uright is formed from it."""
        assert frames.dtype == np.uint8 and frames.ndim == 3 and frames.flags.c_contiguous
        n, h, w = frames.shape
        self._ensure(w, h)
        if camera is not None:
            if out is not None:
                raise HvoError(HVO_ERR_ARG, 'out= is not supported together with camera=')
            return self._extract_batch_undistorted(frames, depth16, depth_factor, bf, camera)
        cap = self.capacity
        if out is None:
            out = dict(counts=np.empty(n, np.int32), kps=np.empty((n, cap), KP_DTYPE), desc=np.empty((n, cap, 32), np.uint8))
            if depth16 is not None:
                out['depth'] = np.empty((n, cap), np.float32)
                out['uright'] = np.empty((n, cap), np.float32)
        rg = None
        if depth16 is not None:
            assert depth16.dtype == np.uint16 and depth16.shape == frames.shape and depth16.flags.c_contiguous
            rg = C.byref(_RgbdParams(float(depth_factor), float(bf), int(bool(distorted))))
        _check(lib().hvo_orb_extract_batch(self._h, _np_ptr(frames), n, _np_ptr(out['kps']), _np_ptr(out['desc']),
                                           _np_ptr(out['counts']), _np_ptr(depth16) if depth16 is not None else None, rg,
                                           _np_ptr(out['depth']) if depth16 is not None else None,
                                           _np_ptr(out['uright']) if depth16 is not None else None))
        return out

    def _extract_batch_undistorted(self, frames, depth16, depth_factor, bf, camera):
        import torch
        n, cap = len(frames), self.capacity
        dev = torch.device('cuda', self.device)
        g = torch.from_numpy(frames).to(dev)
        kps = torch.empty((n, cap, KP_DTYPE.itemsize), dtype=torch.uint8, device=dev)
        kps_un = torch.empty_like(kps)
        desc = torch.empty((n, cap, 32), dtype=torch.uint8, device=dev)
        counts = torch.empty(n, dtype=torch.int32, device=dev)
        rgbd = depth16 is not None
        if rgbd:
            assert depth16.dtype == np.uint16 and depth16.shape == frames.shape
            d16 = torch.from_numpy(np.ascontiguousarray(depth16)).to(dev)
            kd, ku = torch.empty((n, cap), dtype=torch.float32, device=dev), torch.empty((n, cap), dtype=torch.float32, device=dev)
        torch.cuda.synchronize(dev)   # the uploads ran on torch's stream; the handle's stream starts after them
        self.extract_batch_device(g.data_ptr(), n, kps.data_ptr(), desc.data_ptr(), counts.data_ptr(), d16.data_ptr() if rgbd else None,
                                  float(depth_factor or 0.0), float(bf or 0.0), kd.data_ptr() if rgbd else None,
                                  ku.data_ptr() if rgbd else None, distorted=True)
        self.undistort_batch_device(camera, kps.data_ptr(), counts.data_ptr(), n, kd.data_ptr() if rgbd else None, float(bf or 0.0),
                                    kps_un.data_ptr(), ku.data_ptr() if rgbd else None)
        self.sync()
        out = dict(counts=counts.cpu().numpy(), kps=kps.cpu().numpy().view(KP_DTYPE).reshape(n, cap),
                   desc=desc.cpu().numpy(), kps_un=kps_un.cpu().numpy().view(KP_DTYPE).reshape(n, cap))
        if rgbd:
            out['depth'], out['uright'] = kd.cpu().numpy(), ku.cpu().numpy()
        return out

    def undistort_batch_device(self, camera, d_kps, d_counts, nframes, d_kp_depth=None, bf=0.0, d_kps_un=None, d_kp_uright=None):
        """hvo_orb_undistort_batch_device on the handle's stream: camera = (K, dist); raw device pointers (int) or None."""
        K, dist = camera
        _check(lib().hvo_orb_undistort_batch_device(self._h, C.byref(_camera(K, dist)), _vp(d_kps), _vp(d_counts), int(nframes),
                                                    _vp(d_kp_depth) if d_kp_depth else None, float(bf),
                                                    _vp(d_kps_un) if d_kps_un else None, _vp(d_kp_uright) if d_kp_uright else None))

    @staticmethod
    def stereo_uright_from_depth(keys_un, kp_depth, bf):
        """mvuRight of a distorted camera (second half of Frame::ComputeStereoFromRGBD, Frame.cc:1953-1958): keys_un = the keypoints
        after Frame::UndistortKeyPoints, kp_depth = the device's mvDepth."""
        k = np.ascontiguousarray(keys_un, KP_DTYPE)
        d = np.ascontiguousarray(kp_depth, np.float32)
        out = np.empty(len(k), np.float32)
        _check(lib().hvo_stereo_uright_from_depth(_np_ptr(k), _np_ptr(d), len(k), float(bf), _np_ptr(out)))
        return out

    # -- device-resident path (raw device pointers, e.g. torch tensor .data_ptr()) ---------------------
    def extract_batch_device(self, d_gray, nframes, d_kps, d_desc, d_counts, d_depth16=None, depth_factor=0.0, bf=0.0,
                             d_kp_depth=None, d_kp_uright=None, distorted=False):
        rg = C.byref(_RgbdParams(float(depth_factor), float(bf), int(bool(distorted)))) if d_depth16 else None
        _check(lib().hvo_orb_extract_batch_device(self._h, _vp(d_gray), nframes, _vp(d_kps), _vp(d_desc), _vp(d_counts),
                                                  _vp(d_depth16) if d_depth16 else None, rg,
                                                  _vp(d_kp_depth) if d_kp_depth else None,
                                                  _vp(d_kp_uright) if d_kp_uright else None))

    def sync(self):
        _check(lib().hvo_orb_sync(self._h))

    def timer_start(self):
        _check(lib().hvo_orb_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(lib().hvo_orb_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def set_profiling(self, on):
        _check(lib().hvo_orb_set_profiling(self._h, int(on)))

    def stage_times(self):
        ms = (C.c_float * 5)()
        _check(lib().hvo_orb_stage_times(self._h, ms))
        return dict(zip(('pyramid', 'fast', 'octree', 'blur', 'describe'), [float(v) for v in ms]))

    def last_launches(self):
        return lib().hvo_orb_last_launches(self._h)

    # -- inspection -----------------------------------------------------------------------------------
    def level_size(self, level):
        w, h = C.c_int(0), C.c_int(0)
        _check(lib().hvo_orb_level_size(self._h, level, C.byref(w), C.byref(h)))
        return w.value, h.value

    def pyramid_level(self, frame, level):
        """mvImagePyramid[level] of frame `frame` of the last call (ORBextractor.h:85)."""
        w, h = self.level_size(level)
        out = np.empty((h, w), np.uint8)
        _check(lib().hvo_orb_get_pyramid_level(self._h, frame, level, _np_ptr(out), w))
        return out

    def candidates(self, frame, level):
        """Pre-quadtree FAST keypoints of a level (unordered): int32 [n,3] = x, y (level coords), score."""
        w, h = self.level_size(level)
        cap = max(16, (w * h) // 4)
        out = np.empty((cap, 3), np.int32)
        n = C.c_int(0)
        _check(lib().hvo_orb_get_candidates(self._h, frame, level, _np_ptr(out), cap, C.byref(n)))
        return out[:min(n.value, cap)].copy()


KL_DTYPE = np.dtype([('angle', '<f4'), ('class_id', '<i4'), ('octave', '<i4'), ('pt_x', '<f4'), ('pt_y', '<f4'),
                     ('response', '<f4'), ('size', '<f4'), ('startPointX', '<f4'), ('startPointY', '<f4'),
                     ('endPointX', '<f4'), ('endPointY', '<f4'), ('sPointInOctaveX', '<f4'), ('sPointInOctaveY', '<f4'),
                     ('ePointInOctaveX', '<f4'), ('ePointInOctaveY', '<f4'), ('lineLength', '<f4'), ('numOfPixels', '<i4')])


class BinaryDescriptor:
    """Mirror of cv::line_descriptor::BinaryDescriptor::compute(image, keylines, descriptors) (LBD) as the
    reference calls it (src/LineExtractor.cpp:361-363, src/Frame.cc:1094-1096)."""

    def __init__(self, width, height, max_lines=512, max_batch=1, device=0):
        out = _vp()
        _check(lib().hvo_lbd_create(int(width), int(height), int(max_batch), int(max_lines), int(device), C.byref(out)))
        self._h, self.w, self.h, self.max_lines, self.max_batch = out, int(width), int(height), int(max_lines), int(max_batch)

    def close(self):
        if getattr(self, '_h', None):
            lib().hvo_lbd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def compute(self, image, keylines):
        """descriptors [n,32] uint8.  An empty keyline list returns an empty matrix (the reference prints
        'keypoint list is empty' and leaves the output untouched)."""
        kl = np.ascontiguousarray(keylines, KL_DTYPE)
        if image.dtype != np.uint8 or image.ndim != 2 or image.shape != (self.h, self.w):
            raise HvoError(HVO_ERR_ARG, 'image must be 8-bit single channel of the size given at construction')
        if image.strides[1] != 1:
            image = np.ascontiguousarray(image)
        desc = np.empty((len(kl), 32), np.uint8)
        _check(lib().hvo_lbd_compute(self._h, _vp(image.ctypes.data), image.strides[0], _np_ptr(kl), len(kl), _np_ptr(desc)))
        return desc

    def compute_batch(self, frames, keylines, counts, want_float=False):
        """frames [n,h,w]; keylines [n,max_lines] KL_DTYPE; counts [n] -> desc [n,max_lines,32] (+ float [n,max_lines,72])."""
        n = len(frames)
        frames = np.ascontiguousarray(frames, np.uint8)
        kl = np.ascontiguousarray(keylines, KL_DTYPE).reshape(n, self.max_lines)
        counts = np.ascontiguousarray(counts, np.int32)
        desc = np.empty((n, self.max_lines, 32), np.uint8)
        fdesc = np.empty((n, self.max_lines, 72), np.float32) if want_float else None
        _check(lib().hvo_lbd_compute_batch(self._h, _np_ptr(frames), n, _np_ptr(kl), _np_ptr(counts), _np_ptr(desc),
                                           _np_ptr(fdesc) if want_float else None))
        return (desc, fdesc) if want_float else desc

    def compute_batch_device(self, d_gray, nframes, d_keylines, d_counts, d_desc):
        _check(lib().hvo_lbd_compute_batch_device(self._h, _vp(d_gray), nframes, _vp(d_keylines), _vp(d_counts), _vp(d_desc)))

    def gradients(self, frame=0):
        dx = np.empty((self.h, self.w), np.int16)
        dy = np.empty((self.h, self.w), np.int16)
        _check(lib().hvo_lbd_get_gradients(self._h, frame, _np_ptr(dx), _np_ptr(dy)))
        return dx, dy

    def sync(self):
        _check(lib().hvo_lbd_sync(self._h))

    def timer_start(self):
        _check(lib().hvo_lbd_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(lib().hvo_lbd_timer_stop(self._h, C.byref(ms)))
        return ms.value


class _LineParams(C.Structure):
    _fields_ = [('n_octaves', C.c_int), ('scale', C.c_float), ('n_features', C.c_int), ('min_line_length', C.c_double)]


class LINEextractor:
    """Mirror of ORB_SLAM2::LINEextractor (reference include/LineExtractor.h:187-262).

        LINEextractor(numOctaves, scale, nLSDFeature, min_line_length)          LineExtractor.h:190
        __call__(image, mask) -> (keylines, descriptors, lineVec2d)             LineExtractor.h:193, .cpp:329-380

    keylines is a KL_DTYPE array (cv::line_descriptor::KeyLine POD), descriptors n x 32 uint8, lineVec2d n x 3 float64.
    """

    def __init__(self, numOctaves=1, scale=1.2, nLSDFeature=200, min_line_length=0.125, width=None, height=None, max_batch=1,
                 device=0):
        self.numOctaves, self.scale, self.nLSDFeature, self.min_line_length = int(numOctaves), float(scale), int(nLSDFeature), float(min_line_length)
        self.max_batch, self.device = int(max_batch), int(device)
        self._h = None
        self.w = self.h = None
        if width is not None:
            self._create(int(width), int(height))

    def _create(self, w, h):
        self.close()
        prm = _LineParams(self.numOctaves, self.scale, self.nLSDFeature, self.min_line_length)
        out = _vp()
        _check(lib().hvo_line_create(C.byref(prm), w, h, self.max_batch, self.device, C.byref(out)))
        self._h, self.w, self.h = out, w, h
        self.max_lines = lib().hvo_line_max_lines(out)
        self.segment_capacity = lib().hvo_line_segment_capacity(out)

    def close(self):
        if getattr(self, '_h', None):
            lib().hvo_line_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # getters of LineExtractor.h:239-261
    def GetLevels(self):
        return self.numOctaves

    def GetScaleFactor(self):
        return self.scale

    def __call__(self, image, mask=None):
        if image is None or image.size == 0:  # LineExtractor.cpp:331-332
            return np.empty(0, KL_DTYPE), np.empty((0, 32), np.uint8), np.empty((0, 3), np.float64)
        if image.dtype != np.uint8 or image.ndim != 2:
            raise HvoError(HVO_ERR_ARG, 'image must be 8-bit single channel (assert(image.type() == CV_8UC1))')
        if image.strides[1] != 1:
            image = np.ascontiguousarray(image)
        if self._h is None or (self.h, self.w) != image.shape:
            self._create(image.shape[1], image.shape[0])
        kl = np.empty(self.max_lines, KL_DTYPE)
        desc = np.empty((self.max_lines, 32), np.uint8)
        lv = np.empty((self.max_lines, 3), np.float64)
        n = C.c_int(0)
        _check(lib().hvo_line_extract(self._h, _vp(image.ctypes.data), image.strides[0], _np_ptr(kl), _np_ptr(desc), _np_ptr(lv),
                                      self.max_lines, C.byref(n)))
        return kl[:n.value].copy(), desc[:n.value].copy(), lv[:n.value].copy()

    def set_culling(self, enable):
        """True: every extraction also runs Frame::cullingLine (src/Frame.cc:939, 952-1116) as Frame::ExtractLSD does."""
        if self._h is None:
            raise HvoError(HVO_ERR_ARG, 'create the extractor with width/height first')
        _check(lib().hvo_line_set_culling(self._h, int(bool(enable))))

    def cullingLine(self, image, keylines, lineVec2d):
        """Frame::cullingLine(imGray, 5, 2.5, 15, 30): (keylines, descriptors, lineVec2d) after merging."""
        image = np.ascontiguousarray(image, np.uint8)
        if self._h is None or (self.h, self.w) != image.shape:
            self._create(image.shape[1], image.shape[0])
        n = len(keylines)
        kl = np.zeros(self.max_lines, KL_DTYPE); kl[:n] = keylines
        lv = np.zeros((self.max_lines, 3), np.float64); lv[:n] = lineVec2d
        desc = np.empty((self.max_lines, 32), np.uint8)
        m = C.c_int(0)
        _check(lib().hvo_line_cull(self._h, _vp(image.ctypes.data), image.strides[0], _np_ptr(kl), _np_ptr(lv), n, _np_ptr(desc), C.byref(m)))
        return kl[:m.value].copy(), desc[:m.value].copy(), lv[:m.value].copy()

    def extract_batch(self, frames, out=None):
        """frames [n,h,w] uint8 -> dict(counts [n], keylines [n,max_lines], desc [n,max_lines,32], linevec [n,max_lines,3])"""
        frames = np.ascontiguousarray(frames, np.uint8)
        n = len(frames)
        if out is None:
            out = dict(counts=np.zeros(n, np.int32), keylines=np.empty((n, self.max_lines), KL_DTYPE),
                       desc=np.empty((n, self.max_lines, 32), np.uint8), linevec=np.empty((n, self.max_lines, 3), np.float64))
        _check(lib().hvo_line_extract_batch(self._h, _np_ptr(frames), n, _np_ptr(out['keylines']), _np_ptr(out['desc']),
                                            _np_ptr(out['linevec']), _np_ptr(out['counts'])))
        return out

    def extract_batch_device(self, d_gray, nframes, d_keylines, d_desc, d_linevec, d_counts):
        _check(lib().hvo_line_extract_batch_device(self._h, _vp(d_gray), nframes, _vp(d_keylines), _vp(d_desc), _vp(d_linevec), _vp(d_counts)))

    def detect_segments(self, frames):
        """cv::LineSegmentDetector::detect on each frame: list of [k,4] float32 arrays (x1,y1,x2,y2)."""
        frames = np.ascontiguousarray(frames, np.uint8)
        if frames.ndim == 2:
            frames = frames[None]
        n = len(frames)
        cap = self.segment_capacity
        seg = np.empty((n, cap, 4), np.float32)
        counts = np.zeros(n, np.int32)
        _check(lib().hvo_line_detect_batch(self._h, _np_ptr(frames), n, _np_ptr(seg), cap, _np_ptr(counts)))
        return [seg[i, :counts[i]].copy() for i in range(n)]

    def scaled_image(self, frame=0):
        sw, sh = C.c_int(0), C.c_int(0)
        _check(lib().hvo_line_scaled_size(self._h, C.byref(sw), C.byref(sh)))
        out = np.empty((sh.value, sw.value), np.uint8)
        _check(lib().hvo_line_get_scaled(self._h, frame, _np_ptr(out)))
        return out

    def seed_order(self, frame=0):
        sw, sh = C.c_int(0), C.c_int(0)
        _check(lib().hvo_line_scaled_size(self._h, C.byref(sw), C.byref(sh)))
        out = np.empty(sw.value * sh.value, np.uint32)
        n = C.c_int(0)
        _check(lib().hvo_line_get_seed_order(self._h, frame, _np_ptr(out), len(out), C.byref(n)))
        return out[:n.value].copy()

    def set_profiling(self, on):
        _check(lib().hvo_line_set_profiling(self._h, int(bool(on))))

    def stage_times(self):
        ms = (C.c_float * 4)()
        _check(lib().hvo_line_stage_times(self._h, ms))
        return dict(prep=ms[0], order=ms[1], grow=ms[2], keylines_lbd=ms[3])

    def last_launches(self):
        return lib().hvo_line_last_launches(self._h)

    def sync(self):
        _check(lib().hvo_line_sync(self._h))

    def timer_start(self):
        _check(lib().hvo_line_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(lib().hvo_line_timer_stop(self._h, C.byref(ms)))
        return ms.value


class _PlaneParams(C.Structure):
    _fields_ = [('fx', C.c_float), ('fy', C.c_float), ('cx', C.c_float), ('cy', C.c_float), ('depth_factor', C.c_float)]


class PlaneDetection:
    """Mirror of the reference's PlaneDetection (include/PlaneExtractor.h:36-56): readDepthImage(depth16U, K, factor)
    followed by runPlaneDetection(H, W); results as plane_num_, plane normals/centers, plane_vertices_, membership."""
    MAX_PLANES = 64

    def __init__(self, width, height, max_batch=1, device=0):
        self.w, self.h, self.max_batch, self.device = int(width), int(height), int(max_batch), int(device)
        self._h = None
        self._depth = None
        self.plane_num_ = 0
        self.plane_vertices_ = []

    def close(self):
        if getattr(self, '_h', None):
            lib().hvo_plane_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def readDepthImage(self, depthImg, K, kScaleFactor):
        """K: 3x3 (only fx, fy, cx, cy are read, as float32).  Returns False on a non-16U image, as the reference."""
        if depthImg is None or depthImg.size == 0 or depthImg.dtype != np.uint16:
            print('WARNING: cannot read depth image. No such a file, or the image format is not 16UC1')
            return False
        K = np.asarray(K, np.float32)
        params = _PlaneParams(float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2]), float(np.float32(kScaleFactor)))
        key = (params.fx, params.fy, params.cx, params.cy, params.depth_factor)
        if self._h is None or getattr(self, '_key', None) != key:
            self.close()
            out = _vp()
            _check(lib().hvo_plane_create(C.byref(params), self.w, self.h, self.max_batch, self.device, C.byref(out)))
            self._h, self._key = out, key
        self._depth = np.ascontiguousarray(depthImg)
        return True

    def runPlaneDetection(self, kDepthHeight=None, kDepthWidth=None):
        assert self._depth is not None and self._depth.shape == (self.h, self.w)
        n = np.zeros(1, np.int32)
        planes = np.zeros((self.MAX_PLANES, 7), np.float64)
        self.membership = np.empty(self.h * self.w, np.int32)
        _check(lib().hvo_plane_detect(self._h, _np_ptr(self._depth), _np_ptr(n), _np_ptr(planes), self.MAX_PLANES, _np_ptr(self.membership)))
        self.plane_num_ = int(n[0])
        self.normals = planes[:self.plane_num_, 0:3].copy()
        self.centers = planes[:self.plane_num_, 3:6].copy()
        self.supports = planes[:self.plane_num_, 6].astype(np.int64)
        self.plane_vertices_ = [np.nonzero(self.membership == i)[0] for i in range(self.plane_num_)]
        return self.plane_num_

    def detect_batch(self, depths):
        """depths [n,h,w] uint16 -> (n_planes [n], planes [n,MAX,7], membership [n,h*w])"""
        depths = np.ascontiguousarray(depths, np.uint16)
        nf = len(depths)
        n = np.zeros(nf, np.int32)
        planes = np.zeros((nf, self.MAX_PLANES, 7), np.float64)
        mem = np.empty((nf, self.h * self.w), np.int32)
        _check(lib().hvo_plane_detect_batch(self._h, _np_ptr(depths), nf, _np_ptr(n), _np_ptr(planes), self.MAX_PLANES, _np_ptr(mem)))
        return n, planes, mem

    def blocks(self, frame=0):
        """initial graph nodes of the last call: [Nh*Nw, 9] = queued, N, center(3), normal(3), mse"""
        out = np.empty(((self.h // 10) * (self.w // 10), 9), np.float64)
        _check(lib().hvo_plane_get_blocks(self._h, frame, _np_ptr(out)))
        return out

    def detect_batch_device(self, d_depth, nframes, d_nplanes, d_planes7, max_planes, d_membership):
        _check(lib().hvo_plane_detect_batch_device(self._h, _vp(d_depth), nframes, _vp(d_nplanes), _vp(d_planes7), max_planes, _vp(d_membership)))

    def last_launches(self):
        return lib().hvo_plane_last_launches(self._h)

    def phase_cycles(self, frame=0):
        out = np.zeros(4, np.int64)
        _check(lib().hvo_plane_get_phase_cycles(self._h, frame, _np_ptr(out)))
        return dict(cluster=int(out[0]), seeds=int(out[1]), flood=int(out[2]), merge_relabel=int(out[3]))

    def blocks_device(self, d_depth, nframes):
        _check(lib().hvo_plane_blocks_device(self._h, _vp(d_depth), nframes))

    def sync(self):
        _check(lib().hvo_plane_sync(self._h))

    def timer_start(self):
        _check(lib().hvo_plane_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(lib().hvo_plane_timer_stop(self._h, C.byref(ms)))
        return ms.value


class _NormalsParams(C.Structure):
    _fields_ = [('fx', C.c_float), ('fy', C.c_float), ('cx', C.c_float), ('cy', C.c_float), ('depth_factor', C.c_float),
                ('max_depth_change_factor', C.c_float), ('normal_smoothing_size', C.c_float)]


class SurfaceNormals:
    """The surface-normal block of Frame::ComputePlanes (reference src/Frame.cc:2155-2212): returns the
    std::vector<SurfaceNormal> as an [n,8] float32 array = normal.xyz, cameraPosition.xyz, FramePosition.xy."""

    def __init__(self, width, height, fx, fy, cx, cy, depth_factor, max_depth_change=0.05, smoothing=10.0, max_batch=1, device=0):
        prm = _NormalsParams(fx, fy, cx, cy, float(np.float32(depth_factor)), max_depth_change, smoothing)
        out = _vp()
        _check(lib().hvo_normals_create(C.byref(prm), int(width), int(height), int(max_batch), int(device), C.byref(out)))
        self._h, self.w, self.h = out, int(width), int(height)
        self.count = lib().hvo_normals_count(self._h)

    def close(self):
        if getattr(self, '_h', None):
            lib().hvo_normals_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def compute(self, depth16):
        d = np.ascontiguousarray(depth16, np.uint16)
        batched = d.ndim == 3
        d3 = d if batched else d[None]
        out = np.empty((len(d3), self.count, 8), np.float32)
        _check(lib().hvo_normals_compute_batch(self._h, _np_ptr(d3), len(d3), _np_ptr(out)))
        return out if batched else out[0]

    def compute_device(self, d_depth, nframes, d_out):
        _check(lib().hvo_normals_compute_batch_device(self._h, _vp(d_depth), nframes, _vp(d_out)))

    def distance_map(self, frame=0):
        cw, ch = -(-self.w // 3), -(-self.h // 3)
        out = np.empty((ch, cw), np.float32)
        _check(lib().hvo_normals_get_distance_map(self._h, frame, _np_ptr(out)))
        return out

    def sync(self):
        _check(lib().hvo_normals_sync(self._h))

    def timer_start(self):
        _check(lib().hvo_normals_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(lib().hvo_normals_timer_stop(self._h, C.byref(ms)))
        return ms.value


class Manhattan:
    """The normal-extraction half of ORB_SLAM2::Manhattan (reference src/Manhattan.cpp): computeNormalsLPVO on the GPU.
    Constructed from K like the reference (Manhattan.cpp:8-19); depth is the raw 16-bit image and depth_factor."""

    def __init__(self, K, width, height, depth_factor, max_batch=1, device=0):
        K = np.asarray(K, np.float32)
        prm = _PlaneParams(float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2]), float(np.float32(depth_factor)))
        out = _vp()
        _check(lib().hvo_lpvo_create(C.byref(prm), int(width), int(height), int(max_batch), int(device), C.byref(out)))
        self._h, self.w, self.h = out, int(width), int(height)
        self.capacity = lib().hvo_lpvo_capacity(self._h)

    def close(self):
        if getattr(self, '_h', None):
            lib().hvo_lpvo_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def computeNormalsLPVO_batch(self, depth16):
        """[n,h,w] uint16 -> list of (pt_normals [m,3] float64, depth_normals [m] float32, pixels (u, v) [m,2] int32)."""
        d = np.ascontiguousarray(depth16, np.uint16)
        n, c = len(d), self.capacity
        nrm = np.empty((n, c, 3), np.float64); dep = np.empty((n, c), np.float32); pix = np.empty((n, c, 2), np.int32)
        cnt = np.empty(n, np.int32)
        _check(lib().hvo_lpvo_compute_batch(self._h, _np_ptr(d), n, _np_ptr(nrm), _np_ptr(dep), _np_ptr(pix), _np_ptr(cnt)))
        return [(nrm[f, :cnt[f]], dep[f, :cnt[f]], pix[f, :cnt[f]]) for f in range(n)]

    def computeNormalsLPVO(self, depth16):
        return self.computeNormalsLPVO_batch(np.asarray(depth16)[None])[0]

    def compute_device(self, d_depth, nframes, d_normals3, d_depth_out, d_pix2, d_counts):
        _check(lib().hvo_lpvo_compute_batch_device(self._h, _vp(d_depth), nframes, _vp(d_normals3), _vp(d_depth_out), _vp(d_pix2), _vp(d_counts)))

    def sync(self):
        _check(lib().hvo_lpvo_sync(self._h))

    def timer_start(self):
        _check(lib().hvo_lpvo_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(lib().hvo_lpvo_timer_stop(self._h, C.byref(ms)))
        return ms.value


class BFMatcherHamming:
    """cv::BFMatcher(NORM_HAMMING, crossCheck=false).knnMatch(k=2) on the GPU (hvo_match_knn2)."""

    def __init__(self, device=0):
        out = _vp()
        _check(lib().hvo_matcher_create(int(device), C.byref(out)))
        self._h = out

    def close(self):
        if getattr(self, '_h', None):
            lib().hvo_matcher_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def knnMatch2(self, desc1, desc2):
        """(idx [n1,2] int32, dist [n1,2] int32); ties resolve to the lower train index; -1 where desc2 has < 2 rows."""
        q = np.ascontiguousarray(desc1, np.uint8).reshape(-1, 32)
        t = np.ascontiguousarray(desc2, np.uint8).reshape(-1, 32)
        idx = np.empty((len(q), 2), np.int32)
        dist = np.empty((len(q), 2), np.int32)
        _check(lib().hvo_match_knn2(self._h, _np_ptr(q), len(q), _np_ptr(t), len(t), _np_ptr(idx), _np_ptr(dist)))
        return idx, dist

    def lines_epipolar(self, ldesc1, kls1, ldesc2, kls2, kls2func, F, TH, nnratio):
        """LSDmatcher::FrameBFMatchNew (src/LSDmatcher.cpp:968-1031): knn-2 + the epipolar overlap test of the nearest neighbour."""
        d1 = np.ascontiguousarray(ldesc1, np.uint8).reshape(-1, 32); d2 = np.ascontiguousarray(ldesc2, np.uint8).reshape(-1, 32)
        k1 = np.ascontiguousarray(kls1, KL_DTYPE); k2 = np.ascontiguousarray(kls2, KL_DTYPE)
        f2 = np.ascontiguousarray(kls2func, np.float64).reshape(-1, 3); Fm = np.ascontiguousarray(F, np.float32).reshape(9)
        out = np.full(max(len(d1), 1), -1, np.int32)
        _check(lib().hvo_match_lines_epipolar(self._h, _np_ptr(d1), _np_ptr(k1), len(d1), _np_ptr(d2), _np_ptr(k2), _np_ptr(f2), len(d2), _np_ptr(Fm),
                                              float(TH), float(nnratio), _np_ptr(out)))
        return out[:len(d1)]

    def distinctive(self, desc, offsets):
        """MapPoint / MapLine::ComputeDistinctiveDescriptors for a batch of map elements: group g = desc[offsets[g]:offsets[g+1]]
        (the descriptors of its observations).  Returns (best index inside each group or -1, its median distance)."""
        d = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        off = np.ascontiguousarray(offsets, np.int32)
        n = len(off) - 1
        bi = np.full(max(n, 1), -1, np.int32); bm = np.full(max(n, 1), -1, np.int32)
        _check(lib().hvo_match_distinctive(self._h, _np_ptr(d), _np_ptr(off), n, _np_ptr(bi), _np_ptr(bm)))
        return bi[:n], bm[:n]

    def knn2_device(self, d_q, nq, d_t, nt, d_idx, d_dist):
        _check(lib().hvo_match_knn2_device(self._h, _vp(d_q), nq, _vp(d_t), nt, _vp(d_idx), _vp(d_dist)))

    def sync(self):
        _check(lib().hvo_matcher_sync(self._h))

    def timer_start(self):
        _check(lib().hvo_matcher_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(lib().hvo_matcher_timer_stop(self._h, C.byref(ms)))
        return ms.value


LPROJ_QUERY_DTYPE = np.dtype([('x1', '<f4'), ('y1', '<f4'), ('x2', '<f4'), ('y2', '<f4'), ('r', '<f4'), ('cos_th', '<f4'), ('dir', '<f8', (3,)),
                              ('length', '<f4'), ('claims', '<i4'), ('reserved', '<i4', (2,))])
assert LPROJ_QUERY_DTYPE.itemsize == 64


class LineProjectionMatcher:
    """Device side of the windowed line matchers: the line grid (Frame::AssignFeaturesToGridForLine, src/Frame.cc:849-872),
    Frame::GetFeaturesInAreaForLine (:1557-1631) and the greedy searches of LSDmatcher::SearchByProjection
    (src/LSDmatcher.cpp:561-664, 709-801).  One frame at a time."""

    def __init__(self, device=0):
        out = _vp()
        _check(lib().hvo_lproj_create(int(device), C.byref(out)))
        self._h = out
        self.n = 0

    def close(self):
        if getattr(self, '_h', None):
            lib().hvo_lproj_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_frame(self, keylines_un, line_functions, desc, lines3d, min_x, min_y, max_x, max_y):
        kl = np.ascontiguousarray(keylines_un, KL_DTYPE)
        fn = np.ascontiguousarray(line_functions, np.float64).reshape(-1, 3)
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        l3 = None if lines3d is None else np.ascontiguousarray(lines3d, np.float64).reshape(-1, 6)
        self.n = len(kl)
        _check(lib().hvo_lproj_set_frame(self._h, _np_ptr(kl), _np_ptr(fn), _np_ptr(desc), _np_ptr(l3) if l3 is not None else None, self.n,
                                         float(min_x), float(min_y), float(max_x), float(max_y)))

    def grid(self):
        """(cell_count [64*48], cell_items): cell ix*48+iy lists mGridForLine[ix][iy]."""
        cnt = np.empty(GRID_COLS * GRID_ROWS, np.int32)
        n = C.c_int(0)
        _check(lib().hvo_lproj_get_grid(self._h, _np_ptr(cnt), None, 0, C.byref(n)))
        items = np.empty(max(n.value, 1), np.int32)
        _check(lib().hvo_lproj_get_grid(self._h, _np_ptr(cnt), _np_ptr(items), len(items), C.byref(n)))
        return cnt, items[:n.value].copy()

    def GetFeaturesInAreaForLine(self, x1, y1, x2, y2, r, minLevel=-1, maxLevel=-1, TH=0.998):
        out = np.empty(max(self.n, 1), np.int32)
        n = C.c_int(0)
        _check(lib().hvo_lproj_features_in_area(self._h, float(x1), float(y1), float(x2), float(y2), float(r), float(np.float32(TH)),
                                                _np_ptr(out), len(out), C.byref(n)))
        return out[:n.value].copy()

    def search(self, queries, qdesc, claimed=None, mode=0, nnratio=0.95):
        q = np.ascontiguousarray(queries, LPROJ_QUERY_DTYPE)
        qd = np.ascontiguousarray(qdesc, np.uint8).reshape(-1, 32)
        cl = None if claimed is None else np.ascontiguousarray(claimed, np.uint8)
        idx = np.full(max(len(q), 1), -1, np.int32)
        dist = np.full(max(len(q), 1), 256, np.int32)
        nm = C.c_int(0)
        _check(lib().hvo_lproj_search(self._h, _np_ptr(q), _np_ptr(qd), len(q), _np_ptr(cl) if cl is not None else None, int(mode),
                                      float(np.float32(nnratio)), _np_ptr(idx), _np_ptr(dist), C.byref(nm)))
        return idx[:len(q)], dist[:len(q)], nm.value

    def frustum_lines(self, cam, lines, viewing_cos_limit=0.5):
        """Frame::isInFrustum(MapLine*, viewingCosLimit) (src/Frame.cc:1438-1499) for a batch: lines MAP_LINE_DTYPE."""
        cam = np.ascontiguousarray(cam, FRUSTUM_CAM_DTYPE); ml = np.ascontiguousarray(lines, MAP_LINE_DTYPE)
        out = np.zeros(max(len(ml), 1), TRACK_LINE_DTYPE)
        _check(lib().hvo_lproj_frustum_lines(self._h, _np_ptr(cam), _np_ptr(ml), len(ml), float(viewing_cos_limit), _np_ptr(out)))
        return out[:len(ml)]

    def search_local_map(self, cam, lines, ldesc, skip=None, claims=None, claimed=None, viewing_cos_limit=0.5, th=1.0, nnratio=0.95):
        """isInFrustum over the local map lines + LSDmatcher::SearchByProjection(F, vpMapLines, eval_orient, th) in one call."""
        cam = np.ascontiguousarray(cam, FRUSTUM_CAM_DTYPE); ml = np.ascontiguousarray(lines, MAP_LINE_DTYPE)
        n = len(ml)
        ld = np.ascontiguousarray(ldesc, np.uint8).reshape(-1, 32)
        opt = lambda a: None if a is None else np.ascontiguousarray(a, np.uint8)
        sk, cl, cd = opt(skip), opt(claims), opt(claimed)
        track = np.zeros(max(n, 1), TRACK_LINE_DTYPE); idx = np.full(max(n, 1), -1, np.int32); dist = np.full(max(n, 1), 256, np.int32)
        niv, nm = C.c_int(0), C.c_int(0)
        p = lambda a: _np_ptr(a) if a is not None else None
        _check(lib().hvo_lproj_search_local_map(self._h, _np_ptr(cam), _np_ptr(ml), _np_ptr(ld), p(sk), p(cl), n, float(viewing_cos_limit), float(th),
                                                p(cd), float(nnratio), _np_ptr(track), _np_ptr(idx), _np_ptr(dist), C.byref(niv), C.byref(nm)))
        return track[:n], idx[:n], dist[:n], niv.value, nm.value

    def rounds(self):
        return lib().hvo_lproj_last_rounds(self._h)


class LSDmatcher:
    """Mirror of ORB_SLAM2::LSDmatcher (reference include/LSDmatcher.h:23-60): match / matchNNR (src/LSDmatcher.cpp:803-863),
    FrameBFMatch + lineDescriptorMAD (:942-966, :1110-1135), SearchDouble, SearchByDescriptor, the two SearchByProjection
    (:561-664, :709-801) and DescriptorDistance (:1137-1153).  Distances and the windowed searches run on the GPU; the
    ratio / MAD filters are the reference's float arithmetic on the host.  Frames and map lines are plain arrays:

        F   = dict(keylines_un KL_DTYPE [NL], line_functions [NL,3], ldesc [NL,32], lines3d [NL,6] (mvLines3D first, second),
                   bounds (minX, minY, maxX, maxY), mapline [NL] int (index of the map line held, -1 none),
                   claimed [NL] bool (holds one with observations))
        MLs = dict(proj_x1, proj_y1, proj_x2, proj_y2, view_cos, in_view, bad, has_obs, world_vector [M,3], desc [M,32])
    """
    TH_HIGH, TH_LOW = 80, 50

    def __init__(self, nnratio=0.95, checkOri=True, device=0):
        self.mfNNratio = np.float32(nnratio)
        self.mbCheckOrientation = bool(checkOri)
        self._bf = BFMatcherHamming(device)
        self._device = device
        self._lpm = None

    def close(self):
        self._bf.close()
        if self._lpm is not None:
            self._lpm.close()

    def _line_matcher(self, F, need3d):
        if self._lpm is None:
            self._lpm = LineProjectionMatcher(self._device)
        b = F['bounds']
        self._lpm.set_frame(F['keylines_un'], F['line_functions'], F['ldesc'], F.get('lines3d') if need3d else None, b[0], b[1], b[2], b[3])
        return self._lpm

    @staticmethod
    def RadiusByViewingCos(viewCos):  # LSDmatcher.cpp:1436-1442
        return np.where(np.asarray(viewCos, np.float32) > np.float32(0.998), np.float32(5.0), np.float32(8.0))

    @staticmethod
    def _apply(F, sel, idx, has_obs):
        for k, i in zip(sel, idx):  # F.mvpMapLines[bestIdx] = pML, in query order
            if i >= 0:
                F['mapline'][i] = k
                F['claimed'][i] = bool(has_obs[k])

    def SearchByProjection(self, F, MLs, eval_orient=True, th=1.0):
        """LSDmatcher::SearchByProjection(Frame&, const vector<MapLine*>&, eval_orient, th) (LSDmatcher.cpp:709-801).  Updates
        F['mapline'] / F['claimed'] in place, returns (nmatches, match [M] frame line index or -1)."""
        M = len(MLs['proj_x1'])
        sel = np.nonzero(np.asarray(MLs['in_view'], bool) & ~np.asarray(MLs['bad'], bool))[0]
        r = self.RadiusByViewingCos(np.asarray(MLs['view_cos'])[sel]).astype(np.float32)
        if th != 1.0:
            r = (r * np.float32(th)).astype(np.float32)
        q = np.zeros(len(sel), LPROJ_QUERY_DTYPE)
        for a, b in (('x1', 'proj_x1'), ('y1', 'proj_y1'), ('x2', 'proj_x2'), ('y2', 'proj_y2')):
            q[a] = np.asarray(MLs[b], np.float32)[sel]
        q['r'] = r
        q['cos_th'] = np.float32(0.998)                       # default TH of GetFeaturesInAreaForLine (Frame.h:131)
        q['dir'] = np.asarray(MLs['world_vector'], np.float64)[sel]
        q['claims'] = np.asarray(MLs['has_obs'], bool)[sel]
        has_obs = np.asarray(MLs['has_obs'], bool)
        match = np.full(M, -1, np.int32)
        if len(sel) == 0:
            return 0, match
        idx, _, nm = self._line_matcher(F, True).search(q, np.asarray(MLs['desc'], np.uint8)[sel], F.get('claimed'), 0, self.mfNNratio)
        match[sel] = idx
        self._apply(F, sel, idx, has_obs)
        return nm, match

    def SearchByProjectionLast(self, Cur, last, th):
        """Matching part of LSDmatcher::SearchByProjection(CurrentFrame, LastFrame, th) (LSDmatcher.cpp:561-664).  `last` holds,
        for every last-frame line with a usable map line (not an outlier, in the current frustum), its projection into the
        current frame and its keyline: dict(proj_x1, proj_y1, proj_x2, proj_y2, keylines KL_DTYPE [M], has_obs, desc [M,32]).
        Updates Cur['mapline'] / Cur['claimed'], returns (nmatches, match [M])."""
        M = len(last['proj_x1'])
        kl = np.asarray(last['keylines'], KL_DTYPE)
        q = np.zeros(M, LPROJ_QUERY_DTYPE)
        for a, b in (('x1', 'proj_x1'), ('y1', 'proj_y1'), ('x2', 'proj_x2'), ('y2', 'proj_y2')):
            q[a] = np.asarray(last[b], np.float32)
        q['r'] = np.float32(th)
        q['cos_th'] = np.float32(0.96)
        q['dir'][:, 0] = (kl['ePointInOctaveX'] - kl['sPointInOctaveX']).astype(np.float32)
        q['dir'][:, 1] = (kl['ePointInOctaveY'] - kl['sPointInOctaveY']).astype(np.float32)
        q['length'] = kl['lineLength']
        has_obs = np.asarray(last['has_obs'], bool)
        q['claims'] = has_obs
        if M == 0:
            return 0, np.full(0, -1, np.int32)
        idx, _, nm = self._line_matcher(Cur, False).search(q, np.asarray(last['desc'], np.uint8), Cur.get('claimed'), 1, self.mfNNratio)
        self._apply(Cur, np.arange(M), idx, has_obs)
        return nm, idx.copy()

    @staticmethod
    def DescriptorDistance(a, b):
        a = np.ascontiguousarray(a, np.uint8)
        b = np.ascontiguousarray(b, np.uint8)
        return int(lib().hvo_hamming_distance(_np_ptr(a), _np_ptr(b)))

    def matchNNR(self, desc1, desc2, nnr):
        """returns (number of matches, matches_12) with matches_12[i] = train index or -1."""
        if len(desc2) < 2:
            raise HvoError(HVO_ERR_ARG, 'matchNNR needs at least two train descriptors (the reference reads matches_[idx][1])')
        idx, dist = self._bf.knnMatch2(desc1, desc2)
        ok = dist[:, 0].astype(np.float32) < dist[:, 1].astype(np.float32) * np.float32(nnr)
        m = np.where(ok, idx[:, 0], -1).astype(np.int32)
        return int(ok.sum()), m

    def match(self, desc1, desc2, nnr):
        return self.matchNNR(desc1, desc2, nnr)  # the two-way branch is disabled in the reference (`if (false)`)

    def FrameBFMatch(self, ldesc1, ldesc2, TH):
        n = len(ldesc1)
        out = np.full(n, -1, np.int32)
        if n == 0:
            return out
        idx, dist = self._bf.knnMatch2(ldesc1, ldesc2)
        d0, d1 = dist[:, 0].astype(np.float32), dist[:, 1].astype(np.float32)
        gap = d1 - d0
        med = np.float64(np.sort(gap)[::-1][n // 2])
        dev = np.abs((gap.astype(np.float64) - med).astype(np.float32))
        nn12_th = 1.4826 * np.float64(np.sort(dev)[n // 2]) * 0.5
        ok = (gap.astype(np.float64) > nn12_th) & (d0 < np.float32(TH)) & (d0 < self.mfNNratio * d1)
        out[ok] = idx[ok, 0]
        return out

    def FrameBFMatchNew(self, ldesc1, ldesc2, kls1, kls2, kls2func, F, TH):
        """LSDmatcher::FrameBFMatchNew(ldesc1, ldesc2, LineMatches, kls1, kls2, kls2func, F, TH) (src/LSDmatcher.cpp:968-1031).  Returns LineMatches."""
        return self._bf.lines_epipolar(ldesc1, kls1, ldesc2, kls2, kls2func, F, TH, self.mfNNratio)

    def SearchLocalLines(self, F, cam, lines, ldesc, skip, has_obs, th=1.0, viewing_cos_limit=0.5):
        """The device work of Tracking::SearchLocalLines (src/Tracking.cc:3315-3348): Frame::isInFrustum over the local map lines and
        LSDmatcher::SearchByProjection(F, vpMapLines, eval_orient, th) in one call.  Updates F['mapline'] / F['claimed']; returns
        (track, nmatches, match [M])."""
        lpm = self._line_matcher(F, True)
        track, idx, dist, niv, nm = lpm.search_local_map(cam, lines, ldesc, skip, has_obs, F.get('claimed'), viewing_cos_limit, th, self.mfNNratio)
        self._apply(F, np.arange(len(idx)), idx, has_obs)
        return track, nm, idx

    def SearchDouble(self, ldesc1, ldesc2):
        """LSDmatcher::SearchDouble(InitialFrame, CurrentFrame, LineMatches) (src/LSDmatcher.cpp:903-940): FrameBFMatch in both
        directions (the reference runs them on two threads), kept where they agree.  Returns (nmatches, LineMatches)."""
        if len(ldesc1) == 0 or len(ldesc2) == 0:
            return 0, np.full(len(ldesc1), -1, np.int32)
        m12 = self.FrameBFMatch(ldesc1, ldesc2, self.TH_LOW)
        m21 = self.FrameBFMatch(ldesc2, ldesc1, self.TH_LOW)
        ok = m12 >= 0
        ok[ok] = m21[m12[ok]] == np.nonzero(ok)[0]
        out = np.where(ok, m12, -1).astype(np.int32)
        return int(ok.sum()), out

    def SearchDoubleKF(self, ldesc_kf, has_mapline, ldesc_cur):
        """LSDmatcher::SearchDouble(KeyFrame *KF, Frame &CurrentFrame) (src/LSDmatcher.cpp:865-901): FrameBFMatch in both directions; a
        current-frame line i whose match j agrees (tempMatches1[j] == i) receives the key frame's MapLine j when it holds one.
        Returns (nmatches, match [len(ldesc_cur)] = key-frame line or -1)."""
        out = np.full(len(ldesc_cur), -1, np.int32)
        if len(ldesc_kf) == 0 or len(ldesc_cur) == 0:
            return 0, out
        m12 = self.FrameBFMatch(ldesc_kf, ldesc_cur, self.TH_LOW)
        m21 = self.FrameBFMatch(ldesc_cur, ldesc_kf, self.TH_LOW)
        has = np.asarray(has_mapline, bool)
        for i, j in enumerate(m21):
            if j >= 0 and m12[j] == i and has[j]:
                out[i] = j
        return int((out >= 0).sum()), out

    def SearchForTriangulation(self, ldesc1, has_mapline1, ldesc2, has_mapline2, th=None, is_double=True):
        """LSDmatcher::SearchForTriangulation (src/LSDmatcher.cpp:1155-1231): FrameBFMatch both ways; th = TH_LOW with the cross-check always on
        is the vector<pair> overload (:1155-1193), th = TH_HIGH with is_double the vector<int> overload (:1195-1231); pairs where either line
        already holds a MapLine are dropped.  Returns (nmatches, match [len(ldesc1)] = line of pKF2 or -1)."""
        th = self.TH_LOW if th is None else th
        out = np.full(len(ldesc1), -1, np.int32)
        if len(ldesc1) == 0 or len(ldesc2) == 0:
            return 0, out
        m12 = self.FrameBFMatch(ldesc1, ldesc2, th)
        m21 = self.FrameBFMatch(ldesc2, ldesc1, th)
        h1, h2 = np.asarray(has_mapline1, bool), np.asarray(has_mapline2, bool)
        for i, j in enumerate(m12):
            if j >= 0 and (not is_double or m21[j] == i) and not (h1[i] or h2[j]):
                out[i] = j
        return int((out >= 0).sum()), out

    def SearchByDescriptor(self, ldesc_kf, ldesc_cur, has_mapline=None):
        """Matching part of LSDmatcher::SearchByDescriptor(pKF, currentF, vpMapLineMatches) (src/LSDmatcher.cpp:522-559): knn-2 of
        the key frame's descriptors in the current frame, accepted when d0 / d1 < 1 / 1.5 AND the key-frame line holds a MapLine
        (`if(mapLine)`, :549-553; has_mapline [len(ldesc_kf)] bool, default: all do).  Returns (nmatches, match [len(ldesc_cur)]):
        key-frame line index per current-frame line or -1; a later accepted query overwrites an earlier one on the same
        current-frame line, a query without a MapLine never does, and nmatches counts every accepted query, as in the reference."""
        out = np.full(len(ldesc_cur), -1, np.int32)
        if len(ldesc_kf) == 0 or len(ldesc_cur) < 2:
            return 0, out
        has = np.ones(len(ldesc_kf), bool) if has_mapline is None else np.asarray(has_mapline, bool)
        idx, dist = self._bf.knnMatch2(ldesc_kf, ldesc_cur)
        with np.errstate(divide='ignore', invalid='ignore'):
            ratio = (dist[:, 0].astype(np.float32) / dist[:, 1].astype(np.float32)).astype(np.float64)
        nmatches = 0
        for q in np.nonzero(ratio < np.float32(1.0) / np.float32(1.5))[0]:
            if has[q]:
                out[idx[q, 0]] = q
                nmatches += 1
        return nmatches, out


# ---- Frame-level front-end ----------------------------------------------------------------------------------------
STAGE_ORB, STAGE_LINES, STAGE_PLANES, STAGE_NORMALS, STAGE_ALL = 1, 2, 4, 8, 15


PROJ_QUERY_DTYPE = np.dtype([('u', '<f4'), ('v', '<f4'), ('r', '<f4'), ('min_level', '<i4'), ('max_level', '<i4'), ('ur', '<f4'),
                             ('claims', '<i4'), ('reserved', '<i4')])
assert PROJ_QUERY_DTYPE.itemsize == 32
GRID_COLS, GRID_ROWS = 64, 48


def _vocabulary_args(voc):
    """The vocabulary dict as the leading arguments of hvo_bow_set_vocabulary (n_nodes, child_start, child_ids, node_desc, node_weight,
    node_word, depth_levels); the arrays are returned as well, to be kept alive over the call."""
    cs = np.ascontiguousarray(voc['child_start'], np.int32); ci = np.ascontiguousarray(voc['child_ids'], np.int32)
    nd = np.ascontiguousarray(voc['node_desc'], np.uint8); nw = np.ascontiguousarray(voc['node_weight'], np.float64)
    wd = np.ascontiguousarray(voc['node_word'], np.int32)
    args = (len(nw), _np_ptr(cs), _np_ptr(ci) if len(ci) else None, _np_ptr(nd), _np_ptr(nw), _np_ptr(wd), int(voc['L']))
    return args, (cs, ci, nd, nw, wd)


class ORBVocabulary:
    """Mirror of ORB_SLAM2::ORBVocabulary (= DBoW2::TemplatedVocabulary<FORB::TDescriptor, FORB>, reference include/ORBVocabulary.h) for the
    one call on the path, transform(features, BowVector, FeatureVector, levelsup) as used by Frame::ComputeBoW (src/Frame.cc:1692-1699).
    voc = dict(child_start [n+1], child_ids, node_desc [n,32], node_weight [n], node_word [n], L)."""

    def __init__(self, voc, device=0):
        out = _vp()
        _check(lib().hvo_bow_create(int(device), C.byref(out)))
        self._h = out
        args, _keep = _vocabulary_args(voc)
        _check(lib().hvo_bow_set_vocabulary(self._h, *args))

    def close(self):
        if getattr(self, '_h', None):
            lib().hvo_bow_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def transform_batch(self, desc_list, levelsup=4):
        """[(BowVector as (words, values), FeatureVector as dict node -> feature indices, word_of, node_of)] for every frame."""
        counts = [len(d) for d in desc_list]
        off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
        total = int(off[-1])
        desc = np.concatenate([np.ascontiguousarray(d, np.uint8).reshape(-1, 32) for d in desc_list] + [np.zeros((0, 32), np.uint8)])
        nf = len(desc_list)
        word = np.full(max(total, 1), -1, np.int32); node = np.zeros(max(total, 1), np.int32)
        bc = np.zeros(max(nf, 1), np.int32); bw = np.zeros(max(total, 1), np.int32); bv = np.zeros(max(total, 1), np.float64)
        fo = np.full(max(total, 1), -1, np.int32); fc = np.zeros(max(nf, 1), np.int32)
        _check(lib().hvo_bow_transform(self._h, _np_ptr(desc) if total else None, _np_ptr(off), nf, int(levelsup), _np_ptr(word), _np_ptr(node),
                                       _np_ptr(bc), _np_ptr(bw), _np_ptr(bv), _np_ptr(fo), _np_ptr(fc)))
        out = []
        for f in range(nf):
            a, n = int(off[f]), counts[f]
            order = fo[a:a + fc[f]]
            fv = {}
            for i in order:
                fv.setdefault(int(node[a + i]), []).append(int(i))
            out.append(((bw[a:a + bc[f]].copy(), bv[a:a + bc[f]].copy()), fv, word[a:a + n].copy(), node[a:a + n].copy()))
        return out

    def transform(self, desc, levelsup=4):
        return self.transform_batch([desc], levelsup)[0]


class ProjectionMatcher:
    """Device side of the windowed matchers: the frame grid (Frame::AssignFeaturesToGrid, src/Frame.cc:832-847),
    Frame::GetFeaturesInArea (:1502-1555) and the greedy search of ORBmatcher::SearchByProjection (src/ORBmatcher.cc:45-132,
    1353-1497).  One frame at a time."""

    def __init__(self, device=0):
        out = _vp()
        _check(lib().hvo_proj_create(int(device), C.byref(out)))
        self._h = out
        self.n = 0

    def close(self):
        if getattr(self, '_h', None):
            lib().hvo_proj_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_frame(self, keys_un, uright, desc, min_x, min_y, max_x, max_y, window_origin=None):
        """window_origin = (mnMinX, mnMinY) of a KeyFrame (integers, include/KeyFrame.h:249-252): KeyFrame::GetFeaturesInArea locates its
        windows from them in the cells the Frame assigned with the float bounds (hvo_proj_set_window_origin)."""
        keys = np.ascontiguousarray(keys_un, KP_DTYPE)
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        ur = None if uright is None else np.ascontiguousarray(uright, np.float32)
        self.n = len(keys)
        _check(lib().hvo_proj_set_frame(self._h, _np_ptr(keys), _np_ptr(ur) if ur is not None else None, _np_ptr(desc), self.n,
                                        float(min_x), float(min_y), float(max_x), float(max_y)))
        if window_origin is not None:
            _check(lib().hvo_proj_set_window_origin(self._h, float(window_origin[0]), float(window_origin[1])))

    def grid(self):
        """(cell_start [64*48+1], cell_items): cell ix*48+iy lists mGrid[ix][iy]."""
        cs = np.empty(GRID_COLS * GRID_ROWS + 1, np.int32)
        items = np.empty(max(self.n, 1), np.int32)
        _check(lib().hvo_proj_get_grid(self._h, _np_ptr(cs), _np_ptr(items)))
        return cs, items[:cs[-1]].copy()

    def GetFeaturesInArea(self, x, y, r, minLevel=-1, maxLevel=-1):
        out = np.empty(max(self.n, 1), np.int32)
        n = C.c_int(0)
        _check(lib().hvo_proj_features_in_area(self._h, float(x), float(y), float(r), int(minLevel), int(maxLevel), _np_ptr(out), len(out),
                                               C.byref(n)))
        return out[:n.value].copy()

    def search(self, queries, qdesc, claimed=None, mode=0, th_dist=100, nnratio=0.6):
        q = np.ascontiguousarray(queries, PROJ_QUERY_DTYPE)
        qd = np.ascontiguousarray(qdesc, np.uint8).reshape(-1, 32)
        cl = None if claimed is None else np.ascontiguousarray(claimed, np.uint8)
        idx = np.full(max(len(q), 1), -1, np.int32)
        dist = np.full(max(len(q), 1), 256, np.int32)
        nm = C.c_int(0)
        _check(lib().hvo_proj_search(self._h, _np_ptr(q), _np_ptr(qd), len(q), _np_ptr(cl) if cl is not None else None, int(mode),
                                     int(th_dist), float(nnratio), _np_ptr(idx), _np_ptr(dist), C.byref(nm)))
        return idx[:len(q)], dist[:len(q)], nm.value

    def frustum_points(self, cam, pts, viewing_cos_limit=0.5):
        """Frame::isInFrustum(MapPoint*, viewingCosLimit) (src/Frame.cc:1371-1436) for a batch: cam FRUSTUM_CAM_DTYPE, pts MAP_POINT_DTYPE."""
        cam = np.ascontiguousarray(cam, FRUSTUM_CAM_DTYPE); pts = np.ascontiguousarray(pts, MAP_POINT_DTYPE)
        out = np.zeros(max(len(pts), 1), TRACK_POINT_DTYPE)
        _check(lib().hvo_proj_frustum_points(self._h, _np_ptr(cam), _np_ptr(pts), len(pts), float(viewing_cos_limit), _np_ptr(out)))
        return out[:len(pts)]

    def search_local_map(self, cam, pts, pdesc, scale_factors, skip=None, claims=None, claimed=None, viewing_cos_limit=0.5, th=1.0, th_dist=100,
                         nnratio=0.8):
        """isInFrustum over the local map + ORBmatcher::SearchByProjection(F, vpMapPoints, th) in one call (Tracking.cc:3251-3268)."""
        cam = np.ascontiguousarray(cam, FRUSTUM_CAM_DTYPE); pts = np.ascontiguousarray(pts, MAP_POINT_DTYPE)
        n = len(pts)
        pd = np.ascontiguousarray(pdesc, np.uint8).reshape(-1, 32)
        sf = np.ascontiguousarray(scale_factors, np.float32)
        opt = lambda a: None if a is None else np.ascontiguousarray(a, np.uint8)
        sk, cl, cd = opt(skip), opt(claims), opt(claimed)
        track = np.zeros(max(n, 1), TRACK_POINT_DTYPE); idx = np.full(max(n, 1), -1, np.int32); dist = np.full(max(n, 1), 256, np.int32)
        niv, nm = C.c_int(0), C.c_int(0)
        p = lambda a: _np_ptr(a) if a is not None else None
        _check(lib().hvo_proj_search_local_map(self._h, _np_ptr(cam), _np_ptr(pts), _np_ptr(pd), p(sk), p(cl), n, float(viewing_cos_limit), float(th),
                                               _np_ptr(sf), p(cd), int(th_dist), float(nnratio), _np_ptr(track), _np_ptr(idx), _np_ptr(dist),
                                               C.byref(niv), C.byref(nm)))
        return track[:n], idx[:n], dist[:n], niv.value, nm.value

    def search_initialization(self, prev_matched, octave1, desc1, window_size=100, th_dist=50, nnratio=0.9):
        """The loop of ORBmatcher::SearchForInitialization (src/ORBmatcher.cc:412-497) against the frame set by set_frame (= F2).
        Returns (matches12, accepted12, nmatches) before the rotation-histogram culling."""
        pm = np.ascontiguousarray(prev_matched, np.float32).reshape(-1, 2)
        oc = np.ascontiguousarray(octave1, np.int32); d1 = np.ascontiguousarray(desc1, np.uint8).reshape(-1, 32)
        n1 = len(pm)
        m12 = np.full(max(n1, 1), -1, np.int32); acc = np.full(max(n1, 1), -1, np.int32)
        nm = C.c_int(0)
        _check(lib().hvo_proj_search_initialization(self._h, _np_ptr(pm), _np_ptr(oc), _np_ptr(d1), n1, int(window_size), int(th_dist), float(nnratio),
                                                    _np_ptr(m12), _np_ptr(acc), C.byref(nm)))
        return m12[:n1], acc[:n1], nm.value

    def set_level_sigma(self, inv_level_sigma2):
        s = np.ascontiguousarray(inv_level_sigma2, np.float32)
        _check(lib().hvo_proj_set_level_sigma(self._h, _np_ptr(s), len(s)))

    def rounds(self):
        return lib().hvo_proj_last_rounds(self._h)

    def match_candidates(self, q, t, offsets, cand):
        q = np.ascontiguousarray(q, np.uint8).reshape(-1, 32)
        t = np.ascontiguousarray(t, np.uint8).reshape(-1, 32)
        off = np.ascontiguousarray(offsets, np.int32)
        cd = np.ascontiguousarray(cand, np.int32)
        best4 = np.empty((max(len(q), 1), 4), np.int32)
        _check(lib().hvo_proj_match_candidates(self._h, _np_ptr(q), len(q), _np_ptr(t), len(t), _np_ptr(off), _np_ptr(cd), _np_ptr(best4)))
        self.n = 0
        return best4[:len(q)]

    def search_triangulation(self, qdesc, qkeys, qstereo, tdesc, tkeys, tflags, offsets, cand, F12, ex, ey, scale_factors, level_sigma2,
                             only_stereo=False, th_low=50):
        """the candidate loop of ORBmatcher::SearchForTriangulation (hvo_proj_search_triangulation)."""
        qd = np.ascontiguousarray(qdesc, np.uint8).reshape(-1, 32); qk = np.ascontiguousarray(qkeys, KP_DTYPE)
        qs = np.ascontiguousarray(qstereo, np.uint8)
        td = np.ascontiguousarray(tdesc, np.uint8).reshape(-1, 32); tk = np.ascontiguousarray(tkeys, KP_DTYPE)
        tf = np.ascontiguousarray(tflags, np.uint8)
        off = np.ascontiguousarray(offsets, np.int32); cd = np.ascontiguousarray(cand, np.int32)
        F = np.ascontiguousarray(F12, np.float32).reshape(9)
        sf = np.ascontiguousarray(scale_factors, np.float32); sg = np.ascontiguousarray(level_sigma2, np.float32)
        idx = np.full(max(len(qd), 1), -1, np.int32); dist = np.full(max(len(qd), 1), 256, np.int32)
        nm = C.c_int(0)
        _check(lib().hvo_proj_search_triangulation(self._h, _np_ptr(qd), _np_ptr(qk), _np_ptr(qs), len(qd), _np_ptr(td), _np_ptr(tk), _np_ptr(tf),
                                                   len(td), _np_ptr(off), _np_ptr(cd), _np_ptr(F), float(np.float32(ex)), float(np.float32(ey)),
                                                   _np_ptr(sf), _np_ptr(sg), len(sf), int(bool(only_stereo)), int(th_low), _np_ptr(idx),
                                                   _np_ptr(dist), C.byref(nm)))
        self.n = 0
        return idx[:len(qd)], dist[:len(qd)], nm.value

    def search_candidates(self, q, t, offsets, cand, th_dist=50, nnratio=0.7):
        """greedy best / second over caller-given candidate lists (the loop of ORBmatcher::SearchByBoW)."""
        q = np.ascontiguousarray(q, np.uint8).reshape(-1, 32)
        t = np.ascontiguousarray(t, np.uint8).reshape(-1, 32)
        off = np.ascontiguousarray(offsets, np.int32)
        cd = np.ascontiguousarray(cand, np.int32)
        idx = np.full(max(len(q), 1), -1, np.int32); dist = np.full(max(len(q), 1), 256, np.int32)
        nm = C.c_int(0)
        _check(lib().hvo_proj_search_candidates(self._h, _np_ptr(q), len(q), _np_ptr(t), len(t), _np_ptr(off), _np_ptr(cd), int(th_dist),
                                                float(np.float32(nnratio)), _np_ptr(idx), _np_ptr(dist), C.byref(nm)))
        self.n = 0
        return idx[:len(q)], dist[:len(q)], nm.value

    def timer_start(self):
        _check(lib().hvo_proj_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(lib().hvo_proj_timer_stop(self._h, C.byref(ms)))
        return ms.value


class ORBmatcher:
    """Mirror of ORB_SLAM2::ORBmatcher for the projection searches (reference include/ORBmatcher.h:38-77).  Frames and map
    points are plain arrays (the reference's Frame / MapPoint objects stay with the caller):

        F   = dict(keys_un KP_DTYPE [N], uright [N], desc [N,32], bounds (minX, minY, maxX, maxY), scale_factors [L],
                   mappoint [N] int (index of the map point held, -1 none), claimed [N] bool (holds one with observations))
        MPs = dict(proj_x, proj_y, proj_xr, view_cos, level, in_view, bad, has_obs, desc [M,32])
    """
    TH_LOW, TH_HIGH, HISTO_LENGTH = 50, 100, 30  # ORBmatcher.cc:37-39

    def __init__(self, nnratio=0.6, checkOri=True, device=0):
        self.mfNNratio, self.mbCheckOrientation = float(nnratio), bool(checkOri)
        self._pm = ProjectionMatcher(device)

    @staticmethod
    def DescriptorDistance(a, b):
        a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8)
        return int(lib().hvo_hamming_distance(_np_ptr(a), _np_ptr(b)))

    @staticmethod
    def RadiusByViewingCos(viewCos):  # ORBmatcher.cc:134-140
        return np.where(np.asarray(viewCos, np.float32) > np.float32(0.998), np.float32(2.5), np.float32(4.0))

    def _set_frame(self, F):
        b = F['bounds']
        self._pm.set_frame(F['keys_un'], F.get('uright'), F['desc'], b[0], b[1], b[2], b[3])

    def _set_keyframe(self, KF, with_uright):
        """A key frame searched in: the grid of its Frame (float bounds), windows located from the key frame's integer origin
        (src/KeyFrame.cc:627-666); KF['bounds'] are the Frame's float bounds."""
        b = KF['bounds']
        self._pm.set_frame(KF['keys_un'], KF.get('uright') if with_uright else None, KF['desc'], b[0], b[1], b[2], b[3],
                           window_origin=(int(b[0]), int(b[1])))

    def SearchByProjection(self, F, MPs, th=1.0):
        """ORBmatcher::SearchByProjection(Frame&, const vector<MapPoint*>&, th) (ORBmatcher.cc:45-132).  Updates F['mappoint']
        and F['claimed'] in place, returns (nmatches, match [M] keypoint index or -1)."""
        M = len(MPs['proj_x'])
        use = np.asarray(MPs['in_view'], bool) & ~np.asarray(MPs['bad'], bool)
        sel = np.nonzero(use)[0]
        lvl = np.asarray(MPs['level'], np.int32)[sel]
        r = self.RadiusByViewingCos(np.asarray(MPs['view_cos'])[sel]).astype(np.float32)
        if th != 1.0:
            r = (r * np.float32(th)).astype(np.float32)
        q = np.zeros(len(sel), PROJ_QUERY_DTYPE)
        q['u'] = np.asarray(MPs['proj_x'], np.float32)[sel]; q['v'] = np.asarray(MPs['proj_y'], np.float32)[sel]
        q['r'] = (r * np.asarray(F['scale_factors'], np.float32)[lvl]).astype(np.float32)
        q['min_level'] = lvl - 1; q['max_level'] = lvl
        q['ur'] = np.asarray(MPs['proj_xr'], np.float32)[sel]
        q['claims'] = np.asarray(MPs['has_obs'], bool)[sel]
        self._set_frame(F)
        idx, dist, nm = self._pm.search(q, np.asarray(MPs['desc'], np.uint8)[sel], F.get('claimed'), 0, self.TH_HIGH, self.mfNNratio)
        match = np.full(M, -1, np.int32)
        match[sel] = idx
        for k, i in zip(sel, idx):  # F.mvpMapPoints[bestIdx] = pMP, in query order
            if i >= 0:
                F['mappoint'][i] = k
                if MPs['has_obs'][k]:
                    F['claimed'][i] = True
                else:
                    F['claimed'][i] = False
        return nm, match

    @staticmethod
    def bow_queries(featvec_kf, featvec_f, kf_has_mappoint):
        """The visiting order of SearchByBoW (ORBmatcher.cc:180-266): vocabulary nodes present in both DBoW2::FeatureVectors,
        ascending; inside a node the key frame's index list, keeping features that hold a good map point; candidates = the
        frame's index list of that node.  featvec_* : dict node id -> list of feature indices.  Returns (query feature index
        [nq], offsets [nq+1], cand)."""
        qi, off, cand = [], [0], []
        for node in sorted(set(featvec_kf) & set(featvec_f)):
            fl = list(featvec_f[node])
            for i in featvec_kf[node]:
                if kf_has_mappoint[i]:
                    qi.append(i); cand.extend(fl); off.append(len(cand))
        return np.asarray(qi, np.int32), np.asarray(off, np.int32), np.asarray(cand, np.int32)

    def SearchForTriangulation(self, KF1, KF2, F12, epipole, bOnlyStereo=False):
        """ORBmatcher::SearchForTriangulation(pKF1, pKF2, F12, vMatchedPairs, bOnlyStereo) (ORBmatcher.cc:668-836).
        KFi = dict(desc, keys_un, uright, featvec, has_mappoint [N] bool, scale_factors, level_sigma2); epipole = (ex, ey) of pKF1's
        camera centre in pKF2 (:676-683, host pose algebra).  Returns (nmatches, vMatchedPairs [[idx1, idx2]])."""
        free1 = ~np.asarray(KF1['has_mappoint'], bool)
        qi, off, cand = self.bow_queries(KF1['featvec'], KF2['featvec'], free1)
        if len(qi) == 0:
            return 0, np.zeros((0, 2), np.int32)
        ur1 = np.asarray(KF1['uright'], np.float32); ur2 = np.asarray(KF2['uright'], np.float32)
        tflags = (np.asarray(KF2['has_mappoint'], bool).astype(np.uint8) | ((ur2 >= 0).astype(np.uint8) << 1)).astype(np.uint8)
        idx, _, nm = self._pm.search_triangulation(np.asarray(KF1['desc'], np.uint8)[qi], np.asarray(KF1['keys_un'], KP_DTYPE)[qi],
                                                   (ur1[qi] >= 0), KF2['desc'], KF2['keys_un'], tflags, off, cand, F12, epipole[0], epipole[1],
                                                   KF2['scale_factors'], KF2['level_sigma2'], bOnlyStereo, self.TH_LOW)
        m12 = np.full(len(KF1['desc']), -1, np.int32)
        hist = [[] for _ in range(self.HISTO_LENGTH)]
        factor = np.float32(1.0) / np.float32(self.HISTO_LENGTH)
        for k, i in zip(qi, idx):
            if i < 0:
                continue
            m12[k] = i
            if self.mbCheckOrientation:
                rot = np.float32(KF1['keys_un']['angle'][k]) - np.float32(KF2['keys_un']['angle'][i])
                if rot < 0.0:
                    rot = np.float32(rot + np.float32(360.0))
                b = int(np.floor(float(np.float32(rot * factor)) + 0.5))  # round(): rot >= 0 here
                if b == self.HISTO_LENGTH:
                    b = 0
                hist[b].append(k)
        if self.mbCheckOrientation:
            keep = set(self.ComputeThreeMaxima([len(h) for h in hist]))
            for b in range(self.HISTO_LENGTH):
                if b not in keep:
                    for k in hist[b]:
                        m12[k] = -1
                        nm -= 1
        i1 = np.nonzero(m12 >= 0)[0]
        return nm, np.stack([i1, m12[i1]], axis=1).astype(np.int32)

    def SearchByBoWKF(self, KF1, KF2):
        """ORBmatcher::SearchByBoW(pKF1, pKF2, vpMatches12) (ORBmatcher.cc:531-666).  KFi = dict(desc, keys_un, featvec, has_mappoint [N] bool
        (map point present and not bad)).  Candidates of a node = pKF2's features of that node that hold a good map point; accepted when
        bestDist1 < TH_LOW (strict) and best < ratio * second; a matched pKF2 feature is skipped by later queries.
        Returns (nmatches, match12 [N1] = pKF2 feature whose map point pKF1's feature is matched to, or -1)."""
        qi, off, cand = self.bow_queries(KF1['featvec'], KF2['featvec'], np.asarray(KF1['has_mappoint'], bool))
        m12 = np.full(len(KF1['desc']), -1, np.int32)
        if len(qi) == 0:
            return 0, m12
        good2 = np.asarray(KF2['has_mappoint'], bool)
        off2, cand2 = [0], []
        for a, b in zip(off[:-1], off[1:]):
            seg = cand[a:b]
            cand2.extend(seg[good2[seg]]); off2.append(len(cand2))
        idx, _, nm = self._pm.search_candidates(np.asarray(KF1['desc'], np.uint8)[qi], KF2['desc'], np.asarray(off2, np.int32),
                                                np.asarray(cand2, np.int32), self.TH_LOW - 1, self.mfNNratio)
        hist = [[] for _ in range(self.HISTO_LENGTH)]
        factor = np.float32(1.0) / np.float32(self.HISTO_LENGTH)
        for k, i in zip(qi, idx):
            if i < 0:
                continue
            m12[k] = i
            if self.mbCheckOrientation:
                rot = np.float32(KF1['keys_un']['angle'][k]) - np.float32(KF2['keys_un']['angle'][i])
                if rot < 0.0:
                    rot = np.float32(rot + np.float32(360.0))
                b = int(np.floor(float(np.float32(rot * factor)) + 0.5))  # round(): rot >= 0 here
                if b == self.HISTO_LENGTH:
                    b = 0
                hist[b].append(k)
        if self.mbCheckOrientation:
            keepb = set(self.ComputeThreeMaxima([len(h) for h in hist]))
            for b in range(self.HISTO_LENGTH):
                if b not in keepb:
                    for k in hist[b]:
                        m12[k] = -1
                        nm -= 1
        return nm, m12

    def SearchByBoW(self, KF, F):
        """ORBmatcher::SearchByBoW(KeyFrame*, Frame&, vpMapPointMatches) (ORBmatcher.cc:162-293).
        KF = dict(desc [N,32], keys_un KP_DTYPE, featvec {node: [idx]}, has_mappoint [N] bool (map point present and not bad));
        F  = dict(desc [M,32], keys KP_DTYPE, featvec).  Returns (nmatches, match [M] = key-frame feature whose map point the
        frame feature received, or -1)."""
        qi, off, cand = self.bow_queries(KF['featvec'], F['featvec'], np.asarray(KF['has_mappoint'], bool))
        M = len(F['desc'])
        match = np.full(M, -1, np.int32)
        if len(qi) == 0:
            return 0, match
        idx, _, nm = self._pm.search_candidates(np.asarray(KF['desc'], np.uint8)[qi], F['desc'], off, cand, self.TH_LOW, self.mfNNratio)
        hist = [[] for _ in range(self.HISTO_LENGTH)]
        factor = np.float32(1.0) / np.float32(self.HISTO_LENGTH)
        for k, i in zip(qi, idx):
            if i < 0:
                continue
            match[i] = k
            if self.mbCheckOrientation:
                rot = np.float32(KF['keys_un']['angle'][k]) - np.float32(F['keys']['angle'][i])
                if rot < 0.0:
                    rot = np.float32(rot + np.float32(360.0))
                b = int(np.floor(float(np.float32(rot * factor)) + 0.5))  # round(): rot >= 0 here
                if b == self.HISTO_LENGTH:
                    b = 0
                hist[b].append(i)
        if self.mbCheckOrientation:
            keep = set(self.ComputeThreeMaxima([len(h) for h in hist]))
            for b in range(self.HISTO_LENGTH):
                if b not in keep:
                    for i in hist[b]:
                        match[i] = -1
                        nm -= 1
        return nm, match

    def SearchLocalPoints(self, F, cam, pts, pdesc, skip, has_obs, th=1.0, viewing_cos_limit=0.5):
        """The device work of Tracking::SearchLocalPoints (src/Tracking.cc:3251-3268): Frame::isInFrustum over the local map points and
        ORBmatcher::SearchByProjection(F, vpMapPoints, th), the projected queries never leaving the device.  skip = already matched in
        this frame (mnLastFrameSeen) or isBad().  Updates F['mappoint'] / F['claimed']; returns (track, nmatches, match [M])."""
        self._set_frame(F)
        track, idx, dist, niv, nm = self._pm.search_local_map(cam, pts, pdesc, F['scale_factors'], skip, has_obs, F.get('claimed'),
                                                              viewing_cos_limit, th, self.TH_HIGH, self.mfNNratio)
        for k, i in enumerate(idx):
            if i >= 0:
                F['mappoint'][i] = k
                F['claimed'][i] = bool(has_obs[k])
        return track, nm, idx

    def SearchForInitialization(self, F1, F2, vbPrevMatched, windowSize=10):
        """ORBmatcher::SearchForInitialization(F1, F2, vbPrevMatched, vnMatches12, windowSize) (src/ORBmatcher.cc:412-529): the sequential loop
        on the device, the rotation histogram (:499-523) and the vbPrevMatched update (:525-528) here.  Fi = dict(keys_un, desc, bounds).
        Returns (nmatches, vnMatches12, vbPrevMatched)."""
        k1 = np.ascontiguousarray(F1['keys_un'], KP_DTYPE)
        prev = np.array(vbPrevMatched, np.float32).reshape(-1, 2)
        self._set_frame(F2)
        m12, acc, nm = self._pm.search_initialization(prev, k1['octave'], F1['desc'], windowSize, self.TH_LOW, self.mfNNratio)
        m12 = m12.copy()
        if self.mbCheckOrientation:
            k2 = np.ascontiguousarray(F2['keys_un'], KP_DTYPE)
            hist = [[] for _ in range(self.HISTO_LENGTH)]
            factor = np.float32(1.0) / np.float32(self.HISTO_LENGTH)
            for i1, i2 in enumerate(acc):
                if i2 < 0:
                    continue
                rot = np.float32(k1['angle'][i1] - k2['angle'][i2])
                if rot < 0.0:
                    rot = np.float32(rot + np.float32(360.0))
                b = int(np.floor(float(np.float32(rot * factor)) + 0.5))
                if b == self.HISTO_LENGTH:
                    b = 0
                hist[b].append(i1)
            i1m, i2m, i3m = self.ComputeThreeMaxima([len(h) for h in hist])
            for b in range(self.HISTO_LENGTH):
                if b not in (i1m, i2m, i3m):
                    for i1 in hist[b]:
                        if m12[i1] >= 0:
                            m12[i1] = -1
                            nm -= 1
        k2 = np.ascontiguousarray(F2['keys_un'], KP_DTYPE)
        for i1 in np.nonzero(m12 >= 0)[0]:
            prev[i1, 0] = k2['x'][m12[i1]]; prev[i1, 1] = k2['y'][m12[i1]]
        return nm, m12, prev

    @staticmethod
    def ComputeThreeMaxima(sizes):  # ORBmatcher.cc:1630-1671
        max1 = max2 = max3 = 0
        ind1 = ind2 = ind3 = -1
        for i, s in enumerate(sizes):
            if s > max1:
                max3, max2, max1 = max2, max1, s
                ind3, ind2, ind1 = ind2, ind1, i
            elif s > max2:
                max3, max2 = max2, s
                ind3, ind2 = ind2, i
            elif s > max3:
                max3, ind3 = s, i
        if max2 < np.float32(0.1) * np.float32(max1):
            ind2 = ind3 = -1
        elif max3 < np.float32(0.1) * np.float32(max1):
            ind3 = -1
        return ind1, ind2, ind3

    def SearchByProjectionLast(self, Cur, last, th, forward=False, backward=False):
        """Matching part of SearchByProjection(CurrentFrame, LastFrame, th, mono) (ORBmatcher.cc:1353-1497).  `last` holds, for
        every last-frame keypoint with a usable map point, its projection into the current frame: dict(u, v, ur, octave,
        angle, has_obs, desc), in last-frame index order.  Returns (nmatches, match [len(last)])."""
        n = len(last['u'])
        octv = np.asarray(last['octave'], np.int32)
        q = np.zeros(n, PROJ_QUERY_DTYPE)
        q['u'] = last['u']; q['v'] = last['v']; q['ur'] = last['ur']
        q['r'] = (np.float32(th) * np.asarray(Cur['scale_factors'], np.float32)[octv]).astype(np.float32)
        if forward:
            q['min_level'] = octv; q['max_level'] = -1
        elif backward:
            q['min_level'] = 0; q['max_level'] = octv
        else:
            q['min_level'] = octv - 1; q['max_level'] = octv + 1
        q['claims'] = np.asarray(last['has_obs'], bool)
        self._set_frame(Cur)
        idx, dist, nm = self._pm.search(q, last['desc'], Cur.get('claimed'), 1, self.TH_HIGH, self.mfNNratio)
        return self._apply_with_rotation_check(Cur, last, idx.copy(), nm, np.asarray(last['has_obs'], bool))

    def Fuse(self, KF, MPs, th=3.0):
        """The search of ORBmatcher::Fuse(KeyFrame*, const vector<MapPoint*>&, th) (ORBmatcher.cc:838-990).  KF = dict(keys_un, uright,
        desc, bounds, scale_factors, inv_level_sigma2); MPs = the map points that pass the reference's projection tests (good, not in
        the key frame, positive depth, inside the image, distance and viewing-angle tests): dict(u, v, ur, level (PredictScale), desc).
        Returns (nFused, bestIdx [M] key-frame keypoint or -1); Replace / AddObservation on the result stay with the caller."""
        M = len(MPs['u'])
        lvl = np.asarray(MPs['level'], np.int32)
        q = np.zeros(M, PROJ_QUERY_DTYPE)
        q['u'] = MPs['u']; q['v'] = MPs['v']; q['ur'] = MPs['ur']
        q['r'] = (np.float32(th) * np.asarray(KF['scale_factors'], np.float32)[lvl]).astype(np.float32)
        q['min_level'] = lvl - 1; q['max_level'] = lvl
        self._set_keyframe(KF, True)
        self._pm.set_level_sigma(KF['inv_level_sigma2'])
        idx, _, nm = self._pm.search(q, MPs['desc'], None, 2, self.TH_LOW, self.mfNNratio)
        return nm, idx.copy()

    def FuseSim3(self, KF, pts, th):
        """The search of ORBmatcher::Fuse(KeyFrame*, cv::Mat Scw, const vector<MapPoint*>&, th, vpReplacePoint) (ORBmatcher.cc:992-1121,
        loop closing): window of radius th * sf[level] at levels [level-1, level], best Hamming distance, accepted when <= TH_LOW;
        no reprojection gate, nothing is claimed.  pts = dict(u, v, level, desc) of the points that pass the Sim3 projection tests.
        Returns (count, bestIdx [M])."""
        lvl = np.asarray(pts['level'], np.int32)
        q = np.zeros(len(lvl), PROJ_QUERY_DTYPE)
        q['u'] = pts['u']; q['v'] = pts['v']; q['ur'] = -1
        q['r'] = (np.float32(th) * np.asarray(KF['scale_factors'], np.float32)[lvl]).astype(np.float32)
        q['min_level'] = lvl - 1; q['max_level'] = lvl
        self._set_keyframe(KF, False)
        idx, _, nm = self._pm.search(q, pts['desc'], None, 1, self.TH_LOW, self.mfNNratio)
        return nm, idx.copy()

    def SearchBySim3(self, KF1, KF2, pts1in2, pts2in1, th):
        """The searches of ORBmatcher::SearchBySim3(pKF1, pKF2, vpMatches12, s12, R12, t12, th) (ORBmatcher.cc:1123-1351): the map
        points of KF1 projected into KF2 and those of KF2 projected into KF1 (Sim3 algebra, PredictScale and the already-matched /
        bad / out-of-range filters stay with the caller), each matched to the best descriptor in its window at levels
        [level-1, level] when <= TH_HIGH, kept where both directions agree (:1213-1228).  ptsAinB = dict(index (feature of A),
        u, v, level, desc).  Returns (nFound, pairs [[idx1, idx2]])."""
        def one(KF, pts):
            lvl = np.asarray(pts['level'], np.int32)
            q = np.zeros(len(lvl), PROJ_QUERY_DTYPE)
            q['u'] = pts['u']; q['v'] = pts['v']; q['ur'] = -1
            q['r'] = (np.float32(th) * np.asarray(KF['scale_factors'], np.float32)[lvl]).astype(np.float32)
            q['min_level'] = lvl - 1; q['max_level'] = lvl
            self._set_keyframe(KF, False)
            return self._pm.search(q, pts['desc'], None, 1, self.TH_HIGH, self.mfNNratio)[0]
        m1 = np.full(len(KF1['desc']), -1, np.int32); m2 = np.full(len(KF2['desc']), -1, np.int32)
        if len(pts1in2['u']):
            m1[np.asarray(pts1in2['index'], np.int64)] = one(KF2, pts1in2)
        if len(pts2in1['u']):
            m2[np.asarray(pts2in1['index'], np.int64)] = one(KF1, pts2in1)
        i1 = np.nonzero(m1 >= 0)[0]
        ok = m2[m1[i1]] == i1
        pairs = np.stack([i1[ok], m1[i1[ok]]], axis=1).astype(np.int32)
        return len(pairs), pairs

    def SearchByProjectionSim3(self, KF, pts, matched, th):
        """The search of ORBmatcher::SearchByProjection(KeyFrame*, cv::Mat Scw, vpPoints, vpMatched, th) (ORBmatcher.cc:295-410, loop
        detection): like FuseSim3, but key-frame features already in vpMatched are skipped and every match is entered into it.
        `matched` [N] bool is updated in place.  Returns (nmatches, bestIdx [M])."""
        lvl = np.asarray(pts['level'], np.int32)
        q = np.zeros(len(lvl), PROJ_QUERY_DTYPE)
        q['u'] = pts['u']; q['v'] = pts['v']; q['ur'] = -1
        q['r'] = (np.float32(th) * np.asarray(KF['scale_factors'], np.float32)[lvl]).astype(np.float32)
        q['min_level'] = lvl - 1; q['max_level'] = lvl
        q['claims'] = 1
        self._set_keyframe(KF, False)
        idx, _, nm = self._pm.search(q, pts['desc'], np.asarray(matched, np.uint8), 1, self.TH_LOW, self.mfNNratio)
        matched[idx[idx >= 0]] = True
        return nm, idx.copy()

    def SearchByProjectionKF(self, Cur, kf, th, ORBdist):
        """Matching part of SearchByProjection(CurrentFrame, KeyFrame*, sAlreadyFound, th, ORBdist) (ORBmatcher.cc:1499-1628, used by
        relocalisation).  `kf` holds, for every key-frame map point that is good, not already found and projects inside the image
        at a valid distance: dict(u, v, level (PredictScale), angle (of the key frame's keypoint), desc), in key-frame index order.
        A frame keypoint that holds any map point is skipped (:1568-1569), the right coordinate is not checked, accept best <= ORBdist.
        Cur['claimed'] must mark every keypoint with a map point.  Returns (nmatches, match [len(kf)])."""
        n = len(kf['u'])
        lvl = np.asarray(kf['level'], np.int32)
        q = np.zeros(n, PROJ_QUERY_DTYPE)
        q['u'] = kf['u']; q['v'] = kf['v']; q['ur'] = -1
        q['r'] = (np.float32(th) * np.asarray(Cur['scale_factors'], np.float32)[lvl]).astype(np.float32)
        q['min_level'] = lvl - 1; q['max_level'] = lvl + 1
        q['claims'] = 1
        b = Cur['bounds']
        self._pm.set_frame(Cur['keys_un'], None, Cur['desc'], b[0], b[1], b[2], b[3])   # no uRight: this variant has no stereo check
        idx, dist, nm = self._pm.search(q, kf['desc'], Cur.get('claimed'), 1, int(ORBdist), self.mfNNratio)
        return self._apply_with_rotation_check(Cur, kf, idx.copy(), nm, np.ones(n, bool))

    def _apply_with_rotation_check(self, Cur, last, idx, nm, has_obs):
        for k, i in enumerate(idx):
            if i >= 0:
                Cur['mappoint'][i] = k
                Cur['claimed'][i] = bool(has_obs[k])
        if self.mbCheckOrientation:  # rotation consistency (:1458-1494, :1594-1622)
            hist = [[] for _ in range(self.HISTO_LENGTH)]
            factor = np.float32(1.0) / np.float32(self.HISTO_LENGTH)
            ang_c = np.asarray(Cur['keys_un']['angle'], np.float32)
            for k, i in enumerate(idx):
                if i < 0:
                    continue
                rot = np.float32(last['angle'][k]) - ang_c[i]
                if rot < 0.0:
                    rot = np.float32(rot + np.float32(360.0))
                b = int(np.floor(float(np.float32(rot * factor)) + 0.5))  # round(): rot >= 0 here
                if b == self.HISTO_LENGTH:
                    b = 0
                hist[b].append(i)
            i1, i2, i3 = self.ComputeThreeMaxima([len(h) for h in hist])
            for b in range(self.HISTO_LENGTH):
                if b not in (i1, i2, i3):
                    for i in hist[b]:
                        Cur['mappoint'][i] = -1
                        Cur['claimed'][i] = False
                        nm -= 1
        return nm, idx


class _FrameParams(C.Structure):
    _fields_ = [('orb', _OrbParams), ('line', _LineParams), ('fx', C.c_float), ('fy', C.c_float), ('cx', C.c_float), ('cy', C.c_float),
                ('depth_factor', C.c_float), ('bf', C.c_float), ('distorted', C.c_int), ('stages', C.c_int), ('max_planes', C.c_int), ('line_cull', C.c_int),
                ('lanes', C.c_int), ('k1', C.c_float), ('k2', C.c_float), ('p1', C.c_float), ('p2', C.c_float), ('k3', C.c_float)]


class _FrameOutputs(C.Structure):
    _fields_ = [(n, _vp) for n in ('kps', 'desc', 'kp_counts', 'kp_depth', 'kp_uright', 'keylines', 'line_desc', 'linevec3',
                                   'line_counts', 'n_planes', 'planes7', 'membership', 'normals8', 'membership8', 'membership4', 'normals3', 'kps_un')]


class _FrameBowOutputs(C.Structure):
    _fields_ = [(n, _vp) for n in ('bow_counts', 'bow_words', 'bow_values', 'fv_order', 'fv_counts', 'node_of', 'word_of')]


class _FrameGridOutputs(C.Structure):
    _fields_ = [(n, _vp) for n in ('grid_counts', 'grid_items', 'lgrid_counts', 'lgrid_items')]


class _FrameLpvoOutputs(C.Structure):
    _fields_ = [(n, _vp) for n in ('normals3', 'depth', 'pix2', 'counts')]


def _check_lpvo_stage(lpvo, stages):
    if lpvo and not stages & STAGE_NORMALS:
        raise HvoError(HVO_ERR_ARG, 'lpvo=True needs the normals stage (STAGE_NORMALS)')


class FrameFrontEnd:
    """The extraction part of ORB_SLAM2::Frame::Frame(imGray, imDepth, ...) (reference src/Frame.cc:188-233): ORB + RGB-D
    depth lookup, LSD/LBD lines, PEAC planes and surface normals (and, on request, the LPVO normals) of a batch of frames, on
    concurrent CUDA streams."""
    FIELDS = [f[0] for f in _FrameOutputs._fields_]
    BOW_FIELDS = [f[0] for f in _FrameBowOutputs._fields_]
    GRID_FIELDS = [f[0] for f in _FrameGridOutputs._fields_]
    LPVO_FIELDS = ['lpvo_' + f[0] for f in _FrameLpvoOutputs._fields_]   # output keys; the struct's fields without the prefix
    vocabulary = None
    grids = False
    with_lpvo = False

    def __init__(self, width, height, fx, fy, cx, cy, depth_factor, bf=40.0, nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20,
                 min_th=7, n_lines=200, stages=STAGE_ALL, max_planes=16, max_batch=1, device=0, line_cull=False, lanes=0, membership='i32',
                 distorted=False, normals='n8', dist=None, vocabulary=None, levelsup=4, grids=False, lpvo=False):
        """membership: 'i32' (int32 labels, -1 = none), 'u8' (one byte per pixel, 255 = none: what a host caller needs to
        rebuild plane_vertices_), 'both', or 'u4' (host calls only: two pixels per byte, 15 = none, max_planes <= 15; expand with
        membership4_expand).  The int32 image is always the device-side working image.
        normals: 'n8' (SurfaceNormal rows: normal, position, pixel) or 'n3' (host calls only: the normal alone; normals3_expand
        rebuilds the rows from the depth image).
        dist: mDistCoef (k1, k2, p1, p2 [, k3]).  With a non-zero coefficient the handle runs Frame::UndistortKeyPoints on the device:
        kp_uright is formed from the undistorted keypoints and the outputs gain kps_un (mvKeysUn).
        vocabulary: the dict ORBVocabulary takes.  Every frame then also gets what Frame::ComputeBoW computes, transform(mDescriptors,
        mBowVec, mFeatVec, levelsup), on the device right after its descriptors: the outputs gain the BoW arrays (see bow()).
        grids: every frame also gets Frame::AssignFeaturesToGrid / AssignFeaturesToGridForLine (mGrid, mGridForLine) with the handle's
        image_bounds(): the outputs gain grid_counts / grid_items (ORB stage) and lgrid_counts / lgrid_items (line stage), see grid().
        lpvo: every frame also gets Manhattan::computeNormalsLPVO (what Frame::Frame runs while !bManhInit) after its surface normals:
        the outputs gain lpvo_normals3 / lpvo_depth / lpvo_pix2 / lpvo_counts, see lpvo().  Needs the normals stage."""
        assert membership in ('i32', 'u8', 'both', 'u4') and normals in ('n8', 'n3')
        _check_lpvo_stage(lpvo, stages)
        self.membership_mode, self.normals_mode = membership, normals
        self.cam = (float(fx), float(fy), float(cx), float(cy), float(np.float32(depth_factor)))
        prm = self._params(fx, fy, cx, cy, depth_factor, bf, nfeatures, scale_factor, nlevels, ini_th, min_th, n_lines, stages, max_planes,
                           line_cull, lanes, distorted, dist)
        out = _vp()
        _check(lib().hvo_frame_create(C.byref(prm), int(width), int(height), int(max_batch), int(device), C.byref(out)))
        self._h = out
        self.w, self.h, self.max_batch, self.stages, self.max_planes = int(width), int(height), int(max_batch), stages, max_planes
        a, b, c = C.c_int(0), C.c_int(0), C.c_int(0)
        _check(lib().hvo_frame_capacities(out, C.byref(a), C.byref(b), C.byref(c)))
        self.orb_capacity, self.max_lines, self.normals_count = a.value, b.value, c.value
        _check(lib().hvo_frame_lanes(out, C.byref(a), C.byref(b)))
        self.lanes, self.chunk = a.value, b.value
        self.grids, self.line_grid_capacity = bool(grids), lib().hvo_frame_line_grid_capacity(out)
        self.with_lpvo, self.lpvo_capacity = bool(lpvo), lib().hvo_frame_lpvo_capacity(out)
        if vocabulary is not None:
            self.set_vocabulary(vocabulary, levelsup)

    def set_vocabulary(self, vocabulary, levelsup=4):
        """Attach a vocabulary (the dict ORBVocabulary takes) or, with None, detach it (hvo_frame_set_vocabulary / hvo_seq_set_vocabulary)."""
        f, h = (lib().hvo_seq_set_vocabulary, self._seq) if getattr(self, '_seq', None) else (lib().hvo_frame_set_vocabulary, self._h)
        self.vocabulary = None
        if vocabulary is None:
            _check(f(h, 0, None, None, None, None, None, 0, 0))
            return
        args, _keep = _vocabulary_args(vocabulary)
        _check(f(h, *args, int(levelsup)))
        self.vocabulary, self.levelsup = vocabulary, int(levelsup)

    def image_bounds(self):
        """(mnMinX, mnMaxX, mnMinY, mnMaxY) the grids are built with (hvo_frame_image_bounds), float32 as module-level image_bounds()."""
        f, h = (lib().hvo_seq_image_bounds, self._seq) if getattr(self, '_seq', None) else (lib().hvo_frame_image_bounds, self._h)
        v = [C.c_float(0) for _ in range(4)]
        _check(f(h, *[C.byref(a) for a in v]))
        return tuple(np.float32(a.value) for a in v)

    def _params(self, fx, fy, cx, cy, depth_factor, bf, nfeatures, scale_factor, nlevels, ini_th, min_th, n_lines, stages, max_planes,
                line_cull, lanes, distorted, dist):
        d5 = _dist5(dist) if dist is not None else np.zeros(5, np.float32)
        self.undistorts = bool(d5.any())
        return _FrameParams(_OrbParams(nfeatures, scale_factor, nlevels, ini_th, min_th), _LineParams(1, 1.2, n_lines, 0.125),
                            fx, fy, cx, cy, float(np.float32(depth_factor)), bf, int(bool(distorted) or self.undistorts), stages, max_planes,
                            int(bool(line_cull)), int(lanes), *[float(v) for v in d5])

    def close(self):
        if getattr(self, '_h', None):
            lib().hvo_frame_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def output_shapes(self, n, device=True):
        """name -> (shape, numpy dtype) of every output of an n-frame batch (for the selected stages); device=False
        leaves out the int32 membership image when the handle reports labels as bytes."""
        sh = {}
        if self.stages & STAGE_ORB:
            c = self.orb_capacity
            sh.update(kps=((n, c), KP_DTYPE), desc=((n, c, 32), np.uint8), kp_counts=((n,), np.int32), kp_depth=((n, c), np.float32),
                      kp_uright=((n, c), np.float32))
            if self.undistorts:
                sh.update(kps_un=((n, c), KP_DTYPE))
            if self.vocabulary is not None:
                sh.update(bow_counts=((n,), np.int32), bow_words=((n, c), np.int32), bow_values=((n, c), np.float64), fv_order=((n, c), np.int32),
                          fv_counts=((n,), np.int32), node_of=((n, c), np.int32), word_of=((n, c), np.int32))
            if self.grids:
                sh.update(grid_counts=((n, 64 * 48), np.uint16), grid_items=((n, c), np.uint16))
        if self.stages & STAGE_LINES:
            c = self.max_lines
            sh.update(keylines=((n, c), KL_DTYPE), line_desc=((n, c, 32), np.uint8), linevec3=((n, c, 3), np.float64),
                      line_counts=((n,), np.int32))
            if self.grids:
                sh.update(lgrid_counts=((n, 64 * 48), np.uint16), lgrid_items=((n, self.line_grid_capacity), np.uint16))
        if self.stages & STAGE_PLANES:
            sh.update(n_planes=((n,), np.int32), planes7=((n, self.max_planes, 7), np.float64))
            if device or self.membership_mode in ('i32', 'both'):
                sh.update(membership=((n, self.h * self.w), np.int32))
            if self.membership_mode in ('u8', 'both') or (device and self.membership_mode == 'u4'):
                sh.update(membership8=((n, self.h * self.w), np.uint8))
            if self.membership_mode == 'u4' and not device:
                sh.update(membership4=((n, self.h * self.w // 2), np.uint8))
        if self.stages & STAGE_NORMALS:
            if device or self.normals_mode == 'n8':
                sh.update(normals8=((n, self.normals_count, 8), np.float32))
            else:
                sh.update(normals3=((n, self.normals_count, 3), np.float32))
            if self.with_lpvo:
                c = self.lpvo_capacity
                sh.update(lpvo_normals3=((n, c, 3), np.float64), lpvo_depth=((n, c), np.float32), lpvo_pix2=((n, c, 2), np.int32),
                          lpvo_counts=((n,), np.int32))
        return sh

    @staticmethod
    def membership4_expand(labels4):
        """[.., H*W/2] uint8 -> [.., H*W] int32 labels (-1 = none): hvo_membership4_expand."""
        a = np.ascontiguousarray(labels4, np.uint8)
        out = np.empty(a.shape[:-1] + (a.shape[-1] * 2,), np.int32)
        for i in range(int(np.prod(a.shape[:-1], dtype=np.int64))):
            _check(lib().hvo_membership4_expand(_vp(a.reshape(-1, a.shape[-1])[i].ctypes.data), a.shape[-1] * 2,
                                                _vp(out.reshape(-1, out.shape[-1])[i].ctypes.data)))
        return out

    def normals3_expand(self, normals3, depth16):
        """normals3 [count,3] of one frame + its raw depth -> normals8 [count,8] (hvo_normals3_expand)."""
        n3 = np.ascontiguousarray(normals3, np.float32)
        d = np.ascontiguousarray(depth16, np.uint16)
        out = np.empty((len(n3), 8), np.float32)
        fx, fy, cx, cy, df = self.cam
        _check(lib().hvo_normals3_expand(_np_ptr(n3), _np_ptr(d), self.w, self.h, fx, fy, cx, cy, df, _np_ptr(out)))
        return out

    def alloc_host(self, n):
        return {k: np.empty(s, d) for k, (s, d) in self.output_shapes(n, device=False).items()}

    def _outputs(self, ptrs):
        o = _FrameOutputs()
        for k in self.FIELDS:
            setattr(o, k, ptrs.get(k))
        return o

    def _bow_outputs(self, ptrs):
        """hvo_frame_bow_outputs by reference, or None without a vocabulary (the call then computes no BoW)."""
        if self.vocabulary is None:
            return None
        o = _FrameBowOutputs()
        for k in self.BOW_FIELDS:
            setattr(o, k, ptrs.get(k))
        return C.byref(o)

    def _grid_outputs(self, ptrs):
        """hvo_frame_grid_outputs by reference, or None for a handle created without grids."""
        if not self.grids:
            return None
        o = _FrameGridOutputs()
        for k in self.GRID_FIELDS:
            setattr(o, k, ptrs.get(k))
        return C.byref(o)

    def _lpvo_outputs(self, ptrs):
        """hvo_frame_lpvo_outputs by reference, or None for a handle created without lpvo."""
        if not self.with_lpvo:
            return None
        o = _FrameLpvoOutputs()
        for k in self.LPVO_FIELDS:
            setattr(o, k[5:], ptrs.get(k))
        return C.byref(o)

    @staticmethod
    def lpvo(out, f):
        """Frame f's LPVO normals: (pt_normals [m,3] float64, depth_normals [m] float32, pixels (u, v) [m,2] int32), the form of
        Manhattan.computeNormalsLPVO."""
        m = int(out['lpvo_counts'][f])
        return out['lpvo_normals3'][f, :m].copy(), out['lpvo_depth'][f, :m].copy(), out['lpvo_pix2'][f, :m].copy()

    @staticmethod
    def _cells(counts, items, f):
        c = np.asarray(counts[f], np.int32)
        return c, np.asarray(items[f, :int(c.sum())], np.int32)

    @staticmethod
    def grid(out, f):
        """Frame f's mGrid: (counts int32 [3072], items int32), cell = ix * 48 + iy, the form of oracle.grid_build."""
        return FrameFrontEnd._cells(out['grid_counts'], out['grid_items'], f)

    @staticmethod
    def line_grid(out, f):
        """Frame f's mGridForLine: (counts int32 [3072], items int32), the form of oracle.line_grid_build."""
        return FrameFrontEnd._cells(out['lgrid_counts'], out['lgrid_items'], f)

    @staticmethod
    def bow(out, f):
        """Frame f's mBowVec / mFeatVec from the outputs of a handle with a vocabulary: ((words, values), {node: [feature, ...]}), the
        form of ORBVocabulary.transform()[:2]."""
        nw, nf = int(out['bow_counts'][f]), int(out['fv_counts'][f])
        fv = {}
        for i in out['fv_order'][f, :nf]:
            fv.setdefault(int(out['node_of'][f, i]), []).append(int(i))
        return (out['bow_words'][f, :nw].copy(), out['bow_values'][f, :nw].copy()), fv

    def extract_batch(self, gray, depth16, out=None, wait=True):
        """gray [n,h,w] uint8, depth16 [n,h,w] uint16 (host) -> dict of host arrays (see output_shapes).  wait=False queues the
        call and returns (pinned buffers, untouched until sync()): the next call's uploads overlap this call's tail."""
        gray = np.ascontiguousarray(gray, np.uint8)
        depth16 = np.ascontiguousarray(depth16, np.uint16)
        n = len(gray)
        if gray.ndim != 3 or gray.shape[1:] != (self.h, self.w) or depth16.shape != gray.shape:
            raise HvoError(HVO_ERR_ARG, f'gray / depth16 must be [n, {self.h}, {self.w}] (got {gray.shape}, {depth16.shape})')
        if out is None:
            out = self.alloc_host(n)
        else:   # the C side writes through raw pointers: every caller-supplied array must have the exact layout
            self._check_out(out, self.output_shapes(n, device=False))
        ptrs = {k: v.ctypes.data for k, v in out.items()}
        o = self._outputs(ptrs)
        f = lib().hvo_frame_extract_batch_lpvo if wait else lib().hvo_frame_extract_batch_async_lpvo
        _check(f(self._h, _np_ptr(gray), _np_ptr(depth16), n, C.byref(o), self._bow_outputs(ptrs), self._grid_outputs(ptrs), self._lpvo_outputs(ptrs)))
        return out

    @staticmethod
    def _check_out(out, shapes):
        for k, (shape, dt) in shapes.items():
            a = out.get(k)
            if a is None or a.shape != tuple(shape) or a.dtype != np.dtype(dt) or not a.flags.c_contiguous:
                raise HvoError(HVO_ERR_ARG, f'out[{k!r}] must be a C-contiguous {np.dtype(dt)} array of shape {tuple(shape)}')

    def extract_batch_device(self, d_gray, d_depth16, n, d_ptrs):
        """d_ptrs: name -> device pointer (int) for every output of output_shapes(n).  Asynchronous."""
        o = self._outputs(d_ptrs)
        _check(lib().hvo_frame_extract_batch_device_lpvo(self._h, _vp(d_gray), _vp(d_depth16), n, C.byref(o), self._bow_outputs(d_ptrs),
                                                         self._grid_outputs(d_ptrs), self._lpvo_outputs(d_ptrs)))

    def last_launches(self):
        return lib().hvo_frame_last_launches(self._h)

    def sync(self):
        _check(lib().hvo_frame_sync(self._h))

    def timer_start(self):
        _check(lib().hvo_frame_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(lib().hvo_frame_timer_stop(self._h, C.byref(ms)))
        return ms.value


class FrameSequence(FrameFrontEnd):
    """Offline sequences on several GPUs of one box from one process (hvo_seq_*): the frames of a call are partitioned across
    `devices` in contiguous ranges, one host thread + one frame handle per device, every device writes its rows of the caller's host
    arrays.  No NCCL.  The Python mirror of a loop of Frame constructions over a recorded sequence."""

    def __init__(self, width, height, fx, fy, cx, cy, depth_factor, devices, frames_per_call=2368, bf=40.0, nfeatures=1000, scale_factor=1.2,
                 nlevels=8, ini_th=20, min_th=7, n_lines=200, stages=STAGE_ALL, max_planes=15, line_cull=True, lanes=0, membership='u4',
                 normals='n3', distorted=False, dist=None, vocabulary=None, levelsup=4, grids=False, lpvo=False):
        assert membership in ('i32', 'u8', 'both', 'u4') and normals in ('n8', 'n3')
        _check_lpvo_stage(lpvo, stages)
        self.membership_mode, self.normals_mode = membership, normals
        self.cam = (float(fx), float(fy), float(cx), float(cy), float(np.float32(depth_factor)))
        prm = self._params(fx, fy, cx, cy, depth_factor, bf, nfeatures, scale_factor, nlevels, ini_th, min_th, n_lines, stages, max_planes,
                           line_cull, lanes, distorted, dist)
        dev = (C.c_int * len(devices))(*[int(d) for d in devices])
        out = _vp()
        _check(lib().hvo_seq_create(C.byref(prm), int(width), int(height), dev, len(devices), int(frames_per_call), C.byref(out)))
        self._h = None          # not a frame handle: FrameFrontEnd.close() must not touch it
        self._seq = out
        self.devices = list(devices)
        self.w, self.h, self.max_batch, self.stages, self.max_planes = int(width), int(height), int(frames_per_call), stages, max_planes
        a, b, c = C.c_int(0), C.c_int(0), C.c_int(0)
        _check(lib().hvo_seq_capacities(out, C.byref(a), C.byref(b), C.byref(c)))
        self.orb_capacity, self.max_lines, self.normals_count = a.value, b.value, c.value
        self.grids, self.line_grid_capacity = bool(grids), lib().hvo_seq_line_grid_capacity(out)
        self.with_lpvo, self.lpvo_capacity = bool(lpvo), lib().hvo_seq_lpvo_capacity(out)
        if vocabulary is not None:
            self.set_vocabulary(vocabulary, levelsup)

    def close(self):
        if getattr(self, '_seq', None):
            lib().hvo_seq_destroy(self._seq)
            self._seq = None

    @staticmethod
    def shard(nframes, ndevices, d):
        a, b = C.c_int(0), C.c_int(0)
        lib().hvo_seq_shard(int(nframes), int(ndevices), int(d), C.byref(a), C.byref(b))
        return a.value, b.value

    def extract(self, gray, depth16, out=None):
        """gray [n,h,w] uint8, depth16 [n,h,w] uint16 (host, ideally pinned) -> dict of host arrays in frame order."""
        gray = np.ascontiguousarray(gray, np.uint8)
        depth16 = np.ascontiguousarray(depth16, np.uint16)
        n = len(gray)
        if gray.ndim != 3 or gray.shape[1:] != (self.h, self.w) or depth16.shape != gray.shape:
            raise HvoError(HVO_ERR_ARG, f'gray / depth16 must be [n, {self.h}, {self.w}]')
        if out is None:
            out = self.alloc_host(n)
        else:   # kps_un, the BoW, grid and LPVO arrays at least: the other arrays' check is a separate change
            self._check_out(out, {k: v for k, v in self.output_shapes(n, device=False).items()
                                  if k == 'kps_un' or k in self.BOW_FIELDS or k in self.GRID_FIELDS or k in self.LPVO_FIELDS})
        ptrs = {k: v.ctypes.data for k, v in out.items()}
        o = self._outputs(ptrs)
        _check(lib().hvo_seq_extract_lpvo(self._seq, _np_ptr(gray), _np_ptr(depth16), n, C.byref(o), self._bow_outputs(ptrs),
                                          self._grid_outputs(ptrs), self._lpvo_outputs(ptrs)))
        return out

    def last_ms(self):
        return float(lib().hvo_seq_last_ms(self._seq))
