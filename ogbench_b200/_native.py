"""ctypes binding of libogbsampler.so (include/ogb_sampler.h).  There is no CPU fallback: if the library is
missing or no CUDA device is usable, every entry point raises."""

from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

OGB_MAX_NDIM = 6
OGB_MAX_SLOTS = 10

OGB_OK, OGB_ERR_INVALID, OGB_ERR_ASSERT, OGB_ERR_INDEX, OGB_ERR_CUDA, OGB_ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5
KIND_GC, KIND_HGC, KIND_PLAIN, KIND_ATC = 0, 1, 2, 3

_DTYPES = [
    (np.uint8, 0), (np.int8, 1), (np.int16, 2), (np.int32, 3), (np.int64, 4), (np.float16, 5), (np.float32, 6),
    (np.float64, 7), (np.bool_, 8), (np.uint16, 9), (np.uint32, 10), (np.uint64, 11),
]
DTYPE_TO_CODE = {np.dtype(d): c for d, c in _DTYPES}
CODE_TO_DTYPE = {c: np.dtype(d) for d, c in _DTYPES}


class Field(C.Structure):
    _fields_ = [('name', C.c_char_p), ('data', C.c_void_p), ('dtype', C.c_int32), ('ndim', C.c_int32),
                ('shape', C.c_int64 * OGB_MAX_NDIM), ('on_device', C.c_int32)]


class Config(C.Structure):
    _fields_ = [
        ('discount', C.c_double),
        ('value_p_curgoal', C.c_double), ('value_p_trajgoal', C.c_double), ('value_p_randomgoal', C.c_double),
        ('actor_p_curgoal', C.c_double), ('actor_p_trajgoal', C.c_double), ('actor_p_randomgoal', C.c_double),
        ('value_geom_sample', C.c_int32), ('actor_geom_sample', C.c_int32),
        ('gc_negative', C.c_int32),
        ('has_p_aug', C.c_int32), ('p_aug', C.c_double),
        ('frame_stack', C.c_int32), ('crop_padding', C.c_int32),
        ('value_subgoal_steps', C.c_int32), ('actor_subgoal_steps', C.c_int32), ('low_subgoal_steps', C.c_int32),
        ('has_low_discount', C.c_int32), ('low_discount', C.c_double),
        ('lut_len', C.c_int32),
        ('neg_reward_lut', C.POINTER(C.c_double)), ('pow_lut', C.POINTER(C.c_double)),
        ('dedup_keys', C.c_int32),
        ('trl', C.c_int32),
        ('jax_compat', C.c_int32), ('pad_', C.c_int32),
    ]


class GoalDraws(C.Structure):
    _fields_ = [('rand_pos', C.c_void_p), ('offset', C.c_void_p), ('dist', C.c_void_p), ('u_traj', C.c_void_p),
                ('u_cur', C.c_void_p)]


class Draws(C.Structure):
    _fields_ = [('idx_pos', C.c_void_p), ('goals', GoalDraws * 3), ('has_aug_coin', C.c_int32),
                ('aug_coin', C.c_double), ('crop', C.c_void_p), ('trl_midpoints', C.c_void_p)]


class KeyInfo(C.Structure):
    _fields_ = [('name', C.c_char_p), ('dtype', C.c_int32), ('ndim', C.c_int32), ('shape', C.c_int64 * (OGB_MAX_NDIM + 1)),
                ('device_ptr', C.c_void_p), ('nbytes', C.c_size_t), ('offset', C.c_size_t), ('alias_of', C.c_int32)]


class TableInfo(C.Structure):
    _fields_ = [('valid_mode', C.c_int32), ('seg_shift', C.c_int32), ('n_seg_table', C.c_int32), ('gap_shift', C.c_int32),
                ('term_shift', C.c_int32), ('pad_', C.c_int32), ('n_choices', C.c_int64)]


class NativeError(RuntimeError):
    pass


_LIB = None

# every symbol include/ogb_sampler.h declares: (name, restype, argtypes)
_P = C.c_void_p
SIGNATURES = [
    ('ogb_last_error', C.c_char_p, []),
    ('ogb_abi_version', C.c_int, []),
    ('ogb_device_count', C.c_int, [C.POINTER(C.c_int)]),
    ('ogb_dataset_create', C.c_int, [C.POINTER(Field), C.c_int32, C.c_int32, C.POINTER(_P)]),
    ('ogb_dataset_size', C.c_int, [_P, C.POINTER(C.c_int64)]),
    ('ogb_dataset_num_valid', C.c_int, [_P, C.POINTER(C.c_int64)]),
    ('ogb_dataset_set_active_rows', C.c_int, [_P, C.c_int64]),
    ('ogb_dataset_resident_bytes', C.c_int, [_P, C.POINTER(C.c_size_t)]),
    ('ogb_dataset_destroy', C.c_int, [_P]),
    ('ogb_dataset_create_empty', C.c_int, [C.POINTER(Field), C.c_int32, C.c_int32, C.POINTER(_P)]),
    ('ogb_dataset_write_rows', C.c_int, [_P, C.c_int64, C.c_int64, C.POINTER(C.c_void_p), C.c_int32]),
    ('ogb_dataset_seal', C.c_int, [_P, C.c_int64]),
    ('ogb_dataset_view', C.c_int, [_P, C.c_int64, C.c_int64, C.POINTER(_P)]),
    ('ogb_sampler_create', C.c_int, [_P, C.POINTER(Config), C.c_int32, C.c_uint64, C.c_uint32, C.POINTER(_P)]),
    ('ogb_sampler_set_stream', C.c_int, [_P, _P]),
    ('ogb_sampler_set_debug', C.c_int, [_P, C.c_int32]),
    ('ogb_sampler_set_profile', C.c_int, [_P, C.c_int32]),
    ('ogb_sampler_set_deferred_index_check', C.c_int, [_P, C.c_int32]),
    ('ogb_sampler_set_host_chunks', C.c_int, [_P, C.c_int32]),
    ('ogb_sampler_num_choices', C.c_int, [_P, C.POINTER(C.c_int64)]),
    ('ogb_sampler_num_terminals', C.c_int, [_P, C.POINTER(C.c_int64)]),
    ('ogb_sampler_write_row', C.c_int, [_P, C.c_int64, C.POINTER(C.c_void_p), C.c_int32]),
    ('ogb_sampler_write_ring', C.c_int, [_P, C.c_int64, C.c_int64, C.c_int64, C.POINTER(C.c_void_p), C.c_int32,
                                         C.POINTER(C.c_int32), _P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    ('ogb_sampler_get_stream', C.c_int, [_P, C.POINTER(_P)]),
    ('ogb_sampler_copy_bounds', C.c_int, [_P, _P, _P]),
    ('ogb_sampler_table_info', C.c_int, [_P, C.POINTER(TableInfo)]),
    ('ogb_sampler_get_counter', C.c_int, [_P, C.POINTER(C.c_uint64)]),
    ('ogb_sampler_set_counter', C.c_int, [_P, C.c_uint64]),
    ('ogb_sampler_destroy', C.c_int, [_P]),
    ('ogb_sampler_sample', C.c_int, [_P, C.c_int64, C.c_int32, _P, C.c_int32, C.POINTER(Draws), C.POINTER(_P)]),
    ('ogb_sampler_gather', C.c_int, [_P, C.c_int32, _P, C.c_int64, C.POINTER(_P)]),
    ('ogb_sampler_gather_cropped', C.c_int, [_P, _P, C.c_int64, _P, C.c_int32, C.POINTER(_P)]),
    ('ogb_sampler_sample_goals', C.c_int, [_P, _P, C.c_int64, C.c_double, C.c_double, C.c_int32, C.c_double, _P, _P]),
    ('ogb_sampler_compute_high_next_idxs', C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int64, _P, _P]),
    ('ogb_sampler_num_atc_anchors', C.c_int, [_P, C.c_int64, C.POINTER(C.c_int64)]),
    ('ogb_sampler_copy_atc_anchors', C.c_int, [_P, C.c_int64, _P]),
    ('ogb_sampler_sample_atc', C.c_int, [_P, C.c_int64, C.c_int32, C.c_int64, C.c_int32, C.POINTER(Draws), C.POINTER(_P)]),
    ('ogb_batch_num_keys', C.c_int, [_P, C.POINTER(C.c_int32)]),
    ('ogb_batch_key_info', C.c_int, [_P, C.c_int32, C.POINTER(KeyInfo)]),
    ('ogb_batch_nbytes', C.c_int, [_P, C.POINTER(C.c_size_t)]),
    ('ogb_batch_device_block', C.c_int, [_P, C.POINTER(_P)]),
    ('ogb_batch_launches', C.c_int, [_P, C.POINTER(C.c_int32)]),
    ('ogb_batch_kernel_names', C.c_int, [_P, C.POINTER(C.c_char_p), C.c_int32, C.POINTER(C.c_int32)]),
    ('ogb_batch_dominant_kernel', C.c_int, [_P, _P, _P]),
    ('ogb_batch_keep_leading_axis', C.c_int, [_P, C.c_int32]),
    ('ogb_batch_sync', C.c_int, [_P]),
    ('ogb_batch_wait_on_stream', C.c_int, [_P, _P]),
    ('ogb_batch_copy_to_host', C.c_int, [_P, _P, C.c_size_t]),
    ('ogb_batch_copy_to_host_begin', C.c_int, [_P, _P, C.c_size_t]),
    ('ogb_batch_copy_to_host_end', C.c_int, [_P]),
    ('ogb_batch_copy_key_to_host', C.c_int, [_P, C.c_int32, _P, C.c_size_t]),
    ('ogb_batch_copy_slice_to_host', C.c_int, [_P, C.c_int32, C.c_int64, _P, C.c_size_t]),
    ('ogb_batch_check_gaps', C.c_int, [_P, _P]),
    ('ogb_batch_index_vector', C.c_int, [_P, C.c_int32, _P]),
    ('ogb_batch_crop_shifts', C.c_int, [_P, _P]),
    ('ogb_batch_dlpack', C.c_int, [_P, C.c_int32, C.POINTER(_P)]),
    ('ogb_batch_dlpack_slice', C.c_int, [_P, C.c_int32, C.c_int64, C.POINTER(_P)]),
    ('ogb_batch_mark_escaped', C.c_int, [_P]),
    ('ogb_batch_retain', C.c_int, [_P]),
    ('ogb_batch_release', C.c_int, [_P]),
    ('ogb_host_alloc', C.c_int, [C.c_size_t, C.POINTER(_P)]),
    ('ogb_host_free', C.c_int, [_P]),
    ('ogb_searchsorted_warp', C.c_int, [_P, C.c_int64, _P, C.c_int64, C.c_int32, C.c_int32, _P]),
    ('ogb_philox_fill', C.c_int, [C.c_uint64, C.c_uint32, C.c_uint64, C.c_uint32, C.c_int64, C.c_int32, _P]),
    ('ogb_debug_timeline', C.c_int, [_P, C.c_int32, _P]),
    ('ogb_geometric_check', C.c_int, [C.c_double, C.c_uint64, C.c_int64, C.c_int32, _P]),
]


def lib():
    """Load (building first if the .so is missing or stale and nvcc is present) and return the library."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.LIB_PATH
    if _build.is_stale():
        try:
            _build.build()
        except Exception as exc:  # no nvcc on this box: use the shipped .so if there is one
            if not os.path.exists(path):
                raise ImportError(
                    f'libogbsampler.so is missing and could not be built ({exc}); '
                    'run `python -m ogbench_b200.build` on a machine with nvcc. There is no CPU fallback.'
                ) from exc
    handle = C.CDLL(path)
    for name, restype, argtypes in SIGNATURES:
        fn = getattr(handle, name)  # AttributeError here means header and library disagree
        fn.restype = restype
        fn.argtypes = argtypes
    if handle.ogb_abi_version() != 1:
        raise ImportError('libogbsampler.so ABI version mismatch')
    _LIB = handle
    return _LIB


def check(rc: int):
    """Map a status code to the exception type the reference would have raised."""
    if rc == OGB_OK:
        return
    msg = lib().ogb_last_error().decode('utf-8', 'replace')
    if rc == OGB_ERR_ASSERT:
        raise AssertionError(msg)
    if rc == OGB_ERR_INDEX:
        raise IndexError(msg)
    if rc == OGB_ERR_INVALID:
        if msg.startswith('KeyError'):
            raise KeyError(msg.split(':', 1)[1].strip().strip("'"))
        raise ValueError(msg)
    if rc == OGB_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise NativeError(msg)


def device_count() -> int:
    n = C.c_int(0)
    rc = lib().ogb_device_count(C.byref(n))
    return n.value if rc == 0 else 0


def require_device():
    if device_count() < 1:
        raise NativeError('no CUDA device is visible; the sampler has no CPU fallback: '
                          + lib().ogb_last_error().decode('utf-8', 'replace'))
