"""ctypes binding of ``libiqw_b200.so`` (C-ABI declared in ``include/iqw_b200.h``).

There is no CPU fallback: if the CUDA library is missing, or a symbol the header declares is not
exported, importing this module raises and every public function of the package is unusable.
"""
from __future__ import annotations

import ctypes
import os

import torch  # noqa: F401  (loads libcudart.so.12 first so the library binds to the same runtime)

_HERE = os.path.dirname(os.path.abspath(__file__))
# IQW_B200_LIB: another build of the same library (kernel experiments, tools/build_variant.sh)
LIB_PATH = os.environ.get('IQW_B200_LIB') or os.path.join(_HERE, 'libiqw_b200.so')

ABI_VERSION = 13

# statuses / enums mirrored from include/iqw_b200.h
IQW_OK = 0
IQW_ERR_INVALID = -1
IQW_ERR_UNSUPPORTED = -2
IQW_ERR_CUDA = -3
IQW_ERR_WORKSPACE = -4

STFT_COMPLEX, STFT_POWER, STFT_DB = 0, 1, 2
STAT_QUANTILE, STAT_MEAN, STAT_MAX, STAT_MIN, STAT_MEDIAN, STAT_ORDER = 0, 1, 2, 3, 4, 5
EW_POWTODB, EW_DBTOPOW, EW_ENVTOPOW, EW_ENVTODB = 0, 1, 2, 3

MAX_RANKS_PER_CALL = 8


class iqw_stat(ctypes.Structure):
    _fields_ = [
        ('kind', ctypes.c_int32),
        ('rank_lo', ctypes.c_int64),
        ('rank_hi', ctypes.c_int64),
        ('gamma', ctypes.c_float),
    ]


_i32, _i64, _f32, _vp, _sz = (ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p,
                              ctypes.c_size_t)

# name -> (restype, argtypes); must list every function include/iqw_b200.h declares
SIGNATURES = {
    'iqw_abi_version': (ctypes.c_int, []),
    'iqw_last_error': (ctypes.c_char_p, []),
    'iqw_stft_workspace_bytes': (_sz, [_i32, _i64, _i64]),
    'iqw_stft_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _vp, _i32, _i64, _i64, _i32, _f32,
                                    _i32, _i32, _vp, _i64, _vp, _sz, _vp]),
    'iqw_stft_bluestein_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _i32, _i32, _i64, _i64, _i32, _f32,
                                              _i32, _i32, _vp, _i64, _vp]),
    'iqw_bluestein_pre_c64': (ctypes.c_int, [_vp, _i64, _vp, _i32, _i32, _i64, _vp, _vp]),
    'iqw_bluestein_mul_c64': (ctypes.c_int, [_vp, _vp, _i32, _i64, _vp]),
    'iqw_bluestein_post_c64': (ctypes.c_int, [_vp, _vp, _i32, _i64, _i32, _f32, _i32, _i32, _vp, _vp]),
    'iqw_stft_reduce_workspace_bytes': (_sz, [_i32]),
    'iqw_stft_reduce_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _vp, _i32, _i64, _i64, _i32, _f32, _i32, _i32,
                                           ctypes.POINTER(iqw_stat), _i32, _vp, _vp, _sz, _vp]),
    'iqw_time_stats_workspace_bytes': (_sz, [_i64, _i64, _i64, _i32]),
    'iqw_time_stats_f32': (ctypes.c_int, [_vp, _i64, _i64, _i64, _i64, ctypes.POINTER(iqw_stat),
                                          _i32, _i32, _f32, _vp, _vp, _sz, _vp]),
    'iqw_bin_power_workspace_bytes': (_sz, [_i64, _i64, _i64]),
    'iqw_bin_power_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    'iqw_envtopow_transposed_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _i64, _vp, _vp]),
    'iqw_elementwise_f32': (ctypes.c_int, [_i32, _vp, _vp, _i64, _i32, _f32, _vp]),
    'iqw_elementwise_c64': (ctypes.c_int, [_i32, _vp, _vp, _i64, _f32, _vp]),
    'iqw_transpose_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _vp, _vp]),
    'iqw_istft_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _i32, _i64, _i32, _i32, _i32, _vp, _f32, _vp, _i64, _vp]),
    'iqw_ifft_c64': (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp]),
    'iqw_ola_filter_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _vp, _i32, _i64, _i64, _i32, _i32, _vp, _i64, _vp]),
    'iqw_upfirdn_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _i64, _vp, _i32, _i32, _i32, _i32, _i64, _i64, _vp,
                                       _i64, _vp]),
    'iqw_oaconvolve_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _i64, _vp, _i64, _i32, _i32, _i32, _i64, _i64,
                                          _vp, _i64, _vp]),
    'iqw_pfb_channelize_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _i64, _vp, _i32, _i32, _i32, _i64, _i64,
                                              _vp, _i64, _vp]),
    'iqw_pfb_synthesize_workspace_bytes': (_sz, [_i64, _i64, _i32]),
    'iqw_pfb_synthesize_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _i64, _i64, _vp, _i32, _i32, _i32, _i64, _i64,
                                              _vp, _i64, _vp, _sz, _vp]),
    'iqw_sosfilt_geometry': (ctypes.c_int, [_i32, ctypes.POINTER(_i32)]),
    'iqw_sosfilt_workspace_bytes': (_sz, [_i64, _i64, _i32]),
    'iqw_sosfilt_carry_workspace_bytes': (_sz, [_i64, _i64, _i32]),
    'iqw_sosfilt_states_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _vp, _i32, _vp, _vp, _vp, _sz, _vp]),
    'iqw_sosfilt_carry_c64': (ctypes.c_int, [_vp, _i64, _i64, _vp, _i32, _vp, _vp, _sz, _vp]),
    'iqw_sosfilt_apply_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _vp, _i32, _vp, _vp, _vp, _sz, _vp, _i64, _vp,
                                             _vp]),
    'iqw_sosfilt_c64': (ctypes.c_int, [_vp, _i64, _i64, _i64, _vp, _i32, _vp, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    'iqw_edge_counts_f32': (ctypes.c_int, [_vp, _i64, _i64, _vp, _i32, _i32, _vp, _vp]),
    'iqw_bracket_collect_workspace_bytes': (_sz, [_i64, _i64]),
    'iqw_bracket_collect_f32': (ctypes.c_int, [_vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    'iqw_candidate_count_f32': (ctypes.c_int, [_vp, _i64, _i64, _i32, _vp, _vp, _i32, _vp, _vp]),
    'iqw_radix_count_f32': (ctypes.c_int, [_vp, _i64, _i64, _i32, _vp, _vp, _i32, _vp, _vp, _vp]),
    'iqw_radix_descend': (ctypes.c_int, [_vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp]),
    'iqw_order_stats_finish_f32': (ctypes.c_int, [_vp, _i32, ctypes.POINTER(_i64), _i64, _i64,
                                                  ctypes.POINTER(iqw_stat), _i32, _i32, _f32, _vp, _vp]),
    'iqw_debug_set_stft_scratch_cap': (ctypes.c_int, [_sz]),
    'iqw_debug_set_stft_variant': (ctypes.c_int, [ctypes.c_int]),
    'iqw_debug_set_sample_min_rows': (ctypes.c_int, [_i64]),
    'iqw_debug_set_sample_margin': (ctypes.c_int, [ctypes.c_double, ctypes.c_int]),
    'iqw_debug_time_stats_counters': (ctypes.c_int, [_vp, _i64, ctypes.POINTER(ctypes.c_uint32)]),
    'iqw_profile_enable': (ctypes.c_int, [ctypes.c_int]),
    'iqw_profile_reset': (ctypes.c_int, []),
    'iqw_profile_report': (ctypes.c_int, [ctypes.c_char_p, _sz]),
}


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; '
            f'g.build()"` or `make -C iqwaveform_b200/csrc`.  iqwaveform_b200 has no CPU fallback.'
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise ImportError(f'{LIB_PATH} does not export {name}') from exc
        fn.restype = restype
        fn.argtypes = argtypes
    got = lib.iqw_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f'{LIB_PATH}: ABI version {got}, python layer expects {ABI_VERSION}')
    return lib


lib = _load()


class IQWError(RuntimeError):
    pass


def check(status: int) -> None:
    """map a C status to the exception type the reference raises for the same condition"""
    if status == IQW_OK:
        return
    msg = (lib.iqw_last_error() or b'').decode(errors='replace')
    if status == IQW_ERR_INVALID:
        raise ValueError(msg)
    if status == IQW_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise IQWError(f'iqw status {status}: {msg}')


def profile(on: bool, fine: bool = False) -> None:
    """kernel timing by CUDA events on the launching stream: the heavy kernels one by one and the
    trains of small follow-up kernels as one scope each; `fine=True` times every launch"""
    lib.iqw_profile_reset()
    lib.iqw_profile_enable((2 if fine else 1) if on else 0)


def profile_report() -> dict:
    """{kernel name: (launches, total_ms)}; synchronise the device first"""
    buf = ctypes.create_string_buffer(1 << 16)
    check(lib.iqw_profile_report(buf, len(buf)))
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms = line.split()
        out[name] = (int(n), float(ms))
    return out
