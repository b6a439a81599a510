"""ctypes binding of libbpv.so (include/bpv.h).  No fallback: if the library is missing or a call
fails, this raises — the product path never routes around the CUDA kernels."""
from __future__ import annotations

import ctypes as C
import os

PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(PKG, 'libbpv.so')

NO_BOX = -(2 ** 31)
GREEN, CHROM_GREEN = 0, 1
DIFF_1, DIFF_2, INTERP_LINEAR, INTERP_CUBIC, DETREND_CONST, DETREND_LINEAR, FILTER_BUTTER, FILTER_FIR = range(1, 9)
DFT_RFFT, PGRAM_WELCH, PGRAM_LS = 1, 2, 3
MAX_METHODS = 8


class BpvError(RuntimeError):
    pass


class WindowParams(C.Structure):
    """struct bpv_window_params (include/bpv.h)."""
    _fields_ = [('S', C.c_int32), ('R', C.c_int32), ('cap', C.c_int32), ('window', C.c_int32),
                ('head0', C.c_int64), ('head_step', C.c_int32), ('jobs_per_stream', C.c_int32),
                ('num_methods', C.c_int32), ('methods', C.c_int32 * MAX_METHODS),
                ('transform', C.c_int32), ('butter_order', C.c_int32), ('fir_taps', C.c_int32),
                ('ls_num_freqs', C.c_int32),
                ('butter_min_bw', C.c_double), ('fir_df', C.c_double), ('min_freq', C.c_double), ('max_freq', C.c_double)]


_P = C.c_void_p
_SIGS = {
    'bpv_version': (C.c_int, []),
    'bpv_last_error': (C.c_char_p, []),
    'bpv_sizeof_window_params': (C.c_int, []),
    'bpv_set_l2_fetch_granularity': (C.c_int, [C.c_int]),
    'bpv_get_l2_fetch_granularity': (C.c_int, []),
    'bpv_roi_sample_u8': (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int64, _P, C.c_int32,
                                    C.c_int32, _P, _P, C.c_int64, _P]),
    'bpv_roi_sample_nv12': (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int64, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    'bpv_roi_sample_resized_u8': (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64, _P,
                                            C.c_int32, C.c_int32, _P, _P, _P]),
    'bpv_roi_sample_masked_u8': (C.c_int, [_P, C.c_int64, C.c_int64, _P, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int64, _P,
                                           C.c_int32, _P, C.c_int32, _P, _P, _P]),
    'bpv_calc_rois': (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P, _P, _P]),
    'bpv_running_mean': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int32, _P, C.c_double, _P, _P, _P]),
    'bpv_view_boxes': (C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    'bpv_pack_records': (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P]),
    'bpv_pack_records32': (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P]),
    'bpv_scratch_discard': (C.c_int, [_P, C.c_int64, _P]),
    'bpv_dft256_tc': (C.c_int, [_P, C.c_int32, _P, _P]),
    'bpv_ring_push': (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int32, _P, _P, _P]),
    'bpv_ring_push_ragged': (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, C.c_int32, _P, _P, _P]),
    'bpv_stream_jobs': (C.c_int, [C.c_int32, _P, _P, C.c_int32, C.c_int64, _P, _P, _P, _P, _P]),
    'bpv_running_mean_jobs': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, C.c_double, _P, _P, _P]),
    'bpv_window_workspace_bytes': (C.c_int64, [C.POINTER(WindowParams)]),
    'bpv_window_preprocess': (C.c_int, [_P, _P, C.POINTER(WindowParams), _P, C.c_int64, _P, _P, _P, _P]),
    'bpv_design_cache_bytes': (C.c_int64, []),
    'bpv_window_design': (C.c_int, [_P, C.POINTER(WindowParams), _P, C.c_int64, _P, C.c_int64, _P]),
    'bpv_window_filter': (C.c_int, [_P, _P, C.POINTER(WindowParams), _P, C.c_int64, _P, C.c_int64, _P, _P, _P, _P]),
    'bpv_window_design_jobs': (C.c_int, [_P, C.POINTER(WindowParams), _P, C.c_int64, _P, C.c_int64, _P, _P, C.c_int64, _P]),
    'bpv_window_filter_jobs': (C.c_int, [_P, _P, C.POINTER(WindowParams), _P, C.c_int64, _P, C.c_int64, _P, _P, _P, _P, _P,
                                         C.c_int64, _P]),
    'bpv_window_preprocess_jobs': (C.c_int, [_P, _P, C.POINTER(WindowParams), _P, C.c_int64, _P, _P, _P, _P, _P, C.c_int64, _P]),
    'bpv_probe_fma': (C.c_int64, [C.c_int32, C.c_int64, C.c_int32, _P, _P]),
    'bpv_spectrum_workspace_bytes': (C.c_int64, [C.POINTER(WindowParams), C.c_int32]),
    'bpv_window_spectrum': (C.c_int, [_P, _P, C.POINTER(WindowParams), C.c_int32, _P, C.c_int64, _P, _P, _P, _P, _P, _P, _P]),
    'bpv_window_xcorr': (C.c_int, [_P, _P, C.POINTER(WindowParams), _P, _P, _P, _P, _P, _P, _P]),
    'bpv_window_spectrum_band': (C.c_int, [_P, _P, C.POINTER(WindowParams), C.c_int32, _P, C.c_int64, _P, _P, _P, _P, _P, _P,
                                           C.c_double, C.c_double, _P]),
    'bpv_window_xcorr_band': (C.c_int, [_P, _P, C.POINTER(WindowParams), _P, _P, _P, _P, _P, _P, C.c_double, C.c_double, _P]),
    'bpv_window_welch_xcorr': (C.c_int, [_P, _P, C.POINTER(WindowParams), C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'bpv_butter_sos_design': (C.c_int, [_P, C.c_int32, C.POINTER(WindowParams), _P, _P]),
    'bpv_firls_design': (C.c_int, [_P, C.c_int32, C.POINTER(WindowParams), _P, _P]),
}
EXPORTS = tuple(_SIGS)

_lib = None


def lib():
    """Load libbpv.so once.  Raises BpvError if it has not been built (python -m bpv.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BpvError(f'{LIB_PATH} not found: build it with `python -m bpv.build` '
                           '(there is no CPU fallback for the signal path)')
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        if l.bpv_sizeof_window_params() != C.sizeof(WindowParams):
            raise BpvError('bpv_window_params layout mismatch between libbpv.so and the ctypes binding')
        _lib = l
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().bpv_last_error().decode(errors='replace')
        if rc == -2:
            raise NotImplementedError(msg or what)
        raise BpvError(f'{what} failed (rc={rc}): {msg}')


def ptr(t):
    """data_ptr of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_handle(device=None):
    """cudaStream_t of torch's current stream on `device` (default: the current device)."""
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
