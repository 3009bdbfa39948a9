"""ctypes binding of libgdeconv.so (C ABI declared in include/gdeconv.h).

There is no fallback: if the shared library is missing it is built with nvcc (gdeconv/build.py); if that fails
the import fails.  Nothing here or above it computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

ARCH_G, ARCH_U = 0, 1
PREC_FP32_SIMT, PREC_FP16_UMMA, PREC_FP16_SIMT = 0, 1, 2
LLH_GAUSSIAN, LLH_POISSON = 0, 1
SOLVER_RL, SOLVER_WIENER, SOLVER_TIKHONOV_ID, SOLVER_TIKHONOV_LAP = 0, 1, 2, 3
SYNTH_SNR_FIXED, SYNTH_SNR_MIXED = 0, 1
SHAPE_OK, SHAPE_MAXITER, SHAPE_FLUX, SHAPE_MOMENTS, SHAPE_CENTROID = 0, 1, 2, 3, 4
PRECISIONS = {'fp32_simt': PREC_FP32_SIMT, 'fp16_umma': PREC_FP16_UMMA, 'fp16_simt': PREC_FP16_SIMT}

#: every symbol include/gdeconv.h declares (tests/test_abi.py checks the header against this list and the .so)
SYMBOLS = ('gd_version', 'gd_last_error', 'gd_pack_weights', 'gd_free_weights', 'gd_workspace_bytes', 'gd_workspace_init', 'gd_workspace_release',
           'gd_admm_forward', 'gd_resunet_forward', 'gd_subnet_forward', 'gd_fft_solver', 'gd_conv_fft', 'gd_moments_e',
           'gd_launch_count', 'gd_debug_geom', 'gd_debug_tapgemm', 'gd_profile_begin', 'gd_profile_end', 'gd_pack_xdense', 'gd_free_xdense', 'gd_xdense_workspace_bytes',
           'gd_xdense_forward', 'gd_tikhonet_forward', 'gd_admm_forward_xdense', 'gd_psf_to_otf', 'gd_conv_otf', 'gd_max_chunk', 'gd_debug_divmagic', 'gd_synth_batch',
           'gd_adaptive_moments')


class GdTensorDesc(C.Structure):
    _fields_ = [('name', C.c_char_p), ('data', C.c_void_p), ('ndim', C.c_int), ('shape', C.c_int64 * 4)]


def _load():
    path = _build.LIB
    # A stale binary must never load silently: the .so is git-ignored and survives source updates, and struct layouts / packed
    # weight layouts can change without any symbol changing.  The source hash is cheap; rebuild on mismatch (nvcc is part of
    # the image, here and on the GPU box) and fail loudly when that is impossible.
    if not _build.is_current():
        try:
            _build.build()
        except Exception as e:
            raise ImportError(f'libgdeconv.so is missing or older than csrc/ and could not be rebuilt with nvcc: {e}') from e
    lib = C.CDLL(path)
    vp, i, f, sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t
    lib.gd_version.restype = i
    lib.gd_last_error.restype = C.c_char_p
    lib.gd_launch_count.restype = C.c_uint64
    lib.gd_pack_weights.argtypes = [i, i, C.POINTER(GdTensorDesc), i, i, i, C.POINTER(vp)]
    lib.gd_free_weights.argtypes = [vp]
    lib.gd_free_weights.restype = None
    lib.gd_workspace_bytes.argtypes = [i, i, i]
    lib.gd_workspace_bytes.restype = sz
    lib.gd_workspace_init.argtypes = [vp, sz, i, i, i, vp]
    lib.gd_workspace_release.argtypes = [vp]
    lib.gd_workspace_release.restype = None
    lib.gd_admm_forward.argtypes = [vp, i, i, vp, vp, vp, vp, vp, vp, i, vp, sz, vp]
    lib.gd_resunet_forward.argtypes = [vp, vp, vp, i, vp, sz, vp]
    lib.gd_subnet_forward.argtypes = [vp, vp, vp, vp, i, vp]
    lib.gd_fft_solver.argtypes = [i, i, f, vp, vp, vp, vp, i, vp]
    lib.gd_conv_fft.argtypes = [vp, vp, vp, i, i, vp]
    lib.gd_moments_e.argtypes = [vp, vp, i, vp]
    lib.gd_profile_begin.restype = None
    lib.gd_pack_xdense.argtypes = [C.POINTER(GdTensorDesc), i, C.c_char_p, i, C.POINTER(vp)]
    lib.gd_free_xdense.argtypes = [vp]
    lib.gd_free_xdense.restype = None
    lib.gd_xdense_workspace_bytes.argtypes = [i]
    lib.gd_xdense_workspace_bytes.restype = sz
    lib.gd_xdense_forward.argtypes = [vp, vp, vp, i, vp, sz, i, vp]
    lib.gd_tikhonet_forward.argtypes = [vp, i, f, vp, vp, vp, vp, i, vp, sz, i, vp]
    lib.gd_admm_forward_xdense.argtypes = [vp, vp, i, i, vp, vp, vp, vp, vp, vp, i, vp, sz, vp, sz, i, vp]
    lib.gd_psf_to_otf.argtypes = [vp, i, i, i, vp, vp, i, vp]
    lib.gd_conv_otf.argtypes = [vp, i, vp, vp, i, vp]
    lib.gd_synth_batch.argtypes = [C.c_int64, i, C.c_int64, i, f, f, f, vp, vp, vp, vp, vp]
    lib.gd_adaptive_moments.argtypes = [vp, i, f, vp, vp, vp]
    lib.gd_max_chunk.restype = i
    lib.gd_debug_divmagic.argtypes = [C.c_uint, C.c_uint, C.c_uint]
    lib.gd_debug_divmagic.restype = C.c_longlong
    lib.gd_profile_end.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    lib.gd_debug_geom.argtypes = [i, i, C.POINTER(C.c_int * 7)]
    lib.gd_debug_tapgemm.argtypes = [i, i, i, i, i, i, i, vp, vp, vp, vp]
    for name in SYMBOLS:
        getattr(lib, name)          # AttributeError here = the .so does not match the header
    want = _header_version()
    if want is not None and lib.gd_version() != want:
        raise ImportError(f'libgdeconv.so reports version {lib.gd_version()}, include/gdeconv.h declares {want}')
    return lib


def _header_version():
    import re
    try:
        text = open(os.path.join(os.path.dirname(_build.PKG), 'include', 'gdeconv.h')).read()
    except OSError:
        return None
    m = re.search(r'#define\s+GD_VERSION\s+(\d+)', text)
    return int(m.group(1)) if m else None


lib = _load()
LIB_PATH = _build.LIB


def check(rc):
    if rc != 0:
        raise RuntimeError(f'libgdeconv error {rc}: {lib.gd_last_error().decode(errors="replace")}')
