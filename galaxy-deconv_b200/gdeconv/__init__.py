"""gdeconv: host-side runtime of the B200-native Galaxy-Deconv hot path (ctypes over libgdeconv.so)."""
from . import _lib  # noqa: F401  (loads / builds the shared library; fails loudly if it cannot)
from .engine import (AdmmEngine, adaptive_moments, conv_fft_batch, fft_solver, fpfs, metacal, moments_e, require_cuda_stamps, resunet_forward,  # noqa: F401
                     launch_count, default_precision)
from .synth import make_batch_device  # noqa: F401
