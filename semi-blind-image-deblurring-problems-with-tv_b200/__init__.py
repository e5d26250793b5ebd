"""sbd_b200 - B200-native engine for the SAPG / MYULA semi-blind TV-deblurring
hot path (host-side Python mirror of the reference's MATLAB interface on top of
the C ABI of libsbd.so; see include/sbd.h and INTEGRATION.md).

The numerical work is done by hand-written CUDA kernels (sm_100a, fp64) in
`csrc/`.  There is no CPU fallback: importing works everywhere (so that the
symbol table can be checked without a GPU), but every compute call needs the
built library and a B200.
"""
from ._lib import lib, LIB_PATH, SbdError, load_library  # noqa: F401
from .host import (  # noqa: F401
    Engine, engine_for, posterior_moments, posterior_diagnostics,
    Gaussian_psf, psf_gaussian, psf_moffat, psf_laplace,
    moffat_psf, laplace_psf, gaussian_fft, diff_fftgaus_w1, diff_fftgaus_w2,
    diff_moffat_alpha, diff_moffat_beta, diff_laplace_b,
    TVnorm, diffh, diffv, chambolle_prox_TV_stop,
    gaussian_closures, moffat_closures, laplace_closures,
    SAPG_algorithm_Guassian, SAPG_algorithm_moffat, SAPG_algorithm_laplace,
    GAUSSIAN, MOFFAT, LAPLACE,
)
from .shard import ChainShard  # noqa: F401

__version__ = "0.1.0"
