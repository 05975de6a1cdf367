"""cmf.jl_b200 -- B200-native drop-in for the convolutive-NMF fit path of degleris1/CMF.jl.

Host-side mirror of the reference's fit interface (``fit_cnmf``, ``MultUpdate``, ``HALSUpdate``,
``init_rand``, ``CNMF_results`` ...) over the C-ABI library ``libcmf_sm100`` (include/cmf_sm100.h),
whose kernels are hand-written CUDA for sm_100a (csrc/).  Import as ``cmf_jl_b200``.
"""
from ._lib import CMFError, F32, F64, HALS, MULT, SO_PATH  # noqa: F401
from .model import (  # noqa: F401
    AbstractCFUpdate, AlternatingOptimizer, CNMF_results, HALSUpdate, MultUpdate, PGDUpdate, compute_loss,
    converged, corr_w, fit, fit_cnmf, fit_cnmf_batch, init_rand, num_components, num_iter, num_lags, num_units,
    tensor_conv, tensor_transconv, compute_resids, shift_and_stack, SparseData, as_csc,
)
from .io import gen_synthetic, load_model, parameter_sweep, save_model  # noqa: F401
from .sharded import DeviceShard, LibraryFit, ShardedMultFit, ShardPlan  # noqa: F401

__all__ = [
    "fit_cnmf", "fit_cnmf_batch", "init_rand", "MultUpdate", "HALSUpdate", "PGDUpdate", "AbstractCFUpdate", "AlternatingOptimizer",
    "fit", "CNMF_results", "converged", "compute_loss", "tensor_conv", "tensor_transconv", "corr_w",
    "num_lags", "num_units", "num_components", "num_iter", "ShardPlan", "DeviceShard",
    "ShardedMultFit", "LibraryFit", "compute_resids", "shift_and_stack", "CMFError", "gen_synthetic", "save_model", "load_model", "parameter_sweep",
    "SparseData", "as_csc",
]
