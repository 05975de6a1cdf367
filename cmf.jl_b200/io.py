"""The steps either side of the fit path (SURVEY.md section 8f row 3): synthetic data and result I/O.

    gen_synthetic(N, T, ...)           README.md:14 `CMF.gen_synthetic(N=500, T=2000)` -> data; the data model is
                                       datasets/synthetic.jl:29-61 (Dirichlet unit weights x Gaussian lag bumps,
                                       Exp(1)*Bernoulli(p_h) activations, Gaussian noise, clipped at 0), generated in HBM by
                                       the library's counter-based generator (cmf_synth_data) -- Julia's RNG stream is not
                                       reproducible here, so the values differ from a Julia run with the same seed.
    save_model / load_model            src/model.jl:149-181, fixed to the fields the struct really has
                                       (data, W, H, time_hist, loss_hist; model.jl:11-17).  HDF5 is not available in this
                                       image, so the container is NumPy's .npz with the reference's dataset names.
    parameter_sweep                    src/model.jl:132-146.
"""
from __future__ import annotations

import itertools
import math

import numpy as np

from ._lib import MULT, Handle, parse_dtype


def gen_synthetic(N=100, T=500, K=3, L=20, p_h=0.5, noise_scale=1.0, seed=1234, dtype="f64", device=0):
    """N x T non-negative synthetic data with K ground-truth motifs of L lags (datasets/synthetic.jl:29-61 defaults:
    alpha = 0.1, sigma = 0.2 are fixed inside the device generator)."""
    with Handle(N, T, K, L, parse_dtype(dtype), MULT, device) as h:
        h.synth_data(seed, K, L, p_h, noise_scale)
        return h.get_data()


def save_model(results, path):
    """src/model.jl:149-163 with the real struct fields."""
    np.savez_compressed(path, W=results.W, H=results.H, data=results.data,
                        loss_hist=np.asarray(results.loss_hist, dtype=np.float64),
                        time_hist=np.asarray(results.time_hist, dtype=np.float64),
                        layout=getattr(results, "layout", "LNK"))


def load_model(path):
    """src/model.jl:166-181."""
    from .model import CNMF_results

    with np.load(path if str(path).endswith(".npz") else str(path) + ".npz") as f:
        return CNMF_results(f["data"], f["W"], f["H"], list(f["time_hist"]), list(f["loss_hist"]), str(f["layout"]))


def parameter_sweep(data, L_vals=(7,), K_vals=(3,), alg_vals=("mult",), max_itr=100, max_time=math.inf, **kwargs):
    """src/model.jl:132-146: one fit per (L, K, alg); returns {(L, K, alg): CNMF_results}."""
    from .model import fit_cnmf

    return {(L, K, alg): fit_cnmf(data, L=L, K=K, alg=alg, max_itr=max_itr, max_time=max_time, **kwargs)
            for L, K, alg in itertools.product(L_vals, K_vals, alg_vals)}
