"""dpmmsubclusters.jl_b200 -- B200-native data-parallel sweep for the DPMM sub-cluster sampler.

The directory name contains a dot, so it is not importable with a plain `import`; use
`dpmm_pkg.load()` at the repository root (registers the package as `dpmmsubclusters_jl_b200`).
"""
from . import _lib  # noqa: F401
from .sweep import GpuSweep, NIW, MULTINOMIAL, DIAG  # noqa: F401
from .priors import (niw_hyperparams, multinomial_hyper, niw_sufficient_statistics,  # noqa: F401
                     multinomial_sufficient_statistics, mv_gaussian, multinomial_dist, diag_niw_hyperparams,
                     diag_niw_sufficient_statistics, diag_gaussian, calc_posterior,
                     sample_distribution, log_marginal_likelihood, aggregate_suff_stats)
from .data_generators import generate_gaussian_data, generate_mnmm_data  # noqa: F401
from .host import (fit, dp_parallel, predict, calculate_posterior, get_labels_histogram,  # noqa: F401
                   run_model_from_checkpoint)
from .checkpoint import load_data, save_model, load_checkpoint  # noqa: F401
