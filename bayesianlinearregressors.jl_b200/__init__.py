"""B200-native FiniteBLR inference path of BayesianLinearRegressors.jl.

Exports the reference's public names (src/BayesianLinearRegressors.jl:11-12: logpdf, rand, mean, std, cov,
BayesianLinearRegressor, marginals, posterior, BasisFunctionRegressor) plus the input wrappers AbstractGPs
re-exports (ColVecs, RowVecs).  Everything computes on the GPU through libblr_cuda; there is no CPU fallback.
"""
from ._lib import BLRError, DimensionMismatch, PosDefException, build, load  # noqa: F401
from .model import (AffineFeatures, TorchFeatureMap, BasisFunctionRegressor, BayesianLinearRegressor, BLRFunctionSample, ColVecs, DeviceRNG,  # noqa: F401
                    Diagonal, FiniteGP, PDMat, RandomFourierFeatures, RowVecs, Symmetric, cov, logpdf, marginals, mean,
                    logpdf_and_grad, mean_and_cov, mean_and_var, posterior, posterior_and_logpdf, posterior_and_logpdf_streamed, rand, rand_into, rand_with_draws, std, torch_features, torch_logpdf, var)
from .runtime import (Context, DeviceMatrix, DevicePosterior, DeviceVector, Stats, default_context,  # noqa: F401
                      set_default_context)
from .sharding import ShardPlan, packed_len  # noqa: F401
