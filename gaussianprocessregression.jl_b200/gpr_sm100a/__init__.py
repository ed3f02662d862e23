"""gpr_sm100a: B200-native (sm_100a) exact-GP hot path behind the reference's model / covariance / cost /
predict API.  All arithmetic runs in libgpr_sm100a.so (hand-written CUDA, C ABI in include/gpr_sm100a.h);
there is no CPU fallback."""
from . import _ffi  # noqa: F401
from ._ffi import Context, GPRError, ModelHandle, MultiContext, MultiModelHandle, DistContext, PosDefException, get_context  # noqa: F401
from .api import *  # noqa: F401,F403
from .api import (Cmap, ComposedKernel, Diagonal, Euclidean, GPRModel, GPRPredictCache, GPRSplitPredictCache,  # noqa: F401
                  LogScale, MarginalLikelihood, Matern52, MllGradCache, MllLossCache, MultiGPUGradCache, MultiGPUPredictCache, NoLogScale, SplitKernel,
                  SquaredExp, UniformScaling, WhiteNoise, add_noise_, alloc_kernels, dim_hp, find_idx, get_sample,
                  grad, grad_, grad_cache, init_params, islog, kernel, kernel_, kernels, log_loss_grad_, loss,
                  loss_cache, loss_grad_, loss_grad_cache, predict, predict_, predict_cache, predict_mean,
                  predict_mean_, rm_noise, split, train, update_cache_, MSE, ChiSq, Mahalanobis, m_loss, kfoldcv, cv_step,
                  cv_step_, cv_batch, BFGSQuad, BFGSQuadCache, updater_cache, bfgs_hessian, bfgs_quad, bfgs_quad_,
                  hessian_fd, hessian_fd_, ReplicaGradient, update_sample_, GaussianProcess, NormalDistribution, sample, gauss_integ, erf_integ,
                  antideriv2, integrate)
