"""cocons_b200 - B200-native dense-likelihood path of blasif/cocons.

The product is libcocons_b200.so (hand-written sm_100a CUDA behind the C ABI of
include/cocons_b200.h).  This package is its host-side mirror of the
reference's R interface; see api.py.
"""
from .api import (  # noqa: F401
    CoconsError,
    DenseLikelihood,
    DenseLikelihoodBatch,
    DenseLikelihoodPool,
    GetNeg2loglikelihood,
    GetNeg2loglikelihoodProfile,
    GetNeg2loglikelihoodREML,
    GetNeg2loglikelihoodTaper,
    GetNeg2loglikelihoodTaperProfile,
    NotPositiveDefinite,
    TaperedLikelihood,
    coco,
    cocoOptim,
    cocoPredict,
    cocoSim,
    cov_rns,
    cov_rns_classic,
    cov_rns_pred,
    cov_rns_taper,
    cov_rns_taper_pred,
    cov_wend1,
    cov_wend2,
    fd_value_and_grad,
    getCovMatrix,
    getDensityFromDelta,
    getDesignMatrix,
    getEstims,
    getHessian,
    getModelLists,
    getScale,
    is_formula,
    nearest_dist,
    reml_contrasts,
    spam,
    sumsmoothlone,
)

__version__ = "0.1.0"
