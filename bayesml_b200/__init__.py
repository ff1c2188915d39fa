"""bayesml_b200 — B200-native variational-Bayes Gaussian mixture, drop-in for `bayesml.gaussianmixture.LearnModel`
(and, sharing its kernels, `bayesml.hiddenmarkovnormal.LearnModel`; both modules also have the reference's `GenModel`, whose
`gen_sample` can draw on the device).

    from bayesml_b200 import gaussianmixture
    model = gaussianmixture.LearnModel(c_num_classes=3, c_degree=2)
    model.update_posterior(x)

The compute path is hand-written CUDA for sm_100a behind a C ABI (include/bgmm.h, libbgmm.so); there is no CPU
fallback.  Importing the package does not need a GPU; fitting does.
"""
from . import gaussianmixture, hiddenmarkovnormal, multivariate_normal  # noqa: F401
from ._exceptions import (CriteriaError, DataFormatError, ParameterFormatError,  # noqa: F401
                          ParameterFormatWarning, ResultWarning)

__version__ = "0.1.0"
