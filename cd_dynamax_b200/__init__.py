"""cd_dynamax_b200 -- B200-native drop-in for the batched continuous-discrete Gaussian filtering / smoothing hot path of
hd-UQ/cd_dynamax.  The reference's entry points keep their names and signatures; the arithmetic runs in hand-written
sm_100a CUDA kernels behind a C ABI (include/cdk.h, cd_dynamax_b200/lib/libcdk.so).  There is no CPU fallback."""
from . import solvers
from .continuous_discrete_linear_gaussian_ssm import (ContDiscreteLinearGaussianSSM, KFHyperParams, ParamsCDLGSSM,
                                                      ParamsCDLGSSMDynamics, cdlgssm_filter,
                                                      cdlgssm_marginal_log_prob_and_grad, cdlgssm_smoother,
                                                      make_cdlgssm_params)
from .continuous_discrete_nonlinear_gaussian_ssm import (ContDiscreteNonlinearGaussianSSM, EKFHyperParams,
                                                         EnKFHyperParams, LearnableLinear, LearnableLorenz63,
                                                         LearnableLorenz96, LearnableMatrix, LearnableQuadratic, LearnableUserDrift,
                                                         LearnableUserEmission,
                                                         LearnableVector, ParamsCDNLGSSM, ParamsCDNLGSSMDynamics,
                                                         ParamsCDNLGSSMEmissions, UKFHyperParams, cdnlgssm_filter,
                                                         cdnlgssm_smoother, ekf_marginal_log_prob_and_grad,
                                                         ekf_dense_marginal_log_prob_and_grad, GSSMForecast,
                                                         MultivariateNormalFullCovariance, cdnlgssm_emissions,
                                                         cdnlgssm_forecast, cdnlgssm_path_sample,
                                                         ukf_marginal_log_prob_and_grad,
                                                         ukf_sigma_points_marginal_log_prob_and_grad)
from .types import (ParameterProperties, ParamsLGSSMEmissions, ParamsLGSSMInitial, PosteriorGSSMFiltered,
                    PosteriorGSSMSmoothed)

__version__ = "0.1.0"
