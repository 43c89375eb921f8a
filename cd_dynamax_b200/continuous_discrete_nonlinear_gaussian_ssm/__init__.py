# mirrors src/continuous_discrete_nonlinear_gaussian_ssm/__init__.py:1-7
from .cdnlgssm_utils import (GSSMForecast, LearnableLinear, LearnableLorenz63, LearnableLorenz96, LearnableMatrix,
                             LearnableQuadratic, LearnableUserDrift, LearnableUserEmission, LearnableVector, ParamsCDNLGSSM, ParamsCDNLGSSMDynamics,
                             ParamsCDNLGSSMEmissions)
from .inference_ekf import (EKFHyperParams, ekf_marginal_log_prob_and_grad,
                            ekf_dense_marginal_log_prob_and_grad, extended_kalman_filter,
                            extended_kalman_smoother, iterated_extended_kalman_filter,
                            iterated_extended_kalman_smoother)
from .inference_enkf import EnKFHyperParams, ensemble_kalman_filter
from .inference_ukf import (UKFHyperParams, ukf_marginal_log_prob_and_grad, ukf_sigma_points_marginal_log_prob_and_grad,
                            unscented_kalman_filter)
from .models import ContDiscreteNonlinearGaussianSSM, cdnlgssm_filter, cdnlgssm_smoother
from .forecast import (MultivariateNormalFullCovariance, cdnlgssm_emissions, cdnlgssm_forecast,  # noqa: E402
                       cdnlgssm_path_sample)
