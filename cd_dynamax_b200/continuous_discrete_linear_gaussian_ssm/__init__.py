# mirrors src/continuous_discrete_linear_gaussian_ssm/__init__.py:1-8 (sampling entry points are out of scope)
from .inference import (KFHyperParams, ParamsCDLGSSM, ParamsCDLGSSMDynamics, cdlgssm_filter,
                        cdlgssm_marginal_log_prob_and_grad, cdlgssm_smoother, make_cdlgssm_params)
from .models import ContDiscreteLinearGaussianSSM
