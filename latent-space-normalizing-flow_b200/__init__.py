"""lsnf_b200 -- B200-native short-run Langevin posterior inference for latent-space normalizing-flow priors.

Drop-in for the hot path of jianwen-xie/Latent-Space-Normalizing-Flow: ``_netG`` / ``_netF`` keep the reference's
module interfaces and checkpoint keys (model.py), ``sample_langevin_post_z_with_flow`` replaces the closure of
train.py:307-335.  All device work is hand-written sm_100a CUDA behind the C ABI of ``include/lsnf.h``.
"""
from . import synth  # noqa: F401
from .ais import ais_log_likelihood, bdmc  # noqa: F401
from .autograd_fns import kernel_autograd  # noqa: F401
from .cli import parse_args  # noqa: F401
from .langevin import (AttrDict, langevin_plan, make_args, make_sampler, sample_langevin_post_z_with_flow,  # noqa: F401
                       reconstruction_error, sample_x)
from .model import _netF, _netG, weights_init_xavier  # noqa: F401
from .plan import Plan, clear_plans, get_plan, invalidate_plans  # noqa: F401
from .optim import FusedAdam  # noqa: F401
from .train import (flow_gradients, flow_update, generator_gradients, generator_update, generator_update_begin,  # noqa: F401
                    make_optimizers, training_iteration)

__all__ = ["_netG", "_netF", "weights_init_xavier", "sample_langevin_post_z_with_flow", "make_sampler", "make_args",
           "sample_x", "training_iteration", "make_optimizers", "flow_update", "flow_gradients", "generator_update", "generator_gradients", "FusedAdam", "Plan", "get_plan", "clear_plans", "invalidate_plans", "langevin_plan", "AttrDict", "synth",
           "parse_args", "reconstruction_error", "kernel_autograd", "ais_log_likelihood", "bdmc"]
