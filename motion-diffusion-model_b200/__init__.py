"""b200mdm -- B200-native sampling engine behind the motion-diffusion-model API.

    from b200mdm import create_model_and_diffusion, ClassifierFreeSampleModel, load_saved_model
    model, diffusion = create_model_and_diffusion(args, data)          # utils/model_util.py:18 of the reference
    model = ClassifierFreeSampleModel(model).to("cuda").eval()         # utils/sampler_util.py:10
    sample = diffusion.p_sample_loop(model, (B, 263, 1, 196), clip_denoised=False, model_kwargs={"y": y})

Python here is host glue only; the per-step path is hand-written sm_100a CUDA in lib/libb200mdm.so
(C ABI: include/b200mdm.h).  Importing this package does not need a GPU; running a model does.
"""
from .utils.model_util import (create_model_and_diffusion, create_gaussian_diffusion, get_model_args,  # noqa: F401
                               load_saved_model, load_model_wo_clip)
from .utils.sampler_util import ClassifierFreeSampleModel, AutoRegressiveSampler  # noqa: F401
from .diffusion.respace import SpacedDiffusion, space_timesteps  # noqa: F401
from .diffusion.gaussian_diffusion import GaussianDiffusion, get_named_beta_schedule  # noqa: F401
from .model.mdm import MDM  # noqa: F401
from .synthetic import (synthetic_state_dict, synthetic_inputs, synthetic_dip_inputs, synthetic_norm_stats,  # noqa: F401
                        synthetic_targets)

__version__ = "0.1.0"
from .data_loaders.humanml.scripts.motion_process import recover_from_ric, sample_to_xyz  # noqa: F401,E402
