"""makeupdiffuse_b200 — B200-native (sm_100a) implementation of MakeupDiffuse's denoising hot path.

Public surface (mirrors the reference's, SURVEY.md §8(b)):
    B200DDIMSampler      <->  diffmk.cddim.MKDDIMSampler / ldm DDIMSampler
    B200PLMSSampler      <->  ldm PLMSSampler (upstream ldm/models/diffusion/plms.py)
    B200DPMSolverSampler <->  ldm DPMSolverSampler (upstream ldm/models/diffusion/dpm_solver/sampler.py)
    B200ControlLDM       <->  the ControlLDM object the sampler calls apply_model(x_t, t, cond) on
    B200ControlNet       <->  cldm.cldm.ControlNet            (yaml control_stage_config target)
    B200ControlledUnet   <->  cldm.cldm.ControlledUnetModel   (yaml unet_config target)
    B200FirstStageDecoder <-> first_stage_model.decode of ldm AutoencoderKL (yaml first_stage_config; SURVEY §8(f) rank 1)
    B200FrozenCLIPEmbedder <-> cond_stage_model (ldm FrozenCLIPEmbedder = HF CLIPTextModel; yaml:109-110; §8(f) rank 3)
Everything computes through libmkd_b200.so (include/mkd_b200.h); there is no CPU or PyTorch-compute fallback.
"""
from .ldm import B200ControlLDM  # noqa: F401
from .nets import B200ControlNet, B200ControlledUnet  # noqa: F401
from .sampler import B200DDIMSampler, B200DPMSolverSampler, B200PLMSSampler  # noqa: F401
from .vae import B200FirstStageDecoder, B200FirstStageEncoder  # noqa: F401
from .clip import B200FrozenCLIPEmbedder  # noqa: F401

__all__ = ["B200DDIMSampler", "B200PLMSSampler", "B200DPMSolverSampler", "B200ControlLDM", "B200ControlNet", "B200ControlledUnet", "B200FirstStageDecoder", "B200FirstStageEncoder",
           "B200FrozenCLIPEmbedder"]
