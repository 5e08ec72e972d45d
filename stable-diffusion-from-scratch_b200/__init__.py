"""sdb200 — B200-native (sm_100a) implementation of the latent-diffusion sampling hot path of
ProgramerSalar/stable-diffusion-from-scratch, behind the reference's own Python module API.

    from sdb200.openai_model import UNetModel          # reference: openai_model/model.py:259
    from sdb200.ddim import DDIMSampler                # reference: ldm/diffusion/ddim.py:12
    from sdb200.plms import PLMSSampler                # reference: CompVis ldm/models/diffusion/plms.py
    from sdb200.dpm_solver import DPMSolverSampler     # reference: CompVis ldm/models/diffusion/dpm_solver/
    from sdb200.autoencoder import AutoencoderKL       # reference: ldm/models/autoencoder.py:292
    from sdb200.ddpm_unet import UNet                  # reference: DDPM/models/unet.py:11

All arithmetic runs in hand-written CUDA kernels from libsdb200.so (include/sdb200.h); there is no
CPU or PyTorch fallback.  The directory is named after the reference (`stable-diffusion-from-scratch_b200`),
which is not a valid Python identifier, so the importable name is the `sdb200` alias package.
"""
__version__ = "0.1.0"
