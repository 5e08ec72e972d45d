"""Minimal, Lightning-free sampling glue around the hot path (SURVEY.md §8 row f1).

`LatentDiffusion` exposes exactly what `DDIMSampler` and the reference's `sample_log` /
`decode_first_stage` call sites need (ldm/diffusion/ddpm.py:1326-1448, 1083-1156, 1814-1826):
schedule buffers, `apply_model(x, t, cond)`, `decode_first_stage(z)`.  It owns a `UNetModel`
(as `model.diffusion_model`, like DiffusionWrapper, ddpm.py:1992-2034, with all five conditioning keys) and an
`AutoencoderKL` (or any first stage given as `first_stage_model`: a `VQModelInterface` for the VQ models, built with
`scale_factor=1.0` and `channels=3`).
It also carries the reference's ancestral sampler (`sample` / `p_sample_loop` / `progressive_denoising`,
ddpm.py:1528-1793), whose per-step update runs as one fused kernel (sdb_ddpm_step).
"""
import numpy as np
import torch
from torch import nn

from . import engine, ops
from .autoencoder import AutoencoderKL, DiagonalGaussianDistribution, VQModelInterface
from .ddim import DDIMSampler, _f32_contiguous
from .dpm_solver import DPMSolverSampler
from .openai_model import UNetModel
from .plms import PLMSSampler

SD_UNET_CONFIG = dict(  # Diffusion/config.yaml:31-44
    image_size=32, in_channels=4, out_channels=4, model_channels=320, attention_resolutions=[4, 2, 1],
    num_res_blocks=2, channel_mult=(1, 2, 4, 4), num_heads=8, use_spatial_transformer=True,
    transformer_depth=1, context_dim=768, use_checkpoint=False, legacy=False)
SD_VAE_DDCONFIG = dict(  # Diffusion/config.yaml:51-64
    double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128, ch_mult=(1, 2, 4, 4),
    num_res_blocks=2, attn_resolutions=[], dropout=0.0)


def make_beta_schedule(schedule, n_timestep, linear_start=1e-4, linear_end=2e-2):
    """ldm/modules/diffusionmodules/util.py:21-44."""
    if schedule == "linear":
        betas = torch.linspace(linear_start ** 0.5, linear_end ** 0.5, n_timestep, dtype=torch.float64) ** 2
    elif schedule == "sqrt_linear":
        betas = torch.linspace(linear_start, linear_end, n_timestep, dtype=torch.float64)
    elif schedule == "sqrt":
        betas = torch.linspace(linear_start, linear_end, n_timestep, dtype=torch.float64) ** 0.5
    else:
        raise ValueError(f"schedule '{schedule}' unknown.")
    return betas.numpy()


class DiffusionWrapper(nn.Module):
    """ldm/diffusion/ddpm.py:1992-2034: routes the conditioning to the UNet by `conditioning_key`.
      None        diffusion_model(x, t)
      "concat"    diffusion_model(cat([x] + c_concat, 1), t)
      "crossattn" diffusion_model(x, t, context=cat(c_crossattn, 1))
      "hybrid"    diffusion_model(cat([x] + c_concat, 1), t, context=cat(c_crossattn, 1))
      "adm"       diffusion_model(x, t, y=c_crossattn[0])
    The channel concat goes to the model's `forward_concat` when it has one (UNetModel: the concat is done by the layout
    kernel feeding conv_in); any other eps-model gets the torch.cat and its plain forward."""

    KEYS = (None, "concat", "crossattn", "hybrid", "adm")

    def __init__(self, diffusion_model, conditioning_key="crossattn"):
        super().__init__()
        self.diffusion_model = diffusion_model
        self.conditioning_key = conditioning_key
        assert conditioning_key in self.KEYS, "unknown conditioning_key %r (one of %s)" % (conditioning_key, self.KEYS)

    @staticmethod
    def _context(c_crossattn):
        # one tensor is passed as is (no copy), so a UNet that caches its K/V projections per context tensor keeps hitting
        return c_crossattn[0] if len(c_crossattn) == 1 else torch.cat(c_crossattn, 1)

    def _concat(self, x, t, c_concat, **kw):
        c_concat = [c_concat] if torch.is_tensor(c_concat) else list(c_concat)
        fc = getattr(self.diffusion_model, "forward_concat", None)
        if fc is not None:
            return fc(x, c_concat, t, **kw)
        return self.diffusion_model(torch.cat([x] + c_concat, dim=1), t, **kw)

    def forward(self, x, t, c_concat=None, c_crossattn=None):
        key = self.conditioning_key
        if key is None:
            return self.diffusion_model(x, t)
        if key == "concat":
            return self._concat(x, t, c_concat)
        if key == "crossattn":
            return self.diffusion_model(x, t, context=self._context(c_crossattn))
        if key == "hybrid":
            return self._concat(x, t, c_concat, context=self._context(c_crossattn))
        return self.diffusion_model(x, t, y=c_crossattn[0])          # "adm"


class LatentDiffusion(nn.Module):
    def __init__(self, unet_config=None, first_stage_config=None, timesteps=1000, linear_start=0.00085, linear_end=0.0120,
                 beta_schedule="linear", scale_factor=0.18215, conditioning_key="crossattn", compute_mode=None,
                 unet=None, first_stage_model=None, cond_stage_model=None, v_posterior=0., clip_denoised=True,
                 log_every_t=100, channels=4, image_size=64, cond_stage_key="image", cond_stage_config=None,
                 cond_stage_forward=None, cond_stage_trainable=False):
        super().__init__()
        # optional conditioner (Diffusion/config.yaml:69-70: FrozenCLIPEmbedder; sdb200.encoders for the other stages);
        # None = the caller supplies the conditioning tensors.  cond_stage_config picks one by the reference's special values.
        self.cond_stage_model = cond_stage_model
        if cond_stage_config == "__is_unconditional__":
            conditioning_key = None                      # ldm/diffusion/ddpm.py LatentDiffusion.__init__
        # sampling only: accepted for the reference's configs, no gradient path is built
        self.cond_stage_trainable = cond_stage_trainable
        self.cond_stage_forward = cond_stage_forward
        unet = unet if unet is not None else UNetModel(**(unet_config or SD_UNET_CONFIG), compute_mode=compute_mode)
        self.model = DiffusionWrapper(unet, conditioning_key)
        if first_stage_model is None and first_stage_config is not False:
            first_stage_model = AutoencoderKL(ddconfig=(first_stage_config or SD_VAE_DDCONFIG), embed_dim=4, compute_mode=compute_mode)
        self.first_stage_model = first_stage_model
        if cond_stage_config is not None:
            self.instantiate_cond_stage(cond_stage_config)
        self.scale_factor = scale_factor
        self.parameterization = "eps"
        self.shorten_cond_schedule = False
        self.v_posterior = v_posterior
        self.clip_denoised = clip_denoised
        self.log_every_t = log_every_t
        self.channels = channels
        self.image_size = image_size
        # read only by the split_input_params branch of apply_model: which conditionings are cut into crops with the latent
        self.cond_stage_key = cond_stage_key
        # split_input_params branch: at most this many crops per model call (None = all L crops of a call in one batch)
        self.patch_batch = None
        self.num_timesteps = int(timesteps)
        betas = make_beta_schedule(beta_schedule, timesteps, linear_start=linear_start, linear_end=linear_end)
        alphas_cumprod = np.cumprod(1. - betas, axis=0)
        alphas_cumprod_prev = np.append(1., alphas_cumprod[:-1])
        to_t = lambda a: torch.tensor(a, dtype=torch.float32)
        self.register_buffer("betas", to_t(betas))
        self.register_buffer("alphas_cumprod", to_t(alphas_cumprod))
        self.register_buffer("alphas_cumprod_prev", to_t(alphas_cumprod_prev))
        self.register_buffer("sqrt_alphas_cumprod", to_t(np.sqrt(alphas_cumprod)))           # ldm/diffusion/ddpm.py:212-213
        self.register_buffer("sqrt_one_minus_alphas_cumprod", to_t(np.sqrt(1. - alphas_cumprod)))
        # the rest of register_schedule (ddpm.py DDPM.register_schedule), float64 numpy cast to fp32, the reference's expressions
        alphas = 1. - betas
        self.register_buffer("log_one_minus_alphas_cumprod", to_t(np.log(1. - alphas_cumprod)))
        self.register_buffer("sqrt_recip_alphas_cumprod", to_t(np.sqrt(1. / alphas_cumprod)))
        self.register_buffer("sqrt_recipm1_alphas_cumprod", to_t(np.sqrt(1. / alphas_cumprod - 1)))
        posterior_variance = (1 - self.v_posterior) * betas * (1. - alphas_cumprod_prev) / (1. - alphas_cumprod) + self.v_posterior * betas
        self.register_buffer("posterior_variance", to_t(posterior_variance))
        self.register_buffer("posterior_log_variance_clipped", to_t(np.log(np.maximum(posterior_variance, 1e-20))))
        self.register_buffer("posterior_mean_coef1", to_t(betas * np.sqrt(alphas_cumprod_prev) / (1. - alphas_cumprod)))
        self.register_buffer("posterior_mean_coef2", to_t((1. - alphas_cumprod_prev) * np.sqrt(alphas) / (1. - alphas_cumprod)))
        self._split_cond_cache = engine.TensorMemo(8)     # _repeat_cond
        self._ddpm_tables = engine.TensorMemo(1)          # _ddpm_cache

    @property
    def device(self):
        return self.betas.device

    def apply_model(self, x_noisy, t, cond, return_ids=False):
        """ldm/diffusion/ddpm.py:1326-1448.  A non-dict `cond` goes under c_concat ("concat") or c_crossattn (other keys).

        With a `split_input_params` attribute (the reference's patch-distributed branch, ddpm.py:1344-1437) x_noisy is cut
        into its crops of split_input_params["ks"] at ["stride"], the model is run on every crop, and the outputs are
        stitched with the border-weighted fold divided by the folded weights.  The reference loops over the L crops; here
        they run as one batch of L*B samples (at most `patch_batch` crops per call), which gives the same bits because
        per-sample results do not depend on the batch.  Conditioning: with cond_stage_key in "image", "LR_image",
        "segmentation", "bbox_img" and a conditioning_key, the single conditioning tensor is cut into the same crops;
        otherwise every crop gets the whole conditioning."""
        if isinstance(cond, dict):
            pass
        else:
            if not isinstance(cond, list):
                cond = [cond]
            key = "c_concat" if self.model.conditioning_key == "concat" else "c_crossattn"
            cond = {key: cond}
        if hasattr(self, "split_input_params"):
            assert len(cond) == 1  # the reference's branch takes one conditioning entry
            assert not return_ids
            return self._apply_model_split(x_noisy, t, cond)
        return self.model(x_noisy, t, **cond)

    # ---- split_input_params: patch-distributed fold / unfold (ldm/diffusion/ddpm.py:1030-1139, 1344-1437) ----------------
    SPLIT_IMAGE_KEYS = ("image", "LR_image", "segmentation", "bbox_img")

    def meshgrid(self, h, w):
        y = torch.arange(0, h).view(h, 1, 1).repeat(1, w, 1)
        x = torch.arange(0, w).view(1, w, 1).repeat(h, 1, 1)
        arr = torch.cat([y, x], dim=-1)
        return arr

    def delta_border(self, h, w):
        """Normalised distance of each pixel of an h x w crop to the crop's border: 0 at the border, 0.5 at the centre."""
        lower_right_corner = torch.tensor([h - 1, w - 1]).view(1, 1, 2)
        arr = self.meshgrid(h, w) / lower_right_corner
        dist_left_up = torch.min(arr, dim=-1, keepdims=True)[0]
        dist_right_down = torch.min(1 - arr, dim=-1, keepdims=True)[0]
        edge_dist = torch.min(torch.cat([dist_left_up, dist_right_down], dim=-1), dim=-1)[0]
        return edge_dist

    def get_weighting(self, h, w, Ly, Lx, device):
        """[1, h*w, Ly*Lx] per-pixel crop weights, evaluated on the host; times the clipped per-crop border weight of the
        Ly x Lx grid with split_input_params["tie_braker"]."""
        weighting = self.delta_border(h, w)
        weighting = torch.clip(weighting, self.split_input_params["clip_min_weight"], self.split_input_params["clip_max_weight"], )
        weighting = weighting.view(1, h * w, 1).repeat(1, 1, Ly * Lx)
        if self.split_input_params["tie_braker"]:
            L_weighting = self.delta_border(Ly, Lx)
            L_weighting = torch.clip(L_weighting, self.split_input_params["clip_min_tie_weight"],
                                     self.split_input_params["clip_max_tie_weight"])
            L_weighting = L_weighting.view(1, 1, Ly * Lx)
            weighting = weighting * L_weighting
        return weighting.to(device)

    def _patch_weights(self, h, w, Ly, Lx, device):
        """The device tables of sdb_patch_fold for crops of h x w on a Ly x Lx grid: (wpix [h*w], wcrop [Ly*Lx] or None).
        fl(wpix[p] * wcrop[l]) is get_weighting's element (p, l).  Cached per geometry, clip values and device, so a
        sampling step makes no host-to-device copy."""
        sp = self.split_input_params
        tie = bool(sp["tie_braker"])
        clips = (sp["clip_min_weight"], sp["clip_max_weight"]) + ((sp["clip_min_tie_weight"], sp["clip_max_tie_weight"]) if tie else ())
        key = (h, w, Ly, Lx, clips, tie, torch.device(device))
        cache = self.__dict__.setdefault("_patch_weight_cache", {})
        if key not in cache:
            wpix = torch.clip(self.delta_border(h, w), sp["clip_min_weight"], sp["clip_max_weight"]).reshape(-1)
            wcrop = None
            if tie:
                wcrop = torch.clip(self.delta_border(Ly, Lx), sp["clip_min_tie_weight"], sp["clip_max_tie_weight"]).reshape(-1)
                wcrop = wcrop.float().contiguous().to(device)
            cache[key] = (wpix.float().contiguous().to(device), wcrop)
        return cache[key]

    def _split_geometry(self, h, w, ks, stride, uf=1, df=1):
        """get_fold_unfold's fold side for an h x w input cut into crops of ks at `stride`: (Ly, Lx), the fold's crop size,
        its stride and its output size.  uf > 1 (decode) scales the crops up, df > 1 (encode) down."""
        Ly, Lx = ops.patch_grid(h, w, ks, stride)
        if uf == 1 and df == 1:
            return (Ly, Lx), tuple(ks), tuple(stride), (h, w)
        if ks[0] != ks[1]:
            # the reference folds with a square (ks[0] * f, ks[0] * f) kernel but weights (ks[0] * f, ks[1] * f) crops
            raise NotImplementedError("split_input_params: a non-square ks %s with vqf > 1 is not supported" % (tuple(ks),))
        if uf > 1:
            return (Ly, Lx), (ks[0] * uf, ks[0] * uf), (stride[0] * uf, stride[1] * uf), (h * uf, w * uf)
        return (Ly, Lx), (ks[0] // df, ks[0] // df), (stride[0] // df, stride[1] // df), (h // df, w // df)

    def _fold_crops(self, o, B, grid, fks, fstride, out_hw, device):
        if tuple(o.shape[2:]) != tuple(fks) or o.shape[0] != grid[0] * grid[1] * B:
            raise ValueError("split_input_params: the crops came back as %s, the fold expects %d x [%d, C, %d, %d]"
                             % (tuple(o.shape), grid[0] * grid[1], B, fks[0], fks[1]))
        wpix, wcrop = self._patch_weights(fks[0], fks[1], grid[0], grid[1], device)
        return ops.patch_fold(o.float().contiguous(), B, grid, fstride, out_hw, wpix, wcrop)

    def _repeat_cond(self, v, n):
        """v repeated n times along the batch (the same conditioning for n crops), cached per (live caller's tensor, n): a
        UNet that caches its context K/V projections per context tensor keeps hitting across steps."""
        if not torch.is_tensor(v) or n == 1:
            return v
        return self._split_cond_cache.get((v,), (id(v), n), lambda: v.repeat(n, *((1,) * (v.dim() - 1))))

    def _apply_model_split(self, x_noisy, t, cond):
        sp = self.split_input_params
        ks, stride = tuple(sp["ks"]), tuple(sp["stride"])
        B, _, h, w = x_noisy.shape
        grid, fks, fstride, out_hw = self._split_geometry(h, w, ks, stride)
        L = grid[0] * grid[1]
        c_key, c_val = next(iter(cond.items()))
        if self.cond_stage_key in self.SPLIT_IMAGE_KEYS and self.model.conditioning_key:
            assert len(c_val) == 1  # one conditioning tensor, cut like the latent
            c = c_val[0]
            if not torch.is_tensor(c) or c.dim() != 4 or tuple(c.shape[-2:]) != (h, w):
                raise ValueError("split_input_params with cond_stage_key %r: the conditioning must be a 4-d tensor of the "
                                 "latent's size %s (got %s)" % (self.cond_stage_key, (h, w),
                                                                tuple(c.shape) if torch.is_tensor(c) else type(c).__name__))
            cc = ops.patch_unfold(c, ks, stride)
            cond_for = lambda l0, l1: {c_key: [cc[l0 * B:l1 * B]]}
        elif self.cond_stage_key == "coordinates_bbox":
            raise NotImplementedError("split_input_params with cond_stage_key 'coordinates_bbox' is not supported")
        else:
            def cond_for(l0, l1):
                rep = lambda v: [self._repeat_cond(e, l1 - l0) for e in v] if isinstance(v, list) else self._repeat_cond(v, l1 - l0)
                return {k: rep(v) for k, v in cond.items()}
        z = ops.patch_unfold(x_noisy, ks, stride)
        n = L if not self.patch_batch else max(1, min(int(self.patch_batch), L))
        outs = [self.model(z[l0 * B:min(L, l0 + n) * B], t.repeat(min(L, l0 + n) - l0), **cond_for(l0, min(L, l0 + n)))
                for l0 in range(0, L, n)]
        assert not isinstance(outs[0], tuple)
        o = outs[0] if len(outs) == 1 else torch.cat(outs)
        out = self._fold_crops(o, B, grid, fks, fstride, out_hw, x_noisy.device)
        return out if x_noisy.dtype == torch.float32 else out.to(x_noisy.dtype)

    def _split_first_stage(self, x, fn, uf=1, df=1):
        """decode_first_stage / encode_first_stage with split_input_params["patch_distributed_vq"]: ks and stride are
        reduced to the input size, the crops go through `fn` as one batch, and the results are folded."""
        sp = self.split_input_params
        ks, stride = tuple(sp["ks"]), tuple(sp["stride"])
        B, _, h, w = x.shape
        if ks[0] > h or ks[1] > w:
            ks = (min(ks[0], h), min(ks[1], w))
            print("reducing Kernel")
        if stride[0] > h or stride[1] > w:
            stride = (min(stride[0], h), min(stride[1], w))
            print("reducing stride")
        grid, fks, fstride, out_hw = self._split_geometry(h, w, ks, stride, uf=uf, df=df)
        o = fn(ops.patch_unfold(x, ks, stride))
        if not torch.is_tensor(o):
            raise NotImplementedError("split_input_params: the first stage returned %s, not a tensor" % type(o).__name__)
        return self._fold_crops(o, B, grid, fks, fstride, out_hw, x.device)

    def instantiate_cond_stage(self, config):
        """ldm/diffusion/ddpm.py `instantiate_cond_stage` for its two special values: "__is_first_stage__" conditions on the
        first stage's encoding (the inpainting LDM), "__is_unconditional__" has no conditioner.  A `target:` config is not
        instantiated here: build the stage (sdb200.encoders) and pass it as `cond_stage_model`."""
        if config not in ("__is_first_stage__", "__is_unconditional__"):
            raise NotImplementedError("cond_stage_config %r: only '__is_first_stage__' and '__is_unconditional__' are "
                                      "resolved here; pass the conditioning stage as cond_stage_model" % (config,))
        assert not self.cond_stage_trainable, "a trainable cond stage cannot be %s" % config
        if self.cond_stage_model is not None:
            raise ValueError("cond_stage_config %r and a cond_stage_model were both given" % (config,))
        self.cond_stage_model = self.first_stage_model if config == "__is_first_stage__" else None

    @torch.no_grad()
    def get_learned_conditioning(self, c):
        """ldm/diffusion/ddpm.py `get_learned_conditioning`: getattr(cond_stage_model, cond_stage_forward)(c) when
        cond_stage_forward is set, else cond_stage_model.encode(c) (the distribution's mode when encode returns a
        DiagonalGaussianDistribution) or, without an encode method, cond_stage_model(c)."""
        assert self.cond_stage_model is not None, "no cond_stage_model was given"
        if self.cond_stage_forward is not None:
            assert hasattr(self.cond_stage_model, self.cond_stage_forward)
            return getattr(self.cond_stage_model, self.cond_stage_forward)(c)
        if hasattr(self.cond_stage_model, "encode") and callable(self.cond_stage_model.encode):
            c = self.cond_stage_model.encode(c)
            if isinstance(c, DiagonalGaussianDistribution):
                c = c.mode()
            return c
        return self.cond_stage_model(c)

    def q_sample_coefficients(self, t):
        """extract_into_tensor(sqrt_alphas_cumprod, t, .) and (sqrt_one_minus_alphas_cumprod, t, .) as two [B] fp32 vectors
        (ldm/diffusion/ddpm.py:411-412; ldm/modules/diffusionmodules/util.py:96-99)."""
        t = t.to(self.sqrt_alphas_cumprod.device)
        return self.sqrt_alphas_cumprod.gather(-1, t).contiguous(), self.sqrt_one_minus_alphas_cumprod.gather(-1, t).contiguous()

    @torch.no_grad()
    def q_sample(self, x_start, t, noise=None):
        """ldm/diffusion/ddpm.py:407-412 as written — the default draw is torch.rand_like (uniform), not randn —
        on the fused q_sample kernel (sdb_q_sample): sqrt(a_t) * x_start + sqrt(1 - a_t) * noise per sample."""
        from . import ops
        if noise is None:
            noise = torch.rand_like(x_start)
        a, c = self.q_sample_coefficients(t)
        out = ops.q_sample(x_start.float().contiguous(), noise.float().contiguous(), a, c)
        return out if x_start.dtype == torch.float32 else out.to(x_start.dtype)

    @torch.no_grad()
    def decode_first_stage(self, z, predict_cids=False, force_not_quantize=False):
        """ldm/diffusion/ddpm.py:1083-1156: z / scale_factor then first_stage_model.decode; a VQModelInterface first
        stage is told whether to quantize (decode(z, force_not_quantize=predict_cids or force_not_quantize)).
        predict_cids needs the UNet's codebook-id head, which is not built.
        With split_input_params["patch_distributed_vq"] the latent is cut into crops (ks and stride reduced to its size),
        all crops are decoded as one batch and the images are stitched by the border-weighted fold at vqf times the size."""
        if predict_cids:
            raise NotImplementedError("decode_first_stage(predict_cids=True) needs the UNet n_embed codebook head, which is not built")
        z = 1. / self.scale_factor * z
        if isinstance(self.first_stage_model, VQModelInterface):
            decode = lambda v: self.first_stage_model.decode(v, force_not_quantize=predict_cids or force_not_quantize)
        else:
            decode = self.first_stage_model.decode
        if hasattr(self, "split_input_params") and self.split_input_params["patch_distributed_vq"]:
            return self._split_first_stage(z, decode, uf=self.split_input_params["vqf"])
        return decode(z)

    @torch.no_grad()
    def encode_first_stage(self, x):
        """ldm/diffusion/ddpm.py `encode_first_stage`: first_stage_model.encode(x) -> posterior (SURVEY.md §8 f3).
        With split_input_params["patch_distributed_vq"] the image is cut into crops, encoded as one batch and folded at
        1/vqf of the size; that needs a first stage whose encode returns a tensor (VQModelInterface, IdentityFirstStage)."""
        if hasattr(self, "split_input_params") and self.split_input_params["patch_distributed_vq"]:
            if isinstance(self.first_stage_model, AutoencoderKL):
                raise NotImplementedError("split_input_params: AutoencoderKL.encode returns a distribution, which cannot be folded")
            self.split_input_params["original_image_size"] = x.shape[-2:]
            return self._split_first_stage(x, self.first_stage_model.encode, df=self.split_input_params["vqf"])
        return self.first_stage_model.encode(x)

    @torch.no_grad()
    def get_first_stage_encoding(self, encoder_posterior, noise=None):
        """ldm/diffusion/ddpm.py `get_first_stage_encoding`: scale_factor * posterior.sample()."""
        if hasattr(encoder_posterior, "sample"):
            z = encoder_posterior.sample() if noise is None else encoder_posterior.sample(noise)
        elif isinstance(encoder_posterior, torch.Tensor):
            z = encoder_posterior
        else:
            raise NotImplementedError(f"encoder_posterior of type '{type(encoder_posterior)}' not yet implemented")
        return self.scale_factor * z

    @torch.no_grad()
    def img2img(self, image, cond, strength=0.75, ddim_steps=50, eta=0.0, unconditional_guidance_scale=1.0,
                unconditional_conditioning=None, noise=None, posterior_noise=None):
        """Encode -> DDIMSampler.stochastic_encode to step t_enc = strength * ddim_steps -> DDIMSampler.decode -> VAE
        decode (the mask-free img2img use of ldm/diffusion/ddim.py:208-243): latents and [-1,1] images.
        `posterior_noise` / `noise`: optional pre-drawn N(0,1) tensors for the posterior sample and the forward noising."""
        sampler = DDIMSampler(self)
        sampler.make_schedule(ddim_num_steps=ddim_steps, ddim_eta=eta, verbose=False)
        t_enc = max(1, min(ddim_steps, int(strength * ddim_steps)))
        z0 = self.get_first_stage_encoding(self.encode_first_stage(image), noise=posterior_noise)
        ts = torch.full((z0.shape[0],), t_enc - 1, device=z0.device, dtype=torch.long)
        zt = sampler.stochastic_encode(z0, ts, noise=noise)
        z = sampler.decode(zt, cond, t_enc, unconditional_guidance_scale=unconditional_guidance_scale,
                           unconditional_conditioning=unconditional_conditioning)
        return z, self.decode_first_stage(z)

    @torch.no_grad()
    def sample_log(self, cond, batch_size, ddim=True, ddim_steps=50, shape=(4, 64, 64), **kwargs):
        """ldm/diffusion/ddpm.py:1814-1826: DDIM-`ddim_steps`, or (ddim=False) the ancestral sampler with intermediates."""
        if not ddim:
            return self.sample(cond=cond, batch_size=batch_size, return_intermediates=True, shape=(batch_size, *shape), **kwargs)
        sampler = DDIMSampler(self)
        return sampler.sample(ddim_steps, batch_size, shape, cond, verbose=False, **kwargs)

    @torch.no_grad()
    def txt2img(self, cond, batch_size, ddim_steps=50, shape=(4, 64, 64), x_T=None, eta=0.0,
                unconditional_guidance_scale=1.0, unconditional_conditioning=None, plms=False, dpm_solver=False):
        """DDIM-`ddim_steps` (plms=True: PLMS-`ddim_steps`, as scripts/txt2img.py --plms; eta must be 0.  dpm_solver=True:
        DPM-Solver++(2M) with `ddim_steps` model evaluations, as --dpm_solver, eta ignored; it wins over plms, as in
        txt2img.py) + VAE decode: latents and [-1,1] images."""
        kw = dict(x_T=x_T, eta=eta, unconditional_guidance_scale=unconditional_guidance_scale,
                  unconditional_conditioning=unconditional_conditioning)
        if dpm_solver:
            z, _ = DPMSolverSampler(self).sample(ddim_steps, batch_size, shape, cond, verbose=False, **kw)
        elif plms:
            z, _ = PLMSSampler(self).sample(ddim_steps, batch_size, shape, cond, verbose=False, **kw)
        else:
            z, _ = self.sample_log(cond, batch_size, ddim=True, ddim_steps=ddim_steps, shape=shape, **kw)
        return z, self.decode_first_stage(z)

    # ---- ancestral sampler (ldm/diffusion/ddpm.py:1528-1793) -------------------------------------------------------------
    def _ancestral_supported(self):
        if self.parameterization != "eps":
            raise NotImplementedError("ancestral sampling is built for parameterization 'eps' only (got %r)" % self.parameterization)
        if self.shorten_cond_schedule:
            raise NotImplementedError("shorten_cond_schedule is not supported")

    def _ddpm_cache(self):
        """(posterior_std [T] on the host, [5, T] device table of sdb_ddpm_step) for the current schedule buffers.  Built once
        per schedule and rebuilt when any buffer it derives from is replaced (.to(), reassignment) or written in place
        (load_state_dict)."""
        src = (self.betas, self.sqrt_recip_alphas_cumprod, self.sqrt_recipm1_alphas_cumprod, self.posterior_mean_coef1,
               self.posterior_mean_coef2, self.posterior_log_variance_clipped)

        def build():
            # (0.5 * model_log_variance).exp() of p_sample, evaluated per element on a [1,1,1,1] fp32 host tensor: torch's CPU
            # exp is not correctly rounded, and the reference applies it to a [b,1,1,1] tensor, i.e. element by element
            lv = self.posterior_log_variance_clipped.detach().float().cpu()
            std = torch.tensor([float((0.5 * torch.full((1, 1, 1, 1), float(v))).exp()) for v in lv], dtype=torch.float32)
            dev = self.betas.device
            return std, torch.stack([b.detach().float().to(dev) for b in src[1:5]] + [std.to(dev)]).contiguous()
        return self._ddpm_tables.get(src, None, build)

    def posterior_std(self):
        """fp32 [T] host table exp(0.5 * posterior_log_variance_clipped[t]): the std p_sample adds noise with."""
        return self._ddpm_cache()[0]

    def ddpm_table(self):
        """[5, T] fp32 device table read by sdb_ddpm_step: sqrt_recip_alphas_cumprod, sqrt_recipm1_alphas_cumprod,
        posterior_mean_coef1, posterior_mean_coef2, posterior_std."""
        return self._ddpm_cache()[1]

    def _timesteps(self, t, x):
        return t if (t.dtype == torch.long and t.device == x.device and t.is_contiguous()) else t.to(x.device, torch.long).contiguous()

    @staticmethod
    def _extract(a, t, x_shape):
        """extract_into_tensor (ldm/modules/diffusionmodules/util.py:96-99)."""
        return a.gather(-1, t).reshape(t.shape[0], *((1,) * (len(x_shape) - 1)))

    @torch.no_grad()
    def predict_start_from_noise(self, x_t, t, noise):
        """sqrt_recip_alphas_cumprod[t] * x_t - sqrt_recipm1_alphas_cumprod[t] * noise, one kernel."""
        x = _f32_contiguous(x_t)
        _, x0 = ops.ddpm_step(x, self._timesteps(t, x), self.ddpm_table(), eps=_f32_contiguous(noise), want_x_prev=False, want_x0=True)
        return x0

    @torch.no_grad()
    def q_posterior(self, x_start, x_t, t):
        """(posterior mean coef1[t] * x_start + coef2[t] * x_t, posterior_variance[t], posterior_log_variance_clipped[t])."""
        x = _f32_contiguous(x_t)
        t = self._timesteps(t, x)
        mean, _ = ops.ddpm_step(x, t, self.ddpm_table(), x0=_f32_contiguous(x_start))
        return mean, self._extract(self.posterior_variance, t, x.shape), self._extract(self.posterior_log_variance_clipped, t, x.shape)

    def _model_eps(self, x, c, t, score_corrector, corrector_kwargs):
        model_out = self.apply_model(x, t, c)
        if score_corrector is not None:
            model_out = score_corrector.modify_score(self, model_out, x, t, c, **corrector_kwargs)
        return _f32_contiguous(model_out)

    def _ancestral_update(self, x, t, eps, clip, quantize_denoised, draw=None):
        """x0 -> (clamp) -> (first_stage_model.quantize) -> posterior mean (+ the noise `draw()` returns, drawn after quantize
        like the reference).  Returns (x_prev, x0)."""
        table = self.ddpm_table()
        if quantize_denoised:
            _, x0 = ops.ddpm_step(x, t, table, eps=eps, clip=clip, want_x_prev=False, want_x0=True)
            x0 = _f32_contiguous(self.first_stage_model.quantize(x0)[0])
            noise, temperature = draw() if draw is not None else (None, 1.)
            x_prev, _ = ops.ddpm_step(x, t, table, x0=x0, noise=noise, temperature=temperature)
            return x_prev, x0
        noise, temperature = draw() if draw is not None else (None, 1.)
        return ops.ddpm_step(x, t, table, eps=eps, noise=noise, clip=clip, temperature=temperature, want_x0=True)

    @torch.no_grad()
    def p_mean_variance(self, x, c, t, clip_denoised, return_codebook_ids=False, quantize_denoised=False, return_x0=False,
                        score_corrector=None, corrector_kwargs=None):
        """(model_mean, posterior_variance, posterior_log_variance[, x_recon]) of one denoising step."""
        self._ancestral_supported()
        if return_codebook_ids:
            raise NotImplementedError("return_codebook_ids is not supported")
        xf = _f32_contiguous(x)
        t = self._timesteps(t, xf)
        eps = self._model_eps(x, c, t, score_corrector, corrector_kwargs)
        mean, x_recon = self._ancestral_update(xf, t, eps, clip_denoised, quantize_denoised)
        var = self._extract(self.posterior_variance, t, xf.shape)
        log_var = self._extract(self.posterior_log_variance_clipped, t, xf.shape)
        return (mean, var, log_var, x_recon) if return_x0 else (mean, var, log_var)

    @torch.no_grad()
    def p_sample(self, x, c, t, clip_denoised=False, repeat_noise=False, return_codebook_ids=False, quantize_denoised=False,
                 return_x0=False, temperature=1., noise_dropout=0., score_corrector=None, corrector_kwargs=None):
        """model_mean + nonzero_mask * (0.5 * model_log_variance).exp() * noise_like(x.shape) * temperature, as one kernel
        (two with quantize_denoised).  The noise is drawn on every step, t == 0 included, exactly as the reference draws it."""
        self._ancestral_supported()
        if return_codebook_ids:
            raise NotImplementedError("return_codebook_ids is not supported")
        xf = _f32_contiguous(x)
        t = self._timesteps(t, xf)
        eps = self._model_eps(x, c, t, score_corrector, corrector_kwargs)

        def draw():
            if repeat_noise:
                noise = torch.randn((1, *x.shape[1:]), device=x.device).repeat(x.shape[0], *((1,) * (x.dim() - 1)))
            else:
                noise = torch.randn(x.shape, device=x.device)
            if noise_dropout > 0.:
                # dropout acts on noise * temperature and draws its own mask: form the product here, the kernel scales by 1
                return torch.nn.functional.dropout(noise * temperature, p=noise_dropout), 1.
            return noise, temperature

        x_prev, x0 = self._ancestral_update(xf, t, eps, clip_denoised, quantize_denoised, draw)
        return (x_prev, x0) if return_x0 else x_prev

    def _inpaint(self, x0, ts, mask, img):
        """img_orig = self.q_sample(x0, ts); img_orig * mask + (1. - mask) * img, fused (the DDIM sampler's blend)."""
        return DDIMSampler(self)._inpaint_blend(x0, ts, mask, img)

    @staticmethod
    def _slice_cond(cond, batch_size):
        if cond is None:
            return None
        if isinstance(cond, dict):
            return {k: cond[k][:batch_size] if not isinstance(cond[k], list) else [x[:batch_size] for x in cond[k]] for k in cond}
        return [c[:batch_size] for c in cond] if isinstance(cond, list) else cond[:batch_size]

    @torch.no_grad()
    def p_sample_loop(self, cond, shape, return_intermediates=False, x_T=None, verbose=True, callback=None, timesteps=None,
                      quantize_denoised=False, mask=None, x0=None, img_callback=None, start_T=None, log_every_t=None):
        """Ancestral sampling from t = timesteps - 1 down to 0; intermediates = [x_T] + img every log_every_t steps."""
        self._ancestral_supported()
        if not log_every_t:
            log_every_t = self.log_every_t
        device = self.betas.device
        b = shape[0]
        img = torch.randn(shape, device=device) if x_T is None else x_T
        intermediates = [img]
        if timesteps is None:
            timesteps = self.num_timesteps
        if start_T is not None:
            timesteps = min(timesteps, start_T)
        if mask is not None:
            assert x0 is not None
            assert x0.shape[2:3] == mask.shape[2:3]  # spatial size has to match
        for i in reversed(range(0, timesteps)):
            ts = torch.full((b,), i, device=device, dtype=torch.long)
            img = self.p_sample(img, cond, ts, clip_denoised=self.clip_denoised, quantize_denoised=quantize_denoised)
            if mask is not None:
                img = self._inpaint(x0, ts, mask, img)
            if i % log_every_t == 0 or i == timesteps - 1:
                intermediates.append(img)
            if callback:
                callback(i)
            if img_callback:
                img_callback(img, i)
        if return_intermediates:
            return img, intermediates
        return img

    @torch.no_grad()
    def sample(self, cond, batch_size=16, return_intermediates=False, x_T=None, verbose=True, timesteps=None,
               quantize_denoised=False, mask=None, x0=None, shape=None, **kwargs):
        """p_sample_loop over (batch_size, channels, image_size, image_size) unless `shape` is given."""
        if shape is None:
            shape = (batch_size, self.channels, self.image_size, self.image_size)
        cond = self._slice_cond(cond, batch_size)
        return self.p_sample_loop(cond, shape, return_intermediates=return_intermediates, x_T=x_T, verbose=verbose,
                                  timesteps=timesteps, quantize_denoised=quantize_denoised, mask=mask, x0=x0)

    @torch.no_grad()
    def progressive_denoising(self, cond, shape, verbose=True, callback=None, quantize_denoised=False, img_callback=None,
                              mask=None, x0=None, temperature=1., noise_dropout=0., score_corrector=None, corrector_kwargs=None,
                              batch_size=None, x_T=None, start_T=None, log_every_t=None):
        """Ancestral sampling that logs the predicted x0 (`x0_partial`) every log_every_t steps; `temperature` is one
        value or a list indexed by the timestep."""
        self._ancestral_supported()
        if not log_every_t:
            log_every_t = self.log_every_t
        timesteps = self.num_timesteps
        if batch_size is not None:
            b = batch_size
            shape = [batch_size] + list(shape)
        else:
            b = batch_size = shape[0]
        img = torch.randn(shape, device=self.device) if x_T is None else x_T
        intermediates = []
        cond = self._slice_cond(cond, batch_size)
        if start_T is not None:
            timesteps = min(timesteps, start_T)
        if isinstance(temperature, (int, float)):
            temperature = [float(temperature)] * timesteps
        for i in reversed(range(0, timesteps)):
            ts = torch.full((b,), i, device=self.device, dtype=torch.long)
            img, x0_partial = self.p_sample(img, cond, ts, clip_denoised=self.clip_denoised, quantize_denoised=quantize_denoised,
                                            return_x0=True, temperature=temperature[i], noise_dropout=noise_dropout,
                                            score_corrector=score_corrector, corrector_kwargs=corrector_kwargs)
            if mask is not None:
                assert x0 is not None
                img = self._inpaint(x0, ts, mask, img)
            if i % log_every_t == 0 or i == timesteps - 1:
                intermediates.append(x0_partial)
            if callback:
                callback(i)
            if img_callback:
                img_callback(img, i)
        return img, intermediates
