"""Drop-in `SelftokPipeline` for the encode / decode path of mimogpt/infer/SelftokPipeline.py.

Same constructor signature, attributes and method contracts as the reference class (SelftokPipeline.py:153-322):

    encoding(images [B,3,H,W] in [-1,1], device)            -> tokens [B,K] int64 on device          (:210-225)
    decoding(idx numpy [B,K] int64, device)                 -> images [B,3,H,W] in [0,1], self.dtype (:227-294)
    decoding_with_renderer(idx, device)                     -> same, one renderer pass               (:296-322)

Everything between the pixel tensors runs in the CUDA library behind include/selftok_b200.h -- the encoder / VQ / sampler /
renderer engine and, through `DeviceVAE`, both halves of the SD3 VAE (SURVEY 8f rank 1; diffusers' AutoencoderKL is only the
source of the VAE weights and the fallback for image sides other than 128 / 256 / 512).  The host keeps what the reference
keeps on the host: YAML/config, checkpoint loading, the CPU-generator noise draw (:262-264) and numpy<->tensor conversion.
The latent-boundary methods `encode_latents` / `decode_latents` / `render_latents` are the same calls without the VAE and are
what the headline of bench.py measures (its `extra.pixel_e2e` record goes through `encoding` / `decoding`).

Reference quirks consciously NOT reproduced (documented in DESIGN.md): cfg is not mutated; the sampler does not
re-run encoder+VQ on the noise every step (rectified_flow.py:212-215, dead for the output); quantizer.steps/count
buffers are not incremented; no host syncs inside the loop.
"""
from __future__ import annotations

import os
from typing import Dict, Optional

import numpy as np
import torch

from .capi import Engine, SelftokError
from .config import SelftokDims
from . import schedule as sched


class NormalizeToTensor(object):
    """uint8 HWC image -> float CHW in [-1,1]; same arithmetic as SelftokPipeline.py:85-97."""

    def __init__(self, reshape=True):
        self.reshape = reshape

    def __call__(self, image):
        image = np.array(image).astype(np.float32)
        image = (image / 127.5 - 1.0).astype(np.float32)
        if self.reshape:
            image = np.reshape(image, (image.shape[0], image.shape[1], -1))
        image = image.transpose((2, 0, 1))
        return torch.from_numpy(image)


def norm_ip(img, low, high):
    # SelftokPipeline.py:135-137
    img.clamp_(min=low, max=high)
    img.sub_(low).div_(max(high - low, 1e-5))


class SD3LatentFormat:
    """sd3/sd3_impls.py:133-144"""
    scale_factor = 1.5305
    shift_factor = 0.0609

    def process_in(self, latent):
        return (latent - self.shift_factor) * self.scale_factor

    def process_out(self, latent):
        return (latent / self.scale_factor) + self.shift_factor


class _LatentDist:
    """What `vae.encode(x, return_dict=False)[0]` is to the pipeline (diffusers DiagonalGaussianDistribution): `.mode()` is the
    call SelftokPipeline.encoding makes (:215); `.sample()` follows the same formula (logvar clamped to [-30, 20])."""

    def __init__(self, mean, logvar):
        self.mean, self.logvar = mean, logvar.clamp(-30.0, 20.0)

    def mode(self):
        return self.mean

    def sample(self, generator=None):
        eps = torch.randn(self.mean.shape, generator=generator, device=self.mean.device, dtype=self.mean.dtype)
        return self.mean + torch.exp(0.5 * self.logvar) * eps


class DeviceVAE:
    """`self.vae` with the call shape the pipeline uses (SelftokPipeline.py:215,288,316) on this repo's device VAE (csrc/vae.cu,
    fp32-faithful split-bf16 GEMMs): `decode` always; `encode` too when the state dict holds the encoder.* half and the images are
    128 / 256 / 512 pixels square -- otherwise it is delegated to `encoder_vae` (e.g. the diffusers AutoencoderKL).
    `state_dict`: SDVAE keys, or diffusers keys (`diffusers_keys=True`)."""

    ENCODE_SIDES = (128, 256, 512)

    def __init__(self, state_dict, device, encoder_vae=None, diffusers_keys: bool = False):
        from .capi import VaeDecoder
        sd = VaeDecoder.from_diffusers_keys(state_dict) if diffusers_keys else state_dict
        self.decoder = VaeDecoder(sd, device=device)
        self.has_encoder = any(k.startswith("encoder.") for k in sd)
        self.encoder_vae = encoder_vae

    def decode(self, z, return_dict=False):
        out = self.decoder.decode(z).to(z.dtype)
        return (out,)

    def encode(self, x, return_dict=False):
        if self.has_encoder and x.dim() == 4 and x.shape[2] == x.shape[3] and int(x.shape[2]) in self.ENCODE_SIDES:
            mean, logvar = self.decoder.encode(x, return_logvar=True)
            return (_LatentDist(mean.to(x.dtype), logvar.to(x.dtype)),)
        if self.encoder_vae is None:
            raise SelftokError("DeviceVAE.encode: images must be 128/256/512 square with encoder.* weights loaded, or pass "
                               "encoder_vae=... (e.g. diffusers.AutoencoderKL)")
        return self.encoder_vae.encode(x, return_dict=return_dict)

    def to(self, *a, **k):
        return self

    def eval(self):
        return self


def _load_vae(sd3_path, device, dtype):
    try:
        from diffusers import AutoencoderKL  # noqa: WPS433 (optional, external weights)
    except Exception as exc:  # pragma: no cover - diffusers is not in the build image
        raise SelftokError("the pixel-space API needs diffusers.AutoencoderKL (SD3 VAE) for the encoder side, or pass vae=...; use "
                           "the *_latents methods at the latent boundary instead") from exc
    vae = AutoencoderKL.from_pretrained(sd3_path, subfolder="vae")
    vae.to(device).to(dtype)
    vae.eval()
    # both halves on this repo's device VAE; the diffusers module stays as the fallback for other image sizes
    return DeviceVAE(vae.state_dict(), device, encoder_vae=vae, diffusers_keys=True)


def _decoder_state(state_dict: Dict, ema_decoder: bool) -> Dict[str, torch.Tensor]:
    """Checkpoint layout (SelftokPipeline.py:190-195): 'encoder.*' / 'model.*' (+ optional 'ema_state_dict' holding the
    MMDiT without the 'model.' prefix, loaded into a deep copy of self.model.model)."""
    sd = {k: v for k, v in state_dict.items() if torch.is_tensor(v)}
    if ema_decoder:
        ema = state_dict["ema_state_dict"]
        sd = {k: v for k, v in sd.items() if not k.startswith("model.")}
        sd.update({"model." + k: v for k, v in ema.items()})
    return sd


class ImageTokenizerShell:
    """`pipeline.model` of the reference is the ImageTokenizer nn.Module (SelftokPipeline.py:168-199): users reach for
    `state_dict()` / `load_state_dict()` / `eval()` on it.  The arithmetic lives in the CUDA engine, so this shell only keeps the
    checkpoint interface: `state_dict()` returns the tensors the engine was built from (re-read from `ckpt_path` when the engine
    came from the prepack cache), `load_state_dict()` rebuilds the engine from new weights and reports missing / unexpected keys
    against the path's state-dict contract (synth.state_dict_spec)."""

    def __init__(self, pipeline: "SelftokPipeline", state_dict):
        self._p = pipeline
        self._sd = state_dict

    def state_dict(self):
        if self._sd is None:
            self._sd = self._p._read_checkpoint()
        return {k: v for k, v in self._sd.items() if torch.is_tensor(v)}

    def load_state_dict(self, state_dict, strict: bool = False):
        from .synth import state_dict_spec
        spec = state_dict_spec(self._p.dims)
        missing = [k for k in spec if k not in state_dict]
        unexpected = [k for k in state_dict if torch.is_tensor(state_dict[k]) and (k.startswith("encoder.") or k.startswith("model."))
                      and k not in spec and not k.startswith("model.y_embedder.")]
        if strict and (missing or unexpected):
            raise RuntimeError(f"Error(s) in loading state_dict: missing {missing[:5]}..., unexpected {unexpected[:5]}...")
        if missing:
            raise SelftokError(f"checkpoint lacks tensors the path needs: {missing[:5]} ...")
        self._p._build_engine(state_dict, pack_path=None)
        self._sd = state_dict
        return missing, unexpected

    def eval(self):
        return self

    def to(self, *a, **k):
        return self

    def cuda(self, *a, **k):
        return self


class SelftokPipeline:
    def __init__(self, cfg, ckpt_path, sd3_path, datasize=256, start=1.0, cfg_scale=1, model_type="sd3",
                 dtype=torch.bfloat16, ema_decoder=False, device=None, *, state_dict=None, vae=None,
                 precision="auto", dims: Optional[SelftokDims] = None, prepack_cache: Optional[str] = None):
        """Same positional signature as the reference (SelftokPipeline.py:154).  Keyword-only extras: `state_dict` (in-memory
        checkpoint), `vae` (any object with the diffusers encode / decode call shape), `precision`, `dims`, and `prepack_cache`
        = a directory for the engine's packed device state: the second construction on the same checkpoint file skips
        torch.load, the uploads, the table MLPs and the operand packing (SURVEY 8f rank 2)."""
        self.cfg = cfg
        self.datasize = datasize
        self.model_type = model_type
        self.dtype = dtype
        if self.model_type != "sd3":
            raise ValueError(f"Unsupported MODEL_TYPE: {self.model_type}. Expected 'sd3'")
        # cfg_scale is stored and -- exactly as in the reference (SelftokPipeline.py:181 stores it, p_sample_loop is called
        # without uncond_scale: rectified_flow.py:173 default 1.0) -- NOT used by decoding(); the guided sampler the reference
        # implements in RectifiedFlow.sample_one_step is reachable through decode_latents(..., cfg_scale=...) / decoding_cfg().
        self.device = torch.device(device if device is not None else "cuda")
        # `datasize` (a CLI argument of the reference's test.py) sets the latent side: the models are built from the cfg but
        # run at datasize // 8 through the centre-cropped positional grids (models_ours.py:183-202, sd3/mmdit.py:877-896)
        self.dims = dims if dims is not None else SelftokDims.from_cfg(cfg, datasize)
        if not self.dims.renderer:
            # the sampler call hard-codes context_see_xt=True whatever the YAML says (SelftokPipeline.py:259); the renderer
            # call passes nothing, i.e. False (SelftokPipeline.py:310, sd3/mmdit.py:1533) -- the engine does that by itself
            import dataclasses
            self.dims = dataclasses.replace(self.dims, context_see_xt=True)
        if self.dims.latent * 8 != int(datasize):
            raise SelftokError(f"datasize {datasize} does not match the engine geometry (latent side {self.dims.latent})")
        self.vae = vae
        if self.vae is None and sd3_path:
            self.vae = _load_vae(sd3_path, self.device, self.dtype)
        self.ema_decoder = ema_decoder
        self.K = self.dims.K
        self.count = 0
        self.count_cfg = 0
        self.start = start
        self.cfg_scale = cfg_scale
        p = cfg["tokenizer"]["params"] if cfg is not None else {}
        self.cut_of_k = p.get("cut_of_k", None) or None
        if self.cut_of_k is not None:
            raise SelftokError("cut_of_k is not on the shipped path")
        self.ckpt_path = ckpt_path
        self._precision_req = precision
        self._steps = 50
        pack_path = None
        if prepack_cache and ckpt_path and os.path.exists(ckpt_path):
            import hashlib
            st = os.stat(ckpt_path)
            key = hashlib.sha1(repr((os.path.abspath(ckpt_path), st.st_size, st.st_mtime_ns, self.dims, precision, self._steps,
                                     float(start), bool(ema_decoder))).encode()).hexdigest()[:20]
            os.makedirs(prepack_cache, exist_ok=True)
            pack_path = os.path.join(prepack_cache, f"selftok_{key}.stkpack")
        print("Loading all...")
        self.engine = None
        if pack_path and os.path.exists(pack_path) and os.path.exists(pack_path + ".json") and state_dict is None:
            self._build_engine(None, pack_path)                      # no torch.load at all
        else:
            if state_dict is None:
                state_dict = self._read_checkpoint()
            self._build_engine(state_dict, pack_path)
        self.model = ImageTokenizerShell(self, state_dict)
        self.diti = sched.DiTiCont(1000, self.dims.K, self.dims.stages, self.dims.k_per_stage)
        self.flow = self.engine.tables           # scheduled t / dt / k tables (RectifiedFlow.make_schedule equivalent)
        self.cond_vary = True
        self.saved_images = 8

    def _read_checkpoint(self):
        return torch.load(self.ckpt_path, map_location="cpu")        # SelftokPipeline.py:190

    def _build_engine(self, state_dict, pack_path) -> None:
        sd = None if state_dict is None else _decoder_state(state_dict, self.ema_decoder)
        new = Engine(self.dims, sd, device=self.device, precision=self._precision_req, steps=self._steps, start=self.start,
                     pack_path=pack_path)
        if self.engine is not None:
            self.engine.close()
        self.engine = new
        self.flow = self.engine.tables

    # ------------------------------------------------------------------ latent-boundary API (the measured path)
    @torch.no_grad()
    def encode_latents(self, x_0: torch.Tensor) -> torch.Tensor:
        """x_0 = SD3LatentFormat().process_in(vae.encode(images).mode()).float() -> tokens [B,K] int64 (device)."""
        return self.engine.encode(x_0)

    @torch.no_grad()
    def decode_latents(self, idx, noise: Optional[torch.Tensor] = None, cfg_scale: Optional[float] = None, *,
                       n_tokens=None) -> torch.Tensor:
        """tokens -> pred_x0 latents after the 50-step Euler loop.  `noise` defaults to the reference's draw:
        torch.randn on the CPU global generator, then moved to the device (SelftokPipeline.py:262-264).
        cfg_scale (None / 1: plain sampler): classifier-free guidance as RectifiedFlow.sample_one_step implements it
        (rectified_flow.py:280-289) -- an explicit argument here because the reference pipeline never forwards its own.
        n_tokens (an int, or one value per image in [1, K]): decode image b from its first n_tokens[b] tokens only, as
        p_sample_loop(..., super_mask = arange(K) < n) does (rectified_flow.py:227-228); later ids are never read."""
        token_idx = torch.from_numpy(idx) if isinstance(idx, np.ndarray) else idx
        B = token_idx.shape[0]
        latent_dim = self.datasize // 8
        if noise is None:
            noise = torch.randn(B, self.dims.in_channels, latent_dim, latent_dim)
        if cfg_scale is None or float(cfg_scale) == 1.0:
            out = self.engine.decode(token_idx, noise, n_tokens=n_tokens)
        else:
            out = self.engine.decode_cfg(token_idx, noise, float(cfg_scale), n_tokens=n_tokens)
        self._raise_on_bad_ids(token_idx)
        return out

    def _raise_on_bad_ids(self, token_idx) -> None:
        # `codebook[idx]` raises for ids outside the codebook in the reference (vector_quantize_pytorch.py:310-314); host ids were
        # checked before the launch, device ids are counted by the lookup kernel
        if token_idx.is_cuda and self.engine.id_errors() > 0:
            raise IndexError("token id out of range for the codebook")

    @torch.no_grad()
    def render_latents(self, idx, *, n_tokens=None) -> torch.Tensor:
        """n_tokens: render image b from its first n_tokens[b] tokens (MMDiT_Renderer.forward(..., mask=...), sd3/mmdit.py:1529)."""
        token_idx = torch.from_numpy(idx) if isinstance(idx, np.ndarray) else idx
        out = self.engine.render(token_idx, n_tokens=n_tokens)
        self._raise_on_bad_ids(token_idx)
        return out

    # ------------------------------------------------------------------ data-parallel entry points (one process per GPU)
    @torch.no_grad()
    def encode_latents_sharded(self, x_0_global: torch.Tensor) -> torch.Tensor:
        """Every rank passes the SAME global batch (host tensor); each encodes its contiguous slice (dist.shard_slice) and the
        token ids are all-gathered (NCCL over NVLink: [B/G, K] int64 per rank -- the path's only collective, SURVEY 8e).
        Returns the global [B, K] ids on every rank; identical, bit for bit, to a single-process encode."""
        from . import dist as D
        rank, world = D.world()
        lo, hi = D.shard_slice(x_0_global.shape[0], rank, world)
        return D.gather_tokens(self.engine.encode(x_0_global[lo:hi]), x_0_global.shape[0])

    @torch.no_grad()
    def decode_latents_sharded(self, idx_global, noise_global: Optional[torch.Tensor] = None, seed: Optional[int] = None,
                               gather: bool = True) -> torch.Tensor:
        """Global tokens [B, K] on every rank -> this rank's slice decoded; `gather` returns the global latents on every rank.
        The initial noise is ONE host draw for the whole batch (dist.host_noise(seed)), sliced per rank."""
        from . import dist as D
        token_idx = torch.from_numpy(idx_global) if isinstance(idx_global, np.ndarray) else idx_global
        n = token_idx.shape[0]
        rank, world = D.world()
        lo, hi = D.shard_slice(n, rank, world)
        if noise_global is None:
            latent_dim = self.datasize // 8
            noise_global = D.host_noise(n, (self.dims.in_channels, latent_dim, latent_dim), 0 if seed is None else seed)
        out = self.engine.decode(token_idx[lo:hi], noise_global[lo:hi])
        return D.gather_rows(out, n) if gather else out

    # ------------------------------------------------------------------ reference API (pixel space, needs the SD3 VAE)
    def _need_vae(self):
        if self.vae is None:
            raise SelftokError("no VAE: pass sd3_path (diffusers AutoencoderKL) or vae=..., or use the *_latents methods")

    def encoding(self, images, device):
        print("Begin encoding.")
        self._need_vae()
        images = images.to(dtype=self.dtype, device=device)
        x_0 = self.vae.encode(images, return_dict=False)[0].mode()
        x_0 = SD3LatentFormat().process_in(x_0)
        x_0 = x_0.to(torch.float32)
        tokens = self.encode_latents(x_0)
        print("End encoding.")
        return tokens

    @torch.no_grad()
    def decoding(self, idx, device, *, n_tokens=None):
        print("Begin decoding.")
        self._need_vae()
        pred_x0 = self.decode_latents(idx, n_tokens=n_tokens)
        pred_x0_out = SD3LatentFormat().process_out(pred_x0).to(self.dtype)
        recons = self.vae.decode(pred_x0_out, return_dict=False)[0]
        norm_ip(recons, -1, 1)
        print("End decoding.")
        return recons

    @torch.no_grad()
    def decoding_cfg(self, idx, device, cfg_scale: Optional[float] = None, *, n_tokens=None):
        """decoding() with the guided sampler (cfg_scale defaults to the constructor's)."""
        self._need_vae()
        pred_x0 = self.decode_latents(idx, cfg_scale=self.cfg_scale if cfg_scale is None else cfg_scale, n_tokens=n_tokens)
        recons = self.vae.decode(SD3LatentFormat().process_out(pred_x0).to(self.dtype), return_dict=False)[0]
        norm_ip(recons, -1, 1)
        return recons

    @torch.no_grad()
    def decoding_with_renderer(self, idx, device, *, n_tokens=None):
        print("Begin decoding with Renderer.")
        self._need_vae()
        pred_x0 = self.render_latents(idx, n_tokens=n_tokens)
        pred_x0_out = SD3LatentFormat().process_out(pred_x0).to(self.dtype)
        recons = self.vae.decode(pred_x0_out)[0]
        norm_ip(recons, -1, 1)
        print("End decoding with Renderer.")
        return recons
