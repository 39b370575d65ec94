"""ctypes binding of include/selftok_b200.h (libselftok_b200.so) — the only way Python reaches the kernels.

There is deliberately no fallback: if the library is missing or no sm_100 GPU is visible, construction raises
(`SelftokError`).  PyTorch appears here only as the owner of device memory (`tensor.data_ptr()`) and of the
current stream handle.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional

import numpy as np
import torch

from . import schedule as sched
from .config import SelftokDims

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libselftok_b200.so")
PREC = {"fp32": 0, "bf16x3": 1, "bf16": 2, "fp16": 3}

# every symbol include/selftok_b200.h declares (tests check the .so exports exactly these)
SYMBOLS = [
    "selftok_create", "selftok_destroy", "selftok_last_error", "selftok_version", "selftok_load_tensor",
    "selftok_set_schedule", "selftok_finalize", "selftok_export_packed", "selftok_import_packed", "selftok_encode", "selftok_vq_argmax", "selftok_lookup",
    "selftok_set_cfg_schedule", "selftok_decode", "selftok_decode_cfg", "selftok_dit_velocity", "selftok_render", "selftok_encode_host", "selftok_decode_host",
    "selftok_decode_prefix", "selftok_render_prefix", "selftok_dit_velocity_prefix",
    "selftok_render_host", "selftok_id_errors", "selftok_workspace_bytes", "selftok_set_workspace", "selftok_last_launch_count", "selftok_device_bytes", "selftok_set_use_graph",
    "selftok_set_profile", "selftok_get_profile", "selftok_k_linear_f32", "selftok_k_linear_tc", "selftok_k_set_gemm_ctas", "selftok_k_ln_mod_f32", "selftok_k_attention_f32",
    "selftok_k_attention_tc",
    "selftok_vae_create", "selftok_vae_destroy", "selftok_vae_load_tensor", "selftok_vae_finalize", "selftok_vae_decode", "selftok_vae_encode", "selftok_vae_device_bytes",
]


class SelftokError(RuntimeError):
    pass


class _Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "K", "latent", "in_channels", "enc_patch", "enc_hidden", "enc_heads", "enc_depth", "enc_qdim", "enc_qheads",
        "enc_pos_max", "codebook_size", "code_dim", "dit_depth", "dit_patch", "dit_pos_max", "renderer",
        "context_see_xt", "precision", "device")]


_lib = None


def load_library(path: Optional[str] = None) -> C.CDLL:
    """dlopen the CUDA library.  Raises if it has not been built (python -m selftoktokenizer_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    path = path or os.environ.get("SELFTOK_B200_LIB", _LIB_PATH)
    if not os.path.exists(path):
        raise SelftokError(f"{path} not found: build it with `python -m selftoktokenizer_b200.build` "
                           "(selftok_b200 has no CPU / PyTorch fallback)")
    lib = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    lib.selftok_last_error.restype = C.c_char_p
    lib.selftok_version.restype = C.c_char_p
    lib.selftok_create.argtypes = [C.POINTER(_Config), C.POINTER(vp)]
    lib.selftok_destroy.argtypes = [vp]
    lib.selftok_load_tensor.argtypes = [vp, C.c_char_p, vp, i32, i32, C.POINTER(i64), i32]
    lib.selftok_set_schedule.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    lib.selftok_finalize.argtypes = [vp, vp]
    lib.selftok_export_packed.argtypes = [vp, C.c_char_p]
    lib.selftok_import_packed.argtypes = [vp, C.c_char_p]
    lib.selftok_encode.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    lib.selftok_vq_argmax.argtypes = [vp, vp, i64, vp, vp, vp]
    lib.selftok_lookup.argtypes = [vp, vp, i32, vp, vp]
    lib.selftok_decode.argtypes = [vp, vp, vp, i32, i32, vp, vp]
    lib.selftok_set_cfg_schedule.argtypes = [vp, vp]
    lib.selftok_decode_cfg.argtypes = [vp, vp, vp, i32, i32, C.c_float, vp, vp]
    lib.selftok_dit_velocity.argtypes = [vp, vp, vp, i32, i32, vp, vp]
    lib.selftok_render.argtypes = [vp, vp, i32, vp, vp]
    lib.selftok_decode_prefix.argtypes = [vp, vp, vp, vp, i32, i32, C.c_float, vp, vp]
    lib.selftok_render_prefix.argtypes = [vp, vp, vp, i32, vp, vp]
    lib.selftok_dit_velocity_prefix.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp]
    lib.selftok_encode_host.argtypes = [vp, vp, i32, vp, vp]
    lib.selftok_decode_host.argtypes = [vp, vp, vp, i32, i32, vp, vp]
    lib.selftok_render_host.argtypes = [vp, vp, i32, vp, vp]
    lib.selftok_id_errors.argtypes = [vp, vp]
    lib.selftok_id_errors.restype = i64
    lib.selftok_workspace_bytes.argtypes = [vp, i32, i32]
    lib.selftok_workspace_bytes.restype = i64
    lib.selftok_set_workspace.argtypes = [vp, i32, vp, C.c_size_t]
    lib.selftok_last_launch_count.argtypes = [vp]
    lib.selftok_last_launch_count.restype = i64
    lib.selftok_device_bytes.argtypes = [vp]
    lib.selftok_device_bytes.restype = i64
    lib.selftok_set_use_graph.argtypes = [vp, i32]
    lib.selftok_set_profile.argtypes = [vp, i32]
    lib.selftok_get_profile.argtypes = [vp, vp, vp]
    lib.selftok_k_linear_f32.argtypes = [vp, vp, vp, vp, i64, i32, i32, i32, vp]
    lib.selftok_k_linear_tc.argtypes = [vp, vp, vp, vp, i64, i32, i32, i32, vp]
    lib.selftok_k_set_gemm_ctas.argtypes = [i32]
    lib.selftok_k_ln_mod_f32.argtypes = [vp, vp, vp, i64, i32, vp, i64, i32, vp]
    lib.selftok_k_attention_f32.argtypes = [vp, i64, vp, vp, i64, i32, vp, vp, i64, i32, vp, i64, i32, i32, i32, i32, vp]
    lib.selftok_k_attention_tc.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp]
    lib.selftok_vae_create.argtypes = [i32, i32, C.POINTER(vp)]
    lib.selftok_vae_destroy.argtypes = [vp]
    lib.selftok_vae_load_tensor.argtypes = [vp, C.c_char_p, vp, i32, C.POINTER(i64), i32]
    lib.selftok_vae_finalize.argtypes = [vp, vp]
    lib.selftok_vae_decode.argtypes = [vp, vp, i32, i32, i32, vp, i32, vp]
    lib.selftok_vae_encode.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp]
    lib.selftok_vae_device_bytes.argtypes = [vp]
    lib.selftok_vae_device_bytes.restype = i64
    for name in SYMBOLS:
        getattr(lib, name)          # AttributeError here == header / library drift
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != 0:
        msg = load_library().selftok_last_error()
        raise SelftokError(f"selftok_b200 status {status}: {msg.decode() if msg else '?'}")


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class Engine:
    """One handle (`selftok_handle_t`) on one device: weights, static tables, workspaces, CUDA graphs."""

    def __init__(self, dims: SelftokDims, state_dict: Optional[Dict[str, torch.Tensor]], device="cuda:0", precision: str = "auto",
                 steps: int = 50, start: float = 1.0, pack_path: Optional[str] = None):
        """`pack_path`: prepack cache file (selftok_export_packed / selftok_import_packed).  If it exists the engine is
        restored from it and `state_dict` may be None (no torch.load of the fp32 checkpoint at all); otherwise the engine is
        built from `state_dict` and, when a path is given, exported there.  The precision chosen by 'auto' is kept in a
        JSON sidecar next to the file."""
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise SelftokError("no CUDA device: selftok_b200 has no CPU fallback")
        self.dims = dims
        self.device = torch.device(device)
        probe = False
        self.restored_from_pack = False
        side = pack_path + ".json" if pack_path else None
        if pack_path and os.path.exists(pack_path) and os.path.exists(side):
            import json
            meta = json.load(open(side))
            if meta.get("requested") == precision and meta.get("steps") == (1 if dims.renderer else steps) and meta.get("start") == start:
                precision = meta["precision"]
                self.restored_from_pack = True
        if state_dict is None and not self.restored_from_pack:
            raise SelftokError("Engine: no state_dict and no usable prepack cache")
        requested = precision if not self.restored_from_pack else meta["requested"]
        if precision == "auto":
            # One-pass renderer: its output IS one network evaluation (single-pass fp16 measures 1.05e-3 there), and a pass
            # costs 1/50 of a decode, so it always runs the fp32-faithful split-bf16 arithmetic (5e-5).
            # 50-step sampler: single-pass IEEE-half operands (2.9e-4 on the final latents of the well-conditioned synthetic
            # checkpoint) -- but only after a PROBE on THIS checkpoint: the reference is fp32, and outlier channels /
            # heavy-tailed weights can push half-precision operands past the 1e-3 bar (tests: mid_stress fixture).  The
            # probe evaluates the velocity at the first and last sampler step in fp16 and in bf16x3 on one seeded image and
            # keeps fp16 only if they agree to `AUTO_PROBE_TOL`; otherwise the engine runs bf16x3.
            precision = "bf16x3" if dims.renderer else "fp16"
            probe = not dims.renderer
        self.precision = precision
        self.auto_probe = None          # {"dev": max-abs velocity deviation fp16 vs bf16x3, "tol": ..., "chosen": ...}
        dims.validate()
        cfg = _Config(K=dims.K, latent=dims.latent, in_channels=dims.in_channels, enc_patch=dims.enc_patch,
                      enc_hidden=dims.enc_hidden, enc_heads=dims.enc_heads, enc_depth=dims.enc_depth,
                      enc_qdim=dims.enc_qdim, enc_qheads=dims.enc_qheads, enc_pos_max=dims.enc_pos_max,
                      codebook_size=dims.codebook_size, code_dim=dims.code_dim, dit_depth=dims.dit_depth,
                      dit_patch=dims.dit_patch, dit_pos_max=dims.dit_pos_max, renderer=int(dims.renderer),
                      context_see_xt=int(dims.context_see_xt), precision=PREC[precision],
                      device=self.device.index or 0)
        h = C.c_void_p()
        check(self.lib.selftok_create(C.byref(cfg), C.byref(h)))
        self.h = h
        try:
            if not self.restored_from_pack:
                self._load(state_dict)
            if dims.renderer:
                # MMDiT_Renderer: one pass at t = 1000 with all K tokens visible (sd3/mmdit.py:1523)
                tb = sched.make_tables(dims.K, dims.stages, dims.k_per_stage, 1)
                self.steps = 1
                t_freq = sched.renderer_t_freq()
                k = np.full(1, dims.K - 1, dtype=np.int32)
            else:
                tb = sched.make_tables(dims.K, dims.stages, dims.k_per_stage, steps, start)
                self.steps = steps
                t_freq = tb.t_freq
                k = tb.k.numpy().astype(np.int32)
            self.tables = tb
            t = np.ascontiguousarray(tb.t.numpy(), dtype=np.float32)
            dt = np.ascontiguousarray(tb.dt.numpy(), dtype=np.float32)
            tf = np.ascontiguousarray(t_freq.numpy(), dtype=np.float32)
            pf = np.ascontiguousarray(tb.pos_freq.numpy(), dtype=np.float32)
            if self.restored_from_pack:
                with torch.cuda.device(self.device):
                    check(self.lib.selftok_import_packed(self.h, pack_path.encode()))
                self.auto_probe = meta.get("auto_probe")
            else:
                check(self.lib.selftok_set_schedule(self.h, self.steps, t.ctypes.data, dt.ctypes.data, k.ctypes.data,
                                                    tf.ctypes.data, pf.ctypes.data))
                if not dims.renderer:                       # tables of the guided sampler's unconditional branch (44 MB)
                    tu = np.ascontiguousarray(tb.t_freq_uncond.numpy(), dtype=np.float32)
                    check(self.lib.selftok_set_cfg_schedule(self.h, tu.ctypes.data))
                with torch.cuda.device(self.device):
                    check(self.lib.selftok_finalize(self.h, _stream_ptr(self.device)))
                if probe:
                    self._auto_probe(state_dict, steps, start)
                if pack_path:
                    import json
                    with torch.cuda.device(self.device):
                        check(self.lib.selftok_export_packed(self.h, pack_path.encode()))
                    json.dump({"requested": requested, "precision": self.precision, "steps": self.steps, "start": start,
                               "auto_probe": self.auto_probe}, open(side, "w"))
        except Exception:
            self.close()
            raise

    AUTO_PROBE_TOL = 1.5e-3     # max-abs velocity deviation; the 50-step result deviates ~0.4x of it (measured ratio)

    def _auto_probe(self, state_dict, steps, start) -> None:
        from . import synth
        d = self.dims
        ref = Engine(d, state_dict, device=self.device, precision="bf16x3", steps=steps, start=start)
        try:
            x = synth.synth_tensor("auto.probe.x", (1, d.in_channels, d.latent, d.latent), "emb", 1.0)
            tok = (torch.arange(d.K, dtype=torch.int64) * 2654435761 % d.codebook_size).reshape(1, d.K)
            dev = 0.0
            for st in (0, self.steps - 1):
                dev = max(dev, float((self.dit_velocity(tok, x, st) - ref.dit_velocity(tok, x, st)).abs().max()))
            ok = dev <= self.AUTO_PROBE_TOL and dev == dev          # NaN -> not ok
            self.auto_probe = {"dev": dev, "tol": self.AUTO_PROBE_TOL, "chosen": "fp16" if ok else "bf16x3"}
            if not ok:                                              # keep the fp32-faithful engine, drop the fp16 one
                self.h, ref.h = ref.h, self.h
                self.precision = "bf16x3"
        finally:
            ref.close()

    def _load(self, sd: Dict[str, torch.Tensor]) -> None:
        for name, t in sd.items():
            if not torch.is_tensor(t) or not t.is_floating_point() or t.numel() == 0:
                continue
            if not (name.startswith("encoder.") or name.startswith("model.")):
                continue
            t = t.detach()
            if t.dtype != torch.float32 or not t.is_contiguous():
                t = t.to(torch.float32).contiguous()
            shape = (C.c_int64 * max(t.dim(), 1))(*t.shape)
            is_dev = int(t.is_cuda)
            if is_dev and t.device != self.device:
                t = t.to(self.device)
            check(self.lib.selftok_load_tensor(self.h, name.encode(), t.data_ptr(), 0, t.dim(), shape, is_dev))

    # ------------------------------------------------------------------ hot path (device tensors)
    def _dev(self, t: torch.Tensor, dtype) -> torch.Tensor:
        return t.to(device=self.device, dtype=dtype).contiguous()

    # The C entry points take raw pointers and a batch size only: shapes are checked HERE so that a latent of another
    # resolution (datasize != the engine's geometry) or a short token row fails loudly instead of reading out of bounds.
    def _check_latent(self, x: torch.Tensor, what: str) -> None:
        d = self.dims
        want = (d.in_channels, d.latent, d.latent)
        if x.dim() != 4 or tuple(x.shape[1:]) != want or x.shape[0] < 1:
            raise SelftokError(f"{what}: expected [B, {want[0]}, {want[1]}, {want[2]}] latents for this engine "
                               f"(image side {8 * d.latent}), got {tuple(x.shape)}")

    def _check_tokens(self, tokens: torch.Tensor, what: str, batch: Optional[int] = None, is_output: bool = False,
                      n_tokens: Optional[torch.Tensor] = None) -> None:
        if tokens.dim() != 2 or tokens.shape[1] != self.dims.K or tokens.shape[0] < 1:
            raise SelftokError(f"{what}: expected [B, {self.dims.K}] token ids, got {tuple(tokens.shape)}")
        if batch is not None and tokens.shape[0] != batch:
            raise SelftokError(f"{what}: {tokens.shape[0]} token rows for a batch of {batch}")
        if not tokens.is_cuda and not is_output:
            # ids outside the codebook are an error in the reference (`codebook[idx]` raises).  Host tensors are checked here
            # for free; device tensors are checked by the kernel (NaN rows + counter, see `id_errors`).  With a token prefix
            # only the ids inside each image's prefix are read.
            if n_tokens is not None:
                tokens = tokens[torch.arange(self.dims.K)[None, :] < n_tokens[:, None].long()]
                if tokens.numel() == 0:
                    return
            lo, hi = int(tokens.min()), int(tokens.max())
            if lo < 0 or hi >= self.dims.codebook_size:
                raise SelftokError(f"{what}: token id out of range [0, {self.dims.codebook_size}): min {lo}, max {hi}")

    def _n_tokens(self, n_tokens, B: int) -> Optional[torch.Tensor]:
        """Per-image prefix lengths (an int for the whole batch, or B values) -> int32 host tensor [B]; None stays None.
        The range [1, K] is checked by the library; values are clamped to [-1, K + 1] first only so that they fit int32."""
        if n_tokens is None:
            return None
        n = torch.as_tensor(n_tokens, dtype=torch.int64).cpu().reshape(-1)
        if n.numel() == 1:
            n = n.expand(B)
        if n.numel() != B:
            raise SelftokError(f"n_tokens: {n.numel()} prefix lengths for a batch of {B}")
        return n.clamp(-1, self.dims.K + 1).to(torch.int32).contiguous()

    def id_errors(self) -> int:
        """Synchronises and returns how many out-of-range token ids the device lookups saw since the last query."""
        with torch.cuda.device(self.device):
            n = int(self.lib.selftok_id_errors(self.h, _stream_ptr(self.device)))
        if n < 0:
            raise SelftokError("selftok_id_errors failed")
        return n

    def encode(self, x0: torch.Tensor, return_aux: bool = False):
        """x0 [B,C,h,w] fp32 latents -> tokens [B,K] int64 (device)."""
        d = self.dims
        self._check_latent(x0, "encode")
        x0 = self._dev(x0, torch.float32)
        B = x0.shape[0]
        tokens = torch.empty(B, d.K, dtype=torch.int64, device=self.device)
        outs_q = torch.empty(B, d.K, d.code_dim, dtype=torch.float32, device=self.device) if return_aux else None
        feats = torch.empty(B, d.K, d.enc_qdim, dtype=torch.float32, device=self.device) if return_aux else None
        with torch.cuda.device(self.device):
            check(self.lib.selftok_encode(self.h, x0.data_ptr(), B, tokens.data_ptr(), _ptr(outs_q), _ptr(feats),
                                          _stream_ptr(self.device)))
        return (tokens, outs_q, feats) if return_aux else tokens

    def vq_argmax(self, z: torch.Tensor, with_outs_q: bool = True):
        z = self._dev(z, torch.float32)
        R = z.numel() // self.dims.enc_qdim
        ids = torch.empty(R, dtype=torch.int64, device=self.device)
        outs_q = torch.empty(R, self.dims.code_dim, dtype=torch.float32, device=self.device) if with_outs_q else None
        with torch.cuda.device(self.device):
            check(self.lib.selftok_vq_argmax(self.h, z.data_ptr(), R, ids.data_ptr(), _ptr(outs_q), _stream_ptr(self.device)))
        return ids, outs_q

    def lookup(self, tokens: torch.Tensor) -> torch.Tensor:
        self._check_tokens(tokens, "lookup")
        tokens = self._dev(tokens, torch.int64)
        B = tokens.shape[0]
        out = torch.empty(B, self.dims.K, self.dims.code_dim, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self.lib.selftok_lookup(self.h, tokens.data_ptr(), B, out.data_ptr(), _stream_ptr(self.device)))
        return out

    # n_tokens (decode, decode_cfg, dit_velocity, render): decode image b from its first n_tokens[b] tokens only -- an int for
    # the whole batch or B values in [1, K]; ids after each prefix are never read.  None: all K tokens (the plain entry points).
    def decode(self, tokens: torch.Tensor, noise: torch.Tensor, steps: Optional[int] = None, n_tokens=None) -> torch.Tensor:
        self._check_latent(noise, "decode (noise)")
        n = self._n_tokens(n_tokens, noise.shape[0])
        self._check_tokens(tokens, "decode", noise.shape[0], n_tokens=n)
        tokens = self._dev(tokens, torch.int64)
        noise = self._dev(noise, torch.float32)
        B = tokens.shape[0]
        out = torch.empty_like(noise)
        with torch.cuda.device(self.device):
            if n is None:
                check(self.lib.selftok_decode(self.h, tokens.data_ptr(), noise.data_ptr(), B, steps or self.steps,
                                              out.data_ptr(), _stream_ptr(self.device)))
            else:
                check(self.lib.selftok_decode_prefix(self.h, tokens.data_ptr(), n.data_ptr(), noise.data_ptr(), B, steps or self.steps,
                                                     1.0, out.data_ptr(), _stream_ptr(self.device)))
        return out

    def decode_cfg(self, tokens: torch.Tensor, noise: torch.Tensor, cfg_scale: float, steps: Optional[int] = None,
                   n_tokens=None) -> torch.Tensor:
        """Guided sampler: the reference's p_sample_loop(..., uncond_scale=cfg_scale) (rectified_flow.py:280-289)."""
        self._check_latent(noise, "decode_cfg (noise)")
        n = self._n_tokens(n_tokens, noise.shape[0])
        self._check_tokens(tokens, "decode_cfg", noise.shape[0], n_tokens=n)
        tokens = self._dev(tokens, torch.int64)
        noise = self._dev(noise, torch.float32)
        out = torch.empty_like(noise)
        with torch.cuda.device(self.device):
            if n is None:
                check(self.lib.selftok_decode_cfg(self.h, tokens.data_ptr(), noise.data_ptr(), tokens.shape[0], steps or self.steps,
                                                  float(cfg_scale), out.data_ptr(), _stream_ptr(self.device)))
            else:
                check(self.lib.selftok_decode_prefix(self.h, tokens.data_ptr(), n.data_ptr(), noise.data_ptr(), tokens.shape[0],
                                                     steps or self.steps, float(cfg_scale), out.data_ptr(), _stream_ptr(self.device)))
        return out

    def dit_velocity(self, tokens: torch.Tensor, x: torch.Tensor, step: int, n_tokens=None) -> torch.Tensor:
        self._check_latent(x, "dit_velocity")
        n = self._n_tokens(n_tokens, x.shape[0])
        self._check_tokens(tokens, "dit_velocity", x.shape[0], n_tokens=n)
        tokens = self._dev(tokens, torch.int64)
        x = self._dev(x, torch.float32)
        out = torch.empty_like(x)
        with torch.cuda.device(self.device):
            if n is None:
                check(self.lib.selftok_dit_velocity(self.h, tokens.data_ptr(), x.data_ptr(), tokens.shape[0], step,
                                                    out.data_ptr(), _stream_ptr(self.device)))
            else:
                check(self.lib.selftok_dit_velocity_prefix(self.h, tokens.data_ptr(), n.data_ptr(), x.data_ptr(), tokens.shape[0], step,
                                                           out.data_ptr(), _stream_ptr(self.device)))
        return out

    def render(self, tokens: torch.Tensor, n_tokens=None) -> torch.Tensor:
        n = self._n_tokens(n_tokens, tokens.shape[0]) if tokens.dim() == 2 else None
        self._check_tokens(tokens, "render", n_tokens=n)
        tokens = self._dev(tokens, torch.int64)
        d = self.dims
        out = torch.empty(tokens.shape[0], d.in_channels, d.latent, d.latent, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            if n is None:
                check(self.lib.selftok_render(self.h, tokens.data_ptr(), tokens.shape[0], out.data_ptr(), _stream_ptr(self.device)))
            else:
                check(self.lib.selftok_render_prefix(self.h, tokens.data_ptr(), n.data_ptr(), tokens.shape[0], out.data_ptr(),
                                                     _stream_ptr(self.device)))
        return out

    # ------------------------------------------------------------------ hot path (host buffers; copies inside the call)
    def encode_host(self, x0: torch.Tensor, tokens_out: torch.Tensor) -> torch.Tensor:
        if x0.is_cuda or tokens_out.is_cuda or x0.dtype != torch.float32 or tokens_out.dtype != torch.int64 \
                or not x0.is_contiguous() or not tokens_out.is_contiguous():
            raise SelftokError("encode_host: contiguous host tensors (fp32 latents, int64 tokens) expected")
        self._check_latent(x0, "encode_host")
        self._check_tokens(tokens_out, "encode_host", x0.shape[0], is_output=True)
        with torch.cuda.device(self.device):
            check(self.lib.selftok_encode_host(self.h, x0.data_ptr(), x0.shape[0], tokens_out.data_ptr(), _stream_ptr(self.device)))
        return tokens_out

    def decode_host(self, tokens: torch.Tensor, noise: torch.Tensor, out: torch.Tensor, steps: Optional[int] = None) -> torch.Tensor:
        if tokens.is_cuda or noise.is_cuda or out.is_cuda or tokens.dtype != torch.int64 or noise.dtype != torch.float32 \
                or out.dtype != torch.float32 or not (tokens.is_contiguous() and noise.is_contiguous() and out.is_contiguous()):
            raise SelftokError("decode_host: contiguous host tensors (int64 tokens, fp32 noise / output) expected")
        self._check_latent(noise, "decode_host (noise)")
        self._check_latent(out, "decode_host (output)")
        self._check_tokens(tokens, "decode_host", noise.shape[0])
        with torch.cuda.device(self.device):
            check(self.lib.selftok_decode_host(self.h, tokens.data_ptr(), noise.data_ptr(), tokens.shape[0],
                                               steps or self.steps, out.data_ptr(), _stream_ptr(self.device)))
        return out

    def render_host(self, tokens: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
        if tokens.is_cuda or out.is_cuda or tokens.dtype != torch.int64 or out.dtype != torch.float32 \
                or not (tokens.is_contiguous() and out.is_contiguous()):
            raise SelftokError("render_host: contiguous host tensors (int64 tokens, fp32 output) expected")
        self._check_latent(out, "render_host (output)")
        self._check_tokens(tokens, "render_host", out.shape[0])
        with torch.cuda.device(self.device):
            check(self.lib.selftok_render_host(self.h, tokens.data_ptr(), tokens.shape[0], out.data_ptr(), _stream_ptr(self.device)))
        return out

    # ------------------------------------------------------------------ misc
    def workspace_bytes(self, B: int, op: str) -> int:
        n = int(self.lib.selftok_workspace_bytes(self.h, B, {"encode": 0, "decode": 1}[op]))
        if n < 0:
            raise SelftokError("selftok_workspace_bytes failed")
        return n

    def use_torch_workspace(self, B: int) -> None:
        """Allocate the activation workspaces for batches up to B from PyTorch's caching allocator and hand them to the library
        (selftok_set_workspace): after this the hot path performs no cudaMalloc of its own."""
        self._ws = {}
        with torch.cuda.device(self.device):
            for op, code in (("encode", 0), ("decode", 1)):
                buf = torch.empty(self.workspace_bytes(B, op) + 256, dtype=torch.uint8, device=self.device)
                off = (-buf.data_ptr()) % 256
                self._ws[op] = buf
                check(self.lib.selftok_set_workspace(self.h, code, buf.data_ptr() + off, buf.numel() - 256))

    def set_use_graph(self, enable: bool) -> None:
        check(self.lib.selftok_set_use_graph(self.h, int(enable)))

    PROFILE_CLASSES = ("gemm_tcgen05", "attention", "ln_modulate", "linear_f32", "vq", "other", "_6", "_7")

    def set_profile(self, enable: bool) -> None:
        check(self.lib.selftok_set_profile(self.h, int(enable)))

    def get_profile(self):
        """-> {class: (milliseconds, launches)} since the last call (synchronises the device)."""
        ms = (C.c_double * 8)()
        cnt = (C.c_int64 * 8)()
        check(self.lib.selftok_get_profile(self.h, ms, cnt))
        return {n: (ms[i], int(cnt[i])) for i, n in enumerate(self.PROFILE_CLASSES) if cnt[i]}

    @property
    def last_launch_count(self) -> int:
        return int(self.lib.selftok_last_launch_count(self.h))

    @property
    def device_bytes(self) -> int:
        return int(self.lib.selftok_device_bytes(self.h))

    def close(self) -> None:
        if getattr(self, "h", None):
            self.lib.selftok_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class VaeDecoder:
    """SD3 VAE on the device (`selftok_vae_t`): the `vae.decode` step of SelftokPipeline.decoding and -- when the state dict also
    holds encoder.* tensors -- the `vae.encode(...).mode()` step of SelftokPipeline.encoding.  `state_dict` uses the in-tree
    SDVAE key names (decoder.* / encoder.*); `from_diffusers_keys` maps a diffusers AutoencoderKL state dict onto them."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], device="cuda:0", ch: int = 128, halves=("decoder.", "encoder.")):
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise SelftokError("no CUDA device: selftok_b200 has no CPU fallback")
        self.device = torch.device(device)
        h = C.c_void_p()
        check(self.lib.selftok_vae_create(ch, self.device.index or 0, C.byref(h)))
        self.h = h
        try:
            for name, t in state_dict.items():
                if not name.startswith(tuple(halves)) or not torch.is_tensor(t):
                    continue
                t = t.detach().to(torch.float32).contiguous()
                if t.is_cuda and t.device != self.device:
                    t = t.to(self.device)
                shape = (C.c_int64 * t.dim())(*t.shape)
                check(self.lib.selftok_vae_load_tensor(self.h, name.encode(), t.data_ptr(), t.dim(), shape, int(t.is_cuda)))
            with torch.cuda.device(self.device):
                check(self.lib.selftok_vae_finalize(self.h, _stream_ptr(self.device)))
        except Exception:
            self.close()
            raise

    def decode(self, z: torch.Tensor, norm_ip: bool = False) -> torch.Tensor:
        """z [B,16,h,w] (VAE latent space) -> [B,3,8h,8w] fp32 on the device."""
        if z.dim() != 4 or z.shape[1] != 16 or z.shape[2] != z.shape[3]:
            raise SelftokError(f"VaeDecoder.decode: expected [B,16,h,h] latents, got {tuple(z.shape)}")
        z = z.to(device=self.device, dtype=torch.float32).contiguous()
        B, _, h, w = z.shape
        out = torch.empty(B, 3, 8 * h, 8 * w, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self.lib.selftok_vae_decode(self.h, z.data_ptr(), B, h, w, out.data_ptr(), int(norm_ip), _stream_ptr(self.device)))
        return out

    def encode(self, images: torch.Tensor, return_logvar: bool = False):
        """images [B,3,H,H] in [-1,1] -> the latent distribution's mode [B,16,H/8,H/8] fp32 (VAE latent space, before
        SD3LatentFormat.process_in); with return_logvar also the log-variance."""
        if images.dim() != 4 or images.shape[1] != 3 or images.shape[2] != images.shape[3]:
            raise SelftokError(f"VaeDecoder.encode: expected [B,3,H,H] images, got {tuple(images.shape)}")
        x = images.to(device=self.device, dtype=torch.float32).contiguous()
        B, _, H, W = x.shape
        mean = torch.empty(B, 16, H // 8, W // 8, dtype=torch.float32, device=self.device)
        logvar = torch.empty_like(mean) if return_logvar else None
        with torch.cuda.device(self.device):
            check(self.lib.selftok_vae_encode(self.h, x.data_ptr(), B, H, W, mean.data_ptr(), logvar.data_ptr() if return_logvar else None,
                                              _stream_ptr(self.device)))
        return (mean, logvar) if return_logvar else mean

    @staticmethod
    def from_diffusers_keys(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """diffusers AutoencoderKL keys -> SDVAE keys (the same weights under the other naming: decoder up_blocks are listed
        lowest resolution first there, attention projections are Linear [C,C] instead of 1x1 convs)."""
        out = {}
        ren = {"conv_norm_out": "norm_out", "mid_block.resnets.0": "mid.block_1", "mid_block.resnets.1": "mid.block_2",
               "mid_block.attentions.0.group_norm": "mid.attn_1.norm", "mid_block.attentions.0.to_q": "mid.attn_1.q",
               "mid_block.attentions.0.to_k": "mid.attn_1.k", "mid_block.attentions.0.to_v": "mid.attn_1.v",
               "mid_block.attentions.0.to_out.0": "mid.attn_1.proj_out"}
        for k, v in sd.items():
            half = "decoder." if k.startswith("decoder.") else "encoder." if k.startswith("encoder.") else None
            if half is None:
                continue
            n = k[len(half):]
            for a, b in ren.items():
                if n.startswith(a + "."):
                    n = b + n[len(a):]
            if n.startswith("down_blocks."):
                parts = n.split(".")
                if parts[2] == "resnets":
                    n = f"down.{parts[1]}.block.{parts[3]}." + ".".join(parts[4:])
                elif parts[2] == "downsamplers":
                    n = f"down.{parts[1]}.downsample." + ".".join(parts[4:])
            if n.startswith("up_blocks."):
                parts = n.split(".")
                lvl = 3 - int(parts[1])
                if parts[2] == "resnets":
                    n = f"up.{lvl}.block.{parts[3]}." + ".".join(parts[4:])
                elif parts[2] == "upsamplers":
                    n = f"up.{lvl}.upsample." + ".".join(parts[4:])
            n = n.replace("conv_shortcut", "nin_shortcut")
            if ".attn_1." in n and n.endswith(".weight") and v.dim() == 2:
                v = v[:, :, None, None]
            out[half + n] = v
        return out

    def close(self) -> None:
        if getattr(self, "h", None):
            self.lib.selftok_vae_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- kernel-level helpers used by tests and micro-benchmarks ---------------------------------------------------
def k_linear_f32(A, W, bias=None, act=0):
    lib = load_library()
    M, K = A.shape
    N = W.shape[0]
    out = torch.empty(M, N, dtype=torch.float32, device=A.device)
    check(lib.selftok_k_linear_f32(A.data_ptr(), W.data_ptr(), _ptr(bias), out.data_ptr(), M, N, K, act, _stream_ptr(A.device)))
    return out


def k_linear_tc(A, W, bias=None, nsplit=3):
    lib = load_library()
    M, K = A.shape
    N = W.shape[0]
    out = torch.empty(M, N, dtype=torch.float32, device=A.device)
    check(lib.selftok_k_linear_tc(A.data_ptr(), W.data_ptr(), _ptr(bias), out.data_ptr(), M, N, K, nsplit, _stream_ptr(A.device)))
    return out


def k_set_gemm_ctas(n: int) -> None:
    check(load_library().selftok_k_set_gemm_ctas(n))


def k_ln_mod_f32(x, shift=None, scale=None, period=1):
    lib = load_library()
    M, D = x.shape
    out = torch.empty_like(x)
    ld = shift.shape[-1] if shift is not None else 0
    check(lib.selftok_k_ln_mod_f32(x.data_ptr(), _ptr(shift), _ptr(scale), ld, period, out.data_ptr(), M, D, _stream_ptr(x.device)))
    return out


def k_attention_f32(q, k1, v1, k2=None, v2=None, heads=1):
    """q [B,Sq,H*hd], k1/v1 [B,S1,H*hd], optional second key/value segment."""
    lib = load_library()
    B, Sq, Dm = q.shape
    S1 = k1.shape[1]
    S2 = 0 if k2 is None else k2.shape[1]
    out = torch.empty_like(q)
    check(lib.selftok_k_attention_f32(q.data_ptr(), Dm, k1.data_ptr(), v1.data_ptr(), Dm, S1, _ptr(k2), _ptr(v2), Dm, S2,
                                      out.data_ptr(), Dm, B, Sq, heads, Dm // heads, _stream_ptr(q.device)))
    return out


def k_attention_tc(qkv, heads, nsplit=3, ctx_rows=0, ctx_keys=0):
    """qkv [B,S,3,H,64] fp32 -> [B,S,H*64]."""
    lib = load_library()
    B, S = qkv.shape[0], qkv.shape[1]
    out = torch.empty(B, S, heads * 64, dtype=torch.float32, device=qkv.device)
    check(lib.selftok_k_attention_tc(qkv.data_ptr(), out.data_ptr(), B, S, heads, nsplit, ctx_rows, ctx_keys, _stream_ptr(qkv.device)))
    return out
