"""TEST INFRASTRUCTURE ONLY -- prefix-decode fixtures (tests/golden/*_prefix*.npz) from the UNMODIFIED reference.

Image b is decoded from its first n_b tokens: the reference's own sampler with `super_mask[b] = arange(K) < n_b`
(RectifiedFlow.p_sample_loop, rectified_flow.py:182,227-228; the guided branch hands the same mask to its conditional
evaluation, :281-288) and the renderer's `mask` argument (MMDiT_Renderer.forward, sd3/mmdit.py:1511,1529).

    python oracle/gen_golden_prefix.py tiny_prefix tiny_renderer_prefix   # seconds
    python oracle/gen_golden_prefix.py mid_prefix                          # ~1 min
    python oracle/gen_golden_prefix.py full_prefix_step full_renderer_prefix   # minutes each (B = 2, full geometry)
"""
from __future__ import annotations

import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import gen_golden as G  # noqa: E402  (puts the repository on sys.path)
import ref_loader  # noqa: E402
from selftoktokenizer_b200 import config as C  # noqa: E402
from selftoktokenizer_b200 import synth  # noqa: E402

FULL_YML = "configs/res256/256-eval.yml"
FULL_R_YML = "configs/renderer/renderer-eval.yml"


def super_mask(n, K):
    return torch.arange(K)[None, :] < torch.tensor(n)[:, None]


def sampler_kwargs(pipe, tokens):
    """model_kwargs of SelftokPipeline.decoding (SelftokPipeline.py:249-262)."""
    B = tokens.shape[0]
    outs_q = G.lookup(pipe, tokens)
    k = pipe.diti.to_indices(torch.tensor([pipe.flow.timestep_map[0]] * B).long())
    enc_mask = pipe.model.encoder.get_encoder_mask(tokens, k)
    ehs = outs_q * enc_mask[..., None].expand_as(outs_q)
    return outs_q, dict(encoder_hidden_states=ehs, mask=enc_mask, context_see_xt=True)


def ref_prefix_decode(pipe, tokens, noise, n, uncond_scale=1.0):
    outs_q, kw = sampler_kwargs(pipe, tokens)
    with torch.no_grad():
        return pipe.flow.p_sample_loop(pipe.model.model, noise.shape, noise.clone(), model_kwargs=kw, start_t=pipe._steps,
                                       cond_vary=pipe.cond_vary, diti=pipe.diti, encoder=pipe.model.encoder, x_0=noise.float(),
                                       ori_hidden_states=outs_q, uncond_scale=uncond_scale,
                                       super_mask=super_mask(n, tokens.shape[1]))


def ref_prefix_velocity(pipe, x, step, outs_q, n):
    """One evaluation exactly as p_sample_loop issues it with a super_mask (rectified_flow.py:198-231,276-279)."""
    flow, diti, enc = pipe.flow, pipe.diti, pipe.model.encoder
    B = x.shape[0]
    t = torch.tensor([flow.scheduled_t[step]] * B)
    k = diti.to_indices(torch.tensor([flow.timestep_map[step]] * B).long())
    mask = enc.get_encoder_mask(x, k) * super_mask(n, outs_q.shape[1])
    with torch.no_grad():
        v, _ = pipe.model.model(x.float(), t, encoder_hidden_states=outs_q, mask=mask, context_see_xt=True)
    return v


def ref_prefix_render(pipe, tokens, n):
    outs_q = G.lookup(pipe, tokens)
    mask = super_mask(n, tokens.shape[1]).float()           # the dtype of the forward's own default (torch.ones)
    with torch.no_grad():
        pred_x0, _ = pipe.model.model(y=None, encoder_hidden_states=outs_q, mask=mask)
    return pred_x0


def gen_tiny_prefix():
    n = [3, 17, 32]
    pipe, _ = G.build(C.TINY, tag="tinyprefix")
    g = np.load(os.path.join(G.GOLD, "tiny.npz"))
    tokens, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    pred = ref_prefix_decode(pipe, tokens, noise, n)
    cfg = ref_prefix_decode(pipe, tokens, noise, n, uncond_scale=2.5)
    outs_q = G.lookup(pipe, tokens)
    vs = {f"v{s}": ref_prefix_velocity(pipe, noise, s, outs_q, n) for s in (0, 30, 49)}
    print("n = 32 row vs tiny.npz pred_x0: max-abs", float((pred[2] - torch.from_numpy(g["pred_x0"][2])).abs().max()))
    G.save("tiny_prefix", n=np.array(n, np.int32), pred_x0=pred, pred_x0_cfg=cfg, cfg_scale=np.float32(2.5), **vs)


def gen_tiny_renderer_prefix():
    n = [1, 9, 32]
    pipe, _ = G.build(G.TINY_R, tag="tinyrprefix")
    g = np.load(os.path.join(G.GOLD, "tiny_renderer.npz"))
    G.save("tiny_renderer_prefix", n=np.array(n, np.int32), pred_x0=ref_prefix_render(pipe, torch.from_numpy(g["tokens"]), n))


def gen_mid_prefix():
    n = [1, 40, 100, 128]
    dims = C.MID
    ref_loader.import_reference()
    sd = synth.synth_state_dict(dims)
    enc_name, dit_name = ref_loader.register_geometry(dims, "midprefix")
    pipe = ref_loader.build_reference_pipeline(ref_loader.dims_to_cfg(dims, enc_name, dit_name), sd)
    g = np.load(os.path.join(G.GOLD, "mid.npz"))
    t0 = time.time()
    pred = ref_prefix_decode(pipe, torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"]), n)
    print(f"mid_prefix: 50-step decode B=4 in {time.time() - t0:.1f}s", flush=True)
    G.save("mid_prefix", n=np.array(n, np.int32), pred_x0=pred)


def gen_full_prefix_step():
    n = [48, 512]
    pipe, _ = G.build(C.FULL, yml=os.path.join(ref_loader.REFERENCE_ROOT, FULL_YML))
    g = np.load(os.path.join(G.GOLD, "full_encode.npz"))
    tokens = torch.from_numpy(g["tokens"])
    outs_q = G.lookup(pipe, tokens)
    x = G.latents("golden.full.xt_prefix", 2, C.FULL)
    out = {}
    for step in (0, 30):
        t0 = time.time()
        out[f"v{step}"] = ref_prefix_velocity(pipe, x, step, outs_q, n)
        print(f"velocity step {step}: {time.time() - t0:.1f}s", flush=True)
    G.save("full_prefix_step", n=np.array(n, np.int32), **out)


def gen_full_renderer_prefix():
    n = [64, 400]
    dims = C.dataclasses.replace(C.FULL, renderer=True)
    pipe, _ = G.build(dims, yml=os.path.join(ref_loader.REFERENCE_ROOT, FULL_R_YML))
    g = np.load(os.path.join(G.GOLD, "full_encode.npz"))
    t0 = time.time()
    pred = ref_prefix_render(pipe, torch.from_numpy(g["tokens"]), n)
    print(f"renderer B=2: {time.time() - t0:.1f}s", flush=True)
    G.save("full_renderer_prefix", n=np.array(n, np.int32), pred_x0=pred)


if __name__ == "__main__":
    targets = {"tiny_prefix": gen_tiny_prefix, "tiny_renderer_prefix": gen_tiny_renderer_prefix, "mid_prefix": gen_mid_prefix,
               "full_prefix_step": gen_full_prefix_step, "full_renderer_prefix": gen_full_renderer_prefix}
    for w in sys.argv[1:] or ["tiny_prefix"]:
        if w not in targets:
            raise SystemExit(f"unknown target {w}")
        targets[w]()
