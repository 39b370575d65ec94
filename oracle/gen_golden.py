"""TEST INFRASTRUCTURE ONLY — generates tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference, imported through oracle/ref_loader.py) on the seeded synthetic checkpoint of
selftoktokenizer_b200/synth.py.  The reference has no tests and no stored vectors of its own (SURVEY 4),
so these dumps are the known-answer material that pins both oracle/selftok_oracle.py and the CUDA path.

    python oracle/gen_golden.py tiny          # seconds
    python oracle/gen_golden.py tiny_renderer # seconds
    python oracle/gen_golden.py full_encode   # ~1 min   (B=2 encode, full geometry)
    python oracle/gen_golden.py full_step     # ~5 min   (single MMDiT velocity evaluations, B=1)
    python oracle/gen_golden.py full_decode   # ~1 h     (B=1, all 50 steps through the reference's own loop)

Inputs are regenerated on the test side from the same integer hash (synth.synth_tensor), except the decode
noise, which the reference draws itself with torch.randn on the CPU global generator
(SelftokPipeline.py:262-264) and which is therefore stored in the fixture.
"""
from __future__ import annotations

import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, REPO)
sys.path.insert(0, HERE)

import ref_loader  # noqa: E402
from selftoktokenizer_b200 import config as C  # noqa: E402
from selftoktokenizer_b200 import synth  # noqa: E402

GOLD = os.path.join(REPO, "tests", "golden")
TINY_R = C.dataclasses.replace(C.TINY, renderer=True, context_see_xt=True)


def latents(name, B, dims):
    """Seeded encoder input (stands for the VAE-encoded, process_in-scaled latent; SelftokPipeline.py:215-218)."""
    return synth.synth_tensor(name, (B, dims.in_channels, dims.latent, dims.latent), "emb", 1.0)


def build(dims, tag=None, yml=None, seed=0):
    ref_loader.import_reference()
    sd = synth.synth_state_dict(dims, seed=seed)
    if yml is not None:
        from mimogpt.infer.infer_utils import parse_args_from_yaml
        cfg = parse_args_from_yaml(yml)
        if dims.renderer:
            cfg.tokenizer.params.decoder_config["repeat"] = True  # mask_token [1,1,D] form used by the released renderer ckpt
    else:
        enc_name, dit_name = ref_loader.register_geometry(dims, tag)
        cfg = ref_loader.dims_to_cfg(dims, enc_name, dit_name)
    t0 = time.time()
    pipe = ref_loader.build_reference_pipeline(cfg, sd)
    print(f"[gen_golden] reference pipeline built in {time.time() - t0:.1f}s", flush=True)
    return pipe, sd


def ref_encode(pipe, x0):
    """SelftokPipeline.encoding after the VAE (SelftokPipeline.py:218-221) + the pre-VQ features."""
    enc = pipe.model.encoder
    feats = {}

    def hook(mod, inp):
        feats["z"] = inp[0].detach().clone()

    h = enc.quantizer.register_forward_pre_hook(hook)
    with torch.no_grad():
        outs_q, tokens = enc(x0.to(torch.float32), d=None)
    h.remove()
    z = feats["z"]
    # top-1 / top-2 cosine margins (for reporting near-ties)
    with torch.no_grad():
        q = enc.quantizer
        zn = torch.nn.functional.normalize(q.project_in(z), p=2, dim=-1)
        sim = zn.reshape(-1, zn.shape[-1]) @ q._codebook.embed[0].t()
        top2 = sim.topk(2, dim=-1).values
        margin = (top2[:, 0] - top2[:, 1]).reshape(tokens.shape)
    return outs_q, tokens, z, margin


def ref_decode(pipe, tokens_np, seed):
    """Reference decoding() (SelftokPipeline.py:227-294) with the sampler's return value and noise recorded."""
    rec = {}
    orig = pipe.flow.p_sample_loop

    def wrapped(model, shape, noise=None, **kw):
        rec["noise"] = noise.detach().clone()
        out = orig(model, shape, noise, **kw)
        rec["pred_x0"] = out.detach().clone()
        return out

    pipe.flow.p_sample_loop = wrapped
    torch.manual_seed(seed)
    try:
        pipe.decoding(tokens_np, device="cpu")
    finally:
        pipe.flow.p_sample_loop = orig
    return rec["noise"], rec["pred_x0"]


def ref_velocity(pipe, x, step, outs_q):
    """One MMDiT velocity evaluation exactly as p_sample_loop/sample_one_step issue it
    (rectified_flow.py:198-215,276-279)."""
    flow, diti, enc = pipe.flow, pipe.diti, pipe.model.encoder
    B = x.shape[0]
    t = torch.tensor([flow.scheduled_t[step]] * B)
    t_mapped = torch.tensor([flow.timestep_map[step]] * B).long()
    k = diti.to_indices(t_mapped)
    mask = enc.get_encoder_mask(x, k)
    with torch.no_grad():
        v, _ = pipe.model.model(x.float(), t, encoder_hidden_states=outs_q, mask=mask, context_see_xt=True)
    return v


def lookup(pipe, tokens):
    enc = pipe.model.encoder
    with torch.no_grad():
        o = enc.quantizer.get_output_from_indices(tokens)
        o = o.reshape(tokens.shape[0], -1, o.shape[-1])
        o = enc.final_layer_norm3(o)
    return o


# ---------------------------------------------------------------------------------------------- pixel boundary (SD3 VAE)
def ref_vae(ch):
    """The reference's in-tree SD3 VAE (`SDVAE`, sd3/sd3_impls.py:447-474) in fp32 on the CPU with the seeded synthetic
    VAE checkpoint -- the stand-in BASELINE.md prescribes for pixel-space parity (no SD3 weights can be fetched)."""
    ref_loader.import_reference()
    from mimogpt.models.selftok.sd3.sd3_impls import VAEDecoder, VAEEncoder

    class _VAE(torch.nn.Module):
        def __init__(self):
            super().__init__()
            with ref_loader.skip_init():
                self.encoder = VAEEncoder(ch=ch)
                self.decoder = VAEDecoder(ch=ch)

    m = _VAE()
    m.load_state_dict(synth.synth_vae_state_dict(ch=ch), strict=True)
    return m.eval()


def ref_pixels(vae, pred_x0):
    """The pixel end of SelftokPipeline.decoding (SelftokPipeline.py:284-294) with the reference's own helpers."""
    from mimogpt.models.selftok.sd3.sd3_impls import SD3LatentFormat
    from mimogpt.infer.SelftokPipeline import norm_ip
    with torch.no_grad():
        rec = vae.decoder(SD3LatentFormat().process_out(pred_x0.float()))
    norm_ip(rec, -1, 1)
    return rec


def gen_vae_tiny():
    """Pins oracle/vae_oracle.py: decoder and encoder of the reference SDVAE at ch = 32 on seeded inputs."""
    vae = ref_vae(32)
    z = synth.synth_tensor("golden.vae.z", (2, 16, 8, 8), "emb", 1.0)
    x = synth.synth_tensor("golden.vae.x", (2, 3, 64, 64), "emb", 0.5)
    with torch.no_grad():
        dec = vae.decoder(z)
        mom = vae.encoder(x)
    save("vae_tiny", dec=dec, moments=mom)


def gen_vae_enc128():
    """The reference's VAEEncoder at the shipped width (ch = 128) on two seeded 128 x 128 images: the direct pin of the device
    VAE encoder (csrc/vae.cu selftok_vae_encode) and of oracle/vae_oracle.encode_moments at full width."""
    vae = ref_vae(128)
    x = synth.synth_tensor("golden.vae.x128", (2, 3, 128, 128), "emb", 0.5)
    with torch.no_grad():
        mom = vae.encoder(x)
    save("vae_enc128", moments=mom)


def gen_pixels_tiny():
    """Pixel fixture of the reduced geometry: the reference's own 50-step result (tests/golden/tiny.npz) through the
    reference SDVAE (full size, ch = 128) exactly as SelftokPipeline.decoding finishes (process_out -> vae.decode -> norm_ip)."""
    g = np.load(os.path.join(GOLD, "tiny.npz"))
    vae = ref_vae(128)
    save("tiny_pixels", pixels=ref_pixels(vae, torch.from_numpy(g["pred_x0"])))


RENDERER_PIXEL_STRIDE = 2


def gen_pixels_full():
    """Full geometry, B = 1: reference latents of tests/golden/full_decode.npz and full_renderer.npz through the
    full-size (ch = 128) reference SDVAE -> [1,3,256,256] pixels in [0,1].  The renderer's image is kept at every second row
    and column (RENDERER_PIXEL_STRIDE): two full fp32 images do not compress below 1 MB."""
    vae = ref_vae(128)
    g = np.load(os.path.join(GOLD, "full_decode.npz"))
    gr = np.load(os.path.join(GOLD, "full_renderer.npz"))
    t0 = time.time()
    px = ref_pixels(vae, torch.from_numpy(g["pred_x0"]))
    pr = ref_pixels(vae, torch.from_numpy(gr["pred_x0"]))
    print(f"SDVAE decode of 2 images: {time.time() - t0:.1f}s; in-range fraction {float(((px > 0) & (px < 1)).float().mean()):.3f}")
    s = RENDERER_PIXEL_STRIDE
    save("full_pixels", pixels=px, renderer_pixels=pr[..., ::s, ::s])


def gen_tiny_module():
    """The reference's own modules built on the TINY geometry: the name and shape of every entry of their state dict (the
    contract synth.state_dict_spec must meet) and the encoder's tokens and quantised outputs for two seeded latents."""
    import json
    dims = C.TINY
    pipe, _ = build(dims, tag="tinymodule")
    shapes = {k: list(v.shape) for k, v in pipe.model.state_dict().items()}
    x0 = synth.synth_tensor("live.x0", (2, dims.in_channels, dims.latent, dims.latent), "emb", 1.0)
    with torch.no_grad():
        outs_q, tokens = pipe.model.encoder(x0, d=None)
    save("tiny_module", state_dict_shapes=np.array(json.dumps(shapes)), tokens=tokens, outs_q=outs_q)


def gen_boundary():
    """The reference's boundary helpers (SelftokPipeline.py:85-97,135-137; sd3/sd3_impls.py:133-144) on seeded inputs:
    NormalizeToTensor of an 8-bit image, norm_ip, and SD3LatentFormat.process_in / process_out."""
    ref_loader.import_reference()
    from mimogpt.infer import SelftokPipeline as SP
    from mimogpt.models.selftok.sd3.sd3_impls import SD3LatentFormat
    img = np.random.RandomState(0).randint(0, 256, size=(24, 40, 3)).astype(np.uint8)
    y = torch.tensor([-3.0, -1.0, 0.0, 0.5, 1.0, 2.0])
    SP.norm_ip(y, -1, 1)
    lat = synth.synth_tensor("golden.boundary.lat", (2, 16, 4, 4), "emb", 1.0)
    save("boundary", normalized=SP.NormalizeToTensor()(img), norm_ip=y, process_in=SD3LatentFormat().process_in(lat),
         process_out=SD3LatentFormat().process_out(lat))


def save(name, **arrs):
    os.makedirs(GOLD, exist_ok=True)
    out = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrs.items()}
    path = os.path.join(GOLD, name + ".npz")
    np.savez_compressed(path, **out)
    print(f"[gen_golden] wrote {path} ({os.path.getsize(path) / 1024:.1f} KiB)", flush=True)


def gen_tiny():
    dims = C.TINY
    pipe, _ = build(dims, tag="tiny")
    B = 3
    x0 = latents("golden.tiny.x0", B, dims)
    outs_q, tokens, z, margin = ref_encode(pipe, x0)
    noise, pred_x0 = ref_decode(pipe, tokens.numpy(), seed=1234)
    v0 = ref_velocity(pipe, noise, 0, outs_q)
    v30 = ref_velocity(pipe, noise, 30, outs_q)
    v49 = ref_velocity(pipe, noise, 49, outs_q)
    save("tiny", tokens=tokens, outs_q=outs_q, z=z, margin=margin, noise=noise, pred_x0=pred_x0,
         v0=v0, v30=v30, v49=v49,
         t=pipe.flow.scheduled_t, t_prev=pipe.flow.scheduled_t_prev, timestep_map=pipe.flow.timestep_map,
         k=pipe.diti.to_indices(pipe.flow.timestep_map.long()))
    print("distinct tokens per image:", [len(set(r.tolist())) for r in tokens], "inter-image diff:",
          float((tokens[0] != tokens[1]).float().mean()))


def gen_mid(stress=False):
    """Mid-size geometry, B = 4 (SURVEY 8d config 3: B >= 4 on a reduced-depth config).  stress=True: the same run on the
    heavy-tailed / outlier-channel checkpoint (synth._stress) -- the fp16-operand stress fixture."""
    dims = C.MID
    ref_loader.import_reference()
    sd = synth.synth_state_dict(dims, stress=stress)
    enc_name, dit_name = ref_loader.register_geometry(dims, "midstress" if stress else "mid")
    cfg = ref_loader.dims_to_cfg(dims, enc_name, dit_name)
    pipe = ref_loader.build_reference_pipeline(cfg, sd)
    B = 4
    x0 = latents("golden.mid.x0", B, dims)
    outs_q, tokens, z, margin = ref_encode(pipe, x0)
    t0 = time.time()
    noise, pred_x0 = ref_decode(pipe, tokens.numpy(), seed=4321)
    print(f"mid{'_stress' if stress else ''}: decode B={B} in {time.time() - t0:.1f}s; |pred_x0|max {float(pred_x0.abs().max()):.2f}; "
          f"min margin {float(margin.min()):.2e}", flush=True)
    v0 = ref_velocity(pipe, noise, 0, outs_q)
    v49 = ref_velocity(pipe, noise, 49, outs_q)
    save("mid_stress" if stress else "mid", tokens=tokens, margin=margin, noise=noise, pred_x0=pred_x0, v0=v0, v49=v49)


def gen_tiny_cfg():
    """The guided sampler of the reference: p_sample_loop(..., uncond_scale = 2.5) on the TINY checkpoint -- the pipeline never
    forwards cfg_scale (SelftokPipeline.py:266-282), so the loop is called here with the pipeline's own arguments + uncond_scale."""
    dims = C.TINY
    pipe, _ = build(dims, tag="tinycfg")
    g = np.load(os.path.join(GOLD, "tiny.npz"))
    tokens = torch.from_numpy(g["tokens"])
    noise = torch.from_numpy(g["noise"])
    B = tokens.shape[0]
    outs_q = lookup(pipe, tokens)
    k = pipe.diti.to_indices(torch.tensor([pipe.flow.timestep_map[0]] * B).long())
    enc_mask = pipe.model.encoder.get_encoder_mask(tokens, k)
    ehs = outs_q * enc_mask[..., None].expand_as(outs_q)
    model_kwargs = dict(encoder_hidden_states=ehs, mask=enc_mask, context_see_xt=True)
    with torch.no_grad():
        pred = pipe.flow.p_sample_loop(pipe.model.model, noise.shape, noise.clone(), model_kwargs=model_kwargs, start_t=pipe._steps,
                                       cond_vary=pipe.cond_vary, diti=pipe.diti, encoder=pipe.model.encoder, x_0=noise.float(),
                                       ori_hidden_states=outs_q, uncond_scale=2.5)
    print("cfg 2.5 vs plain sampler: max-abs difference", float((pred - torch.from_numpy(g["pred_x0"])).abs().max()))
    save("tiny_cfg", pred_x0=pred, cfg_scale=np.float32(2.5))


def gen_tiny_renderer():
    dims = TINY_R
    pipe, _ = build(dims, tag="tinyr")
    B = 3
    tokens = (synth.synth_tensor("golden.tinyr.tokens", (B, dims.K), "emb", 1.0) + 0.5).mul(dims.codebook_size).long().clamp(0, dims.codebook_size - 1)
    outs_q = lookup(pipe, tokens)
    with torch.no_grad():
        pred_x0, _ = pipe.model.model(y=None, encoder_hidden_states=outs_q)   # SelftokPipeline.py:310
    save("tiny_renderer", tokens=tokens, outs_q=outs_q, pred_x0=pred_x0)


def gen_full_encode():
    dims = C.FULL
    pipe, _ = build(dims, yml=os.path.join(ref_loader.REFERENCE_ROOT, "configs/res256/256-eval.yml"))
    B = 2
    x0 = latents("golden.full.x0", B, dims)
    t0 = time.time()
    outs_q, tokens, z, margin = ref_encode(pipe, x0)
    print(f"encode B={B}: {time.time() - t0:.1f}s; inter-image token diff {float((tokens[0] != tokens[1]).float().mean()):.3f}; "
          f"min margin {float(margin.min()):.3e}")
    save("full_encode", tokens=tokens, outs_q=outs_q, margin=margin, z_sample=z[:, :8],
         t=pipe.flow.scheduled_t, t_prev=pipe.flow.scheduled_t_prev, timestep_map=pipe.flow.timestep_map,
         k=pipe.diti.to_indices(pipe.flow.timestep_map.long()))
    return pipe


def gen_full_step(pipe=None):
    dims = C.FULL
    if pipe is None:
        pipe, _ = build(dims, yml=os.path.join(ref_loader.REFERENCE_ROOT, "configs/res256/256-eval.yml"))
    g = np.load(os.path.join(GOLD, "full_encode.npz"))
    tokens = torch.from_numpy(g["tokens"])[:1]
    outs_q = lookup(pipe, tokens)
    x = latents("golden.full.xt", 1, dims)
    out = {}
    for step in (0, 30, 49):
        t0 = time.time()
        out[f"v{step}"] = ref_velocity(pipe, x, step, outs_q)
        print(f"velocity step {step}: {time.time() - t0:.1f}s", flush=True)
    save("full_step", **out)
    return pipe


def gen_full_decode(pipe=None):
    dims = C.FULL
    if pipe is None:
        pipe, _ = build(dims, yml=os.path.join(ref_loader.REFERENCE_ROOT, "configs/res256/256-eval.yml"))
    g = np.load(os.path.join(GOLD, "full_encode.npz"))
    tokens = g["tokens"][:1]
    t0 = time.time()
    noise, pred_x0 = ref_decode(pipe, tokens, seed=1234)
    print(f"full decode B=1 50 steps: {time.time() - t0:.1f}s", flush=True)
    save("full_decode", noise=noise, pred_x0=pred_x0, seconds=np.float64(time.time() - t0),
         threads=np.int64(torch.get_num_threads()))


def gen_full_renderer():
    dims = C.dataclasses.replace(C.FULL, renderer=True)
    pipe, _ = build(dims, yml=os.path.join(ref_loader.REFERENCE_ROOT, "configs/renderer/renderer-eval.yml"))
    g = np.load(os.path.join(GOLD, "full_encode.npz"))
    tokens = torch.from_numpy(g["tokens"])[:1]
    outs_q = lookup(pipe, tokens)
    t0 = time.time()
    with torch.no_grad():
        pred_x0, _ = pipe.model.model(y=None, encoder_hidden_states=outs_q)
    print(f"renderer B=1: {time.time() - t0:.1f}s")
    save("full_renderer", pred_x0=pred_x0)


def gen_full_renderer_1024():
    """BASELINE config 4: one renderer pass with 1024 tokens at the full geometry (README.md:93-94; the reference ships no
    YAML for it -- configs/selftok_renderer_1024tok.yml = the 512-token renderer YAML with k doubled), B = 1."""
    dims = C.dataclasses.replace(C.FULL, K=1024, stages=(1000,), k_per_stage=(1024,), renderer=True)
    ref_loader.import_reference()
    sd = synth.synth_state_dict(dims)
    cfg = ref_loader.dims_to_cfg(dims)
    cfg.tokenizer.params.stages, cfg.tokenizer.params.k_per_stage = "1000", "1024"
    pipe = ref_loader.build_reference_pipeline(cfg, sd)
    tokens = (synth.synth_tensor("golden.r1024.tokens", (1, dims.K), "emb", 1.0) + 0.5).mul(dims.codebook_size).long().clamp(0, dims.codebook_size - 1)
    outs_q = lookup(pipe, tokens)
    t0 = time.time()
    with torch.no_grad():
        pred_x0, _ = pipe.model.model(y=None, encoder_hidden_states=outs_q)
    print(f"renderer K=1024 B=1: {time.time() - t0:.1f}s")
    save("full_renderer_1024", tokens=tokens, pred_x0=pred_x0)


def gen_tiny_datasize():
    """Non-default `datasize` (the reference's CLI argument): the TINY checkpoint (image_size 64) run at datasize 96 --
    latent 12, encoder and decoder positional grids centre-cropped to 6 x 6 (models_ours.py:183-202, sd3/mmdit.py:877-896)."""
    dims = C.TINY
    ref_loader.import_reference()
    sd = synth.synth_state_dict(dims)
    enc_name, dit_name = ref_loader.register_geometry(dims, "tinyds")
    cfg = ref_loader.dims_to_cfg(dims, enc_name, dit_name)
    pipe = ref_loader.build_reference_pipeline(cfg, sd, datasize=96)
    d96 = C.dataclasses.replace(dims, latent=12)
    x0 = latents("golden.tinyds.x0", 2, d96)
    outs_q, tokens, z, margin = ref_encode(pipe, x0)
    noise, pred_x0 = ref_decode(pipe, tokens.numpy(), seed=99)
    assert tuple(noise.shape) == (2, 16, 12, 12)
    save("tiny_ds96", tokens=tokens, margin=margin, noise=noise, pred_x0=pred_x0)


if __name__ == "__main__":
    what = sys.argv[1:] or ["tiny"]
    pipe = None
    for w in what:
        if w == "tiny":
            gen_tiny()
        elif w == "tiny_renderer":
            gen_tiny_renderer()
        elif w == "full_encode":
            pipe = gen_full_encode()
        elif w == "full_step":
            pipe = gen_full_step(pipe)
        elif w == "full_decode":
            gen_full_decode(pipe)
        elif w == "full_renderer":
            gen_full_renderer()
        elif w == "tiny_cfg":
            gen_tiny_cfg()
        elif w == "mid":
            gen_mid(False)
        elif w == "mid_stress":
            gen_mid(True)
        elif w == "full_renderer_1024":
            gen_full_renderer_1024()
        elif w == "tiny_ds96":
            gen_tiny_datasize()
        elif w == "vae_tiny":
            gen_vae_tiny()
        elif w == "vae_enc128":
            gen_vae_enc128()
        elif w == "tiny_pixels":
            gen_pixels_tiny()
        elif w == "full_pixels":
            gen_pixels_full()
        elif w == "tiny_module":
            gen_tiny_module()
        elif w == "boundary":
            gen_boundary()
        else:
            raise SystemExit(f"unknown target {w}")
