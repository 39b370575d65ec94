"""Parity of the CUDA path (through the C ABI) against the oracle and the reference-generated golden fixtures.

Tolerances (north_star): token ids bit-exact (a mismatch is tolerated only where the reference's own top-1/top-2
cosine margin is below 1e-4, and is reported); reconstructed latents within 1e-3 max-abs of the reference's
50-step loop for the fp32-faithful modes (fp32 FFMA and bf16x3).  Single-pass bf16 is measured and reported with a
looser bound — it is NOT the parity mode.
"""
import dataclasses
import os

import numpy as np
import pytest
import torch

import selftok_oracle as O
from selftoktokenizer_b200 import config as C, schedule as S, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = {"fp32": 2e-4, "bf16x3": 1e-3, "fp16": 1e-3, "bf16": 0.35}      # max-abs on latents / velocities of O(3) magnitude


@pytest.fixture(scope="module")
def tiny_sd():
    return synth.synth_state_dict(C.TINY)


@pytest.fixture(scope="module", params=["fp32", "bf16x3", "fp16", "bf16"])
def tiny_engine(request, tiny_sd):
    from selftoktokenizer_b200.capi import Engine
    eng = Engine(C.TINY, tiny_sd, device=DEV, precision=request.param)
    yield eng
    eng.close()


def _check_tokens(tok, gold_tok, margin, what):
    """Token ids must be BIT-EXACT on the committed fixtures (north_star).  Every mismatch is printed with the reference's own
    top-1/top-2 cosine margin so that a rounding-level tie can be told from a real error -- but none is tolerated."""
    mism = tok != gold_tok
    if mism.any():
        print(f"[{what}] {int(mism.sum())} / {mism.size} token mismatches; reference margins: {margin[mism] if margin is not None else '?'}")
    assert int(mism.sum()) == 0, f"{what}: {int(mism.sum())} token ids differ from the reference"


def test_tiny_encode_tokens_bit_exact(tiny_engine, gold):
    g = gold("tiny")
    d = C.TINY
    x0 = synth.synth_tensor("golden.tiny.x0", (3, d.in_channels, d.latent, d.latent), "emb", 1.0)
    tok, outs_q, feats = tiny_engine.encode(x0, return_aux=True)
    assert np.abs(feats.cpu().numpy() - g["z"]).max() < 1e-4
    _check_tokens(tok.cpu().numpy(), g["tokens"], g["margin"], "tiny encode")
    same = tok.cpu().numpy() == g["tokens"]
    assert np.abs(outs_q.cpu().numpy() - g["outs_q"])[same].max() < 1e-5
    # standalone VQ entry on the reference's own pre-VQ features
    ids, oq = tiny_engine.vq_argmax(torch.from_numpy(g["z"]))
    _check_tokens(ids.cpu().numpy().reshape(g["tokens"].shape), g["tokens"], g["margin"], "tiny vq")
    assert np.abs(tiny_engine.lookup(torch.from_numpy(g["tokens"])).cpu().numpy() - g["outs_q"]).max() < 1e-5


def test_tiny_velocity_and_decode(tiny_engine, gold):
    g = gold("tiny")
    tol = TOL[tiny_engine.precision]
    tok, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    for st in (0, 30, 49):
        v = tiny_engine.dit_velocity(tok, noise, st).cpu().numpy()
        err = np.abs(v - g[f"v{st}"]).max()
        print(f"[{tiny_engine.precision}] velocity step {st}: max-abs err {err:.3e}")
        assert err < tol
    for use_graph in (False, True):
        tiny_engine.set_use_graph(use_graph)
        x = tiny_engine.decode(tok, noise).cpu().numpy()
        err = np.abs(x - g["pred_x0"]).max()
        print(f"[{tiny_engine.precision}] 50-step decode (graph={use_graph}): max-abs err {err:.3e}, launches {tiny_engine.last_launch_count}")
        assert err < tol
    # host-buffer entry (H2D / D2H inside the call) gives the same result as the device entry
    out = torch.empty_like(noise).pin_memory()
    tiny_engine.decode_host(tok.pin_memory(), noise.pin_memory(), out)
    assert np.array_equal(out.numpy(), x)


def test_tiny_shard_invariance(tiny_engine, gold):
    """Per-image math must not depend on the batch size or slice position (SURVEY 8e): B=3 == 1 + 2, bitwise."""
    g = gold("tiny")
    d = C.TINY
    x0 = synth.synth_tensor("golden.tiny.x0", (3, d.in_channels, d.latent, d.latent), "emb", 1.0)
    t_all = tiny_engine.encode(x0).cpu()
    t_parts = torch.cat([tiny_engine.encode(x0[:1]).cpu(), tiny_engine.encode(x0[1:]).cpu()])
    assert torch.equal(t_all, t_parts)
    tok, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    full = tiny_engine.decode(tok, noise, steps=5).cpu()
    parts = torch.cat([tiny_engine.decode(tok[:1], noise[:1], steps=5).cpu(), tiny_engine.decode(tok[1:], noise[1:], steps=5).cpu()])
    assert torch.equal(full, parts)


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "fp16"])
def test_tiny_renderer(precision, gold):
    from selftoktokenizer_b200.capi import Engine
    g = gold("tiny_renderer")
    d = dataclasses.replace(C.TINY, renderer=True)
    eng = Engine(d, synth.synth_state_dict(d), device=DEV, precision=precision)
    r = eng.render(torch.from_numpy(g["tokens"])).cpu().numpy()
    err = np.abs(r - g["pred_x0"]).max()
    print(f"[{precision}] renderer max-abs err {err:.3e}")
    assert err < TOL[precision]
    eng.close()


def test_pipeline_api_latent_boundary(tiny_sd, gold):
    """The drop-in class: constructor arguments, attributes and the numpy-in / device-tensor-out asymmetry."""
    from selftoktokenizer_b200 import SelftokPipeline
    from selftoktokenizer_b200.capi import SelftokError
    g = gold("tiny")
    d = C.TINY
    pipe = SelftokPipeline(cfg=None, ckpt_path=None, sd3_path=None, datasize=d.latent * 8, device=DEV, state_dict=tiny_sd,
                           dims=d)
    assert pipe.engine.precision == "fp16"                            # "auto": half operands for the 50-step sampler
    assert pipe.K == d.K and pipe._steps == 50 and pipe.cond_vary is True and pipe.cfg_scale == 1
    x0 = synth.synth_tensor("golden.tiny.x0", (3, d.in_channels, d.latent, d.latent), "emb", 1.0)
    tokens = pipe.encode_latents(x0)
    assert tokens.is_cuda and tokens.dtype == torch.int64
    idx = tokens.cpu().numpy()                                        # test.py: np.save / np.load round trip
    _check_tokens(idx, g["tokens"], g["margin"], "pipeline encode")
    torch.manual_seed(1234)                                           # the reference draws the noise on the CPU generator
    x = pipe.decode_latents(g["tokens"])
    assert np.abs(x.cpu().numpy() - g["pred_x0"]).max() < TOL["fp16"]
    with pytest.raises(SelftokError):
        pipe.decoding(idx, DEV)                                        # pixel API needs the SD3 VAE


# A second reduced geometry with deliberately ragged sizes (K = 40 tokens, 6x6 = 36 image tokens, S = 41..76, rows not multiples of
# any tile): no reference fixture, so the checker is the (pinned) oracle run on the CPU in the same test.
RAGGED = dataclasses.replace(C.TINY, K=40, k_per_stage=(14, 10, 8, 5, 3), latent=12, enc_pos_max=24, dit_pos_max=10, enc_depth=1,
                             dit_depth=2, codebook_size=2040)      # 15 full 128-code chunks + a 120-code tail: both argmax paths of vq_kernel


@pytest.mark.parametrize("precision", ["bf16x3", "fp16"])
def test_ragged_geometry_against_oracle(precision):
    from selftoktokenizer_b200.capi import Engine
    d = RAGGED
    d.validate()
    sd = synth.synth_state_dict(d, seed=3)
    x0 = synth.synth_tensor("ragged.x0", (5, d.in_channels, d.latent, d.latent), "emb", 1.0)
    noise = synth.synth_tensor("ragged.noise", (5, d.in_channels, d.latent, d.latent), "emb", 1.0)
    outs_q_ref, tok_ref, z_ref = O.encode(sd, d, x0)
    x_ref = O.decode(sd, d, tok_ref, noise, steps=50)
    eng = Engine(d, sd, device=DEV, precision=precision)
    tok, outs_q, feats = eng.encode(x0, return_aux=True)
    assert (feats.cpu() - z_ref).abs().max() < 1e-4
    # margins of the oracle's own argmax decide whether a mismatch is a tie
    zn = torch.nn.functional.normalize(torch.nn.functional.linear(z_ref, sd["encoder.quantizer.project_in.weight"],
                                                                  sd["encoder.quantizer.project_in.bias"]), dim=-1)
    top2 = (zn.reshape(-1, 16) @ sd["encoder.quantizer._codebook.embed"][0].t()).topk(2, dim=-1).values
    margin = (top2[:, 0] - top2[:, 1]).reshape(tok_ref.shape).numpy()
    _check_tokens(tok.cpu().numpy(), tok_ref.numpy(), margin, "ragged encode")
    x = eng.decode(tok_ref, noise).cpu()
    err = float((x - x_ref).abs().max())
    print(f"[{precision}] ragged geometry 50-step decode: max-abs err vs oracle {err:.3e}")
    assert err < TOL[precision]
    eng.close()


# ------------------------------------------------------------------------------------------------ full geometry
@pytest.fixture(scope="module")
def full_sd():
    return synth.synth_state_dict(C.FULL, device=DEV)


@pytest.fixture(scope="module", params=["bf16x3", "fp16"])
def full_engine(request, full_sd):
    """Both parity modes of the decoder: split-bf16 (3 MMAs / product) and single-pass IEEE-half operands."""
    from selftoktokenizer_b200.capi import Engine
    eng = Engine(C.FULL, full_sd, device=DEV, precision=request.param)
    yield eng
    eng.close()


def test_full_encode_tokens(full_engine, gold):
    g = gold("full_encode")
    d = C.FULL
    x0 = synth.synth_tensor("golden.full.x0", (2, d.in_channels, d.latent, d.latent), "emb", 1.0)
    tok, outs_q, feats = full_engine.encode(x0, return_aux=True)
    assert np.abs(feats.cpu().numpy()[:, :8] - g["z_sample"]).max() < 2e-4
    _check_tokens(tok.cpu().numpy(), g["tokens"], g["margin"], "full encode")


def test_full_velocity(full_engine, gold):
    g = gold("full_step")
    ge = gold("full_encode")
    d = C.FULL
    tok = torch.from_numpy(ge["tokens"][:1])
    x = synth.synth_tensor("golden.full.xt", (1, d.in_channels, d.latent, d.latent), "emb", 1.0)
    for st in (0, 30, 49):
        v = full_engine.dit_velocity(tok, x, st).cpu().numpy()
        err = np.abs(v - g[f"v{st}"]).max()
        print(f"[{full_engine.precision}] full-geometry velocity step {st}: max-abs err {err:.3e} (|v|max {np.abs(g[f'v{st}']).max():.2f})")
        assert err < 1e-3


def test_full_decode_50_steps(full_engine, gold):
    g = gold("full_decode")
    ge = gold("full_encode")
    tok = torch.from_numpy(ge["tokens"][:1])
    x = full_engine.decode(tok, torch.from_numpy(g["noise"])).cpu().numpy()
    err = np.abs(x - g["pred_x0"]).max()
    mse = float(((x - g["pred_x0"]) ** 2).mean())
    print(f"[{full_engine.precision}] full-geometry 50-step decode: max-abs err {err:.3e}, mse {mse:.3e}")
    assert err < 1e-3


def test_full_renderer_one_pass(gold):
    """decoding_with_renderer at the shipped geometry (BASELINE config[3], 512-token renderer YAML): one MMDiT_Renderer pass."""
    from selftoktokenizer_b200.capi import Engine
    g = gold("full_renderer")
    ge = gold("full_encode")
    d = dataclasses.replace(C.FULL, renderer=True)
    # "auto" resolves to bf16x3 for the renderer: its output is ONE network evaluation, so single-pass half operands land at
    # the edge of the 1e-3 bar (measured 1.05e-3) instead of averaging out as in the 50-step sampler; fp16 is reported only.
    for precision, tol in (("auto", 1e-3), ("fp16", 2.5e-3)):
        eng = Engine(d, synth.synth_state_dict(d, device=DEV), device=DEV, precision=precision)
        precision = eng.precision
        r = eng.render(torch.from_numpy(ge["tokens"][:1])).cpu().numpy()
        err = np.abs(r - g["pred_x0"]).max()
        ref = g["pred_x0"]
        psnr_drop = 10 * np.log10(((ref.max() - ref.min()) ** 2) / max(((r - ref) ** 2).mean(), 1e-30))
        print(f"[{precision}] full-geometry renderer: max-abs err {err:.3e}; PSNR of ours vs reference {psnr_drop:.1f} dB")
        assert err < tol
        out = torch.empty(1, d.in_channels, d.latent, d.latent).pin_memory()
        eng.render_host(torch.from_numpy(ge["tokens"][:1]).pin_memory(), out)
        assert np.array_equal(out.numpy(), r)
        eng.close()


def test_full_batch_roundtrip_properties(full_engine):
    """BASELINE-size property checks the CPU oracle cannot reach (B=64 encode): determinism, shard invariance,
    ids in range, and encode -> lookup -> VQ idempotence (re-quantising a code returns the same id)."""
    d = C.FULL
    x0 = synth.synth_tensor("prop.full.x0", (64, d.in_channels, d.latent, d.latent), "emb", 1.0, device=DEV)
    tok, outs_q, feats = full_engine.encode(x0, return_aux=True)
    tok2 = full_engine.encode(x0)
    assert torch.equal(tok, tok2)
    assert int(tok.min()) >= 0 and int(tok.max()) < d.codebook_size
    assert torch.equal(tok[:16], full_engine.encode(x0[:16]))
    assert torch.equal(tok[48:], full_engine.encode(x0[48:]))
    ids, _ = full_engine.vq_argmax(feats)
    assert torch.equal(ids.reshape(tok.shape), tok)
    assert (tok[0] != tok[1]).float().mean() > 0.3
    # host-buffer entry == device entry
    tok_h = torch.empty(64, d.K, dtype=torch.int64).pin_memory()
    full_engine.encode_host(x0.cpu().pin_memory(), tok_h)
    assert torch.equal(tok_h, tok.cpu())


# ------------------------------------------------------------------------------------------------ round-2 hardening
def _top2_margin(sd, z):
    zn = torch.nn.functional.normalize(torch.nn.functional.linear(z, sd["encoder.quantizer.project_in.weight"],
                                                                  sd["encoder.quantizer.project_in.bias"]), dim=-1)
    cb = sd["encoder.quantizer._codebook.embed"][0]
    out = []
    flat = zn.reshape(-1, zn.shape[-1])
    for lo in range(0, flat.shape[0], 4096):
        t2 = (flat[lo:lo + 4096] @ cb.t()).topk(2, dim=-1).values
        out.append(t2[:, 0] - t2[:, 1])
    return torch.cat(out).reshape(z.shape[:-1]).numpy()


def test_full_batch64_tokens_bit_exact_against_oracle(full_engine):
    """BASELINE batch: all 64 x 512 = 32768 token ids of the bench latents against the (pinned) oracle run on the host
    cores in this test -- zero mismatches allowed; the reference's margins go down to 1e-5 at this sample size."""
    d = C.FULL
    x0 = synth.synth_tensor("bench.x0.0", (64, d.in_channels, d.latent, d.latent), "emb", 1.0)
    spec = synth.state_dict_spec(d)
    sd = {n: synth.synth_tensor(n, sh, k, std) for n, (sh, k, std) in spec.items() if n.startswith("encoder.")}
    tb = S.make_tables(d.K, d.stages, d.k_per_stage)
    toks, zs = [], []
    with torch.no_grad():
        for lo in range(0, 64, 8):
            _, t, z = O.encode(sd, d, x0[lo:lo + 8], tb)
            toks.append(t)
            zs.append(z)
    tok_ref, z_ref = torch.cat(toks), torch.cat(zs)
    margin = _top2_margin(sd, z_ref)
    print(f"oracle B=64 encode done; smallest reference top-1/top-2 margin {margin.min():.3e}, {int((margin < 1e-4).sum())} below 1e-4")
    tok = full_engine.encode(x0).cpu()
    _check_tokens(tok.numpy(), tok_ref.numpy(), margin, "full B=64 encode")
    assert (tok_ref[0] != tok_ref[1]).float().mean() > 0.3


class _OracleVAE:
    """Stand-in for diffusers.AutoencoderKL with the reference's call shapes (SelftokPipeline.py:215,288,316): the SD3 VAE
    arithmetic comes from oracle/vae_oracle.py (the checker; fp32 on the host) -- it is the VAE here, not the path.
    `decoder` (a capi.VaeDecoder) switches decode() to the device VAE of this repo; encode() stays on the oracle arithmetic."""

    class _Dist:
        def __init__(self, m):
            self._m = m

        def mode(self):
            return self._m

    def __init__(self, sd, ch_mult=(1, 2, 4, 4), decoder=None):
        self.sd, self.ch_mult, self.decoder = sd, ch_mult, decoder

    def encode(self, x, return_dict=False):
        import vae_oracle as V
        return (self._Dist(V.encode_mean(self.sd, x.float().cpu()).to(x.device)),)

    def decode(self, z, return_dict=False):
        import vae_oracle as V
        if self.decoder is not None:
            return (self.decoder.decode(z),)
        return (V.decode(self.sd, z.float().cpu()).to(z.device),)


def _psnr(a, b):
    return 10.0 * np.log10(1.0 / max(float(((a - b) ** 2).mean()), 1e-30))


def _pixel_gate(px, px_ref, gt, what):
    """north_star bar at the PIXEL boundary: max-abs <= 1e-3 on [0,1] images and PSNR (against the same target image) within
    0.01 dB of the reference's reconstruction."""
    err = float(np.abs(px - px_ref).max())
    d_psnr = abs(_psnr(px, gt) - _psnr(px_ref, gt))
    print(f"[{what}] pixels: max-abs err {err:.3e}; PSNR vs target ours {_psnr(px, gt):.4f} dB / reference {_psnr(px_ref, gt):.4f} dB "
          f"(delta {d_psnr:.5f} dB); PSNR ours-vs-reference {_psnr(px, px_ref):.1f} dB")
    assert err <= 1e-3, what
    assert d_psnr <= 0.01, what


def test_tiny_pixel_gate_through_pipeline_api(tiny_sd, gold):
    """encoding() / decoding() of the drop-in class with a VAE object of the reference's shape (the in-tree SDVAE arithmetic,
    full size): pixels of the 50-step decode against the reference's own pixels (tests/golden/tiny_pixels.npz) -- once with the
    VAE arithmetic on the host (oracle) and once with this repo's DEVICE VAE decoder (f1)."""
    import vae_oracle as V
    from selftoktokenizer_b200 import SelftokPipeline
    from selftoktokenizer_b200.capi import VaeDecoder
    g, gp = gold("tiny"), gold("tiny_pixels")
    d = C.TINY
    vsd = synth.synth_vae_state_dict(ch=128)
    dev_vae = VaeDecoder(vsd, device=DEV)
    for precision, vae in (("fp16", _OracleVAE(vsd)), ("bf16x3", _OracleVAE(vsd)), ("fp16", _OracleVAE(vsd, decoder=dev_vae))):
        pipe = SelftokPipeline(cfg=None, ckpt_path=None, sd3_path=None, datasize=d.latent * 8, dtype=torch.float32, device=DEV,
                               state_dict=tiny_sd, dims=d, vae=vae, precision=precision)
        torch.manual_seed(1234)                                       # the reference's noise draw (CPU global generator)
        rec = pipe.decoding(g["tokens"], DEV)
        assert rec.dtype == torch.float32 and tuple(rec.shape) == (3, 3, 64, 64)
        x0 = synth.synth_tensor("golden.tiny.x0", (3, d.in_channels, d.latent, d.latent), "emb", 1.0)
        gt = V.images_from_latents(vsd, x0).numpy()
        _pixel_gate(rec.cpu().numpy(), gp["pixels"], gt, f"tiny decoding() {precision}" + (" + device VAE" if vae.decoder else ""))
        # encoding(): images -> VAE -> process_in -> tokens; against the oracle run on the same VAE latents
        img = synth.synth_tensor("tiny.images", (2, 3, 64, 64), "emb", 0.5)
        tok = pipe.encoding(img, DEV)
        lat = V.latents_from_images(vsd, img)
        _, tok_ref, z_ref = O.encode(tiny_sd, d, lat)
        _check_tokens(tok.cpu().numpy(), tok_ref.numpy(), _top2_margin(tiny_sd, z_ref), f"tiny encoding() {precision}")
        pipe.engine.close()
    dev_vae.close()


def test_full_pixel_gate(full_engine, gold):
    """The pixel-boundary parity gate at the full geometry (B = 1): our 50-step latents through the SD3 VAE arithmetic
    (oracle, ch = 128, seeded weights) against the reference's latents through the reference's own SDVAE
    (tests/golden/full_pixels.npz)."""
    import vae_oracle as V
    g, ge, gp = gold("full_decode"), gold("full_encode"), gold("full_pixels")
    d = C.FULL
    vsd = synth.synth_vae_state_dict(ch=128, encoder=False)
    tok = torch.from_numpy(ge["tokens"][:1])
    x = full_engine.decode(tok, torch.from_numpy(g["noise"])).cpu()
    with torch.no_grad():
        px = V.images_from_latents(vsd, x).numpy()
        x0 = synth.synth_tensor("golden.full.x0", (2, d.in_channels, d.latent, d.latent), "emb", 1.0)[:1]
        gt = V.images_from_latents(vsd, x0).numpy()
    _pixel_gate(px, gp["pixels"], gt, f"full decode {full_engine.precision}")


def test_full_renderer_pixel_gate(gold):
    """The pixel gate of the renderer pass; the fixture keeps the reference's pixels at every second row and column
    (oracle/gen_golden.py RENDERER_PIXEL_STRIDE), and ours and the target are compared at the same positions."""
    import vae_oracle as V
    from selftoktokenizer_b200.capi import Engine
    gr, ge, gp = gold("full_renderer"), gold("full_encode"), gold("full_pixels")
    d = dataclasses.replace(C.FULL, renderer=True)
    vsd = synth.synth_vae_state_dict(ch=128, encoder=False)
    eng = Engine(d, synth.synth_state_dict(d, device=DEV), device=DEV, precision="auto")
    assert eng.precision == "bf16x3"
    r = eng.render(torch.from_numpy(ge["tokens"][:1])).cpu()
    eng.close()
    with torch.no_grad():
        px = V.images_from_latents(vsd, r).numpy()
        x0 = synth.synth_tensor("golden.full.x0", (2, d.in_channels, d.latent, d.latent), "emb", 1.0)[:1]
        gt = V.images_from_latents(vsd, x0).numpy()
    s = 2
    assert gp["renderer_pixels"].shape == px[..., ::s, ::s].shape
    _pixel_gate(px[..., ::s, ::s], gp["renderer_pixels"], gt[..., ::s, ::s], "full renderer bf16x3")


@pytest.mark.parametrize("fixture,stress", [("mid", False), ("mid_stress", True)])
def test_mid_batch4_decode_and_fp16_stress(fixture, stress, gold):
    """B = 4 on the mid-size geometry (multi-tile attention / GEMMs), against the reference's own run.  `mid_stress` is the
    same run on the heavy-tailed checkpoint with x30..x100 outlier channels in every qkv / fc1 matrix: the fp16-operand
    stress test.  bf16x3 must stay fp32-faithful; fp16 is measured, and must hold the 1e-3 bar here (if a checkpoint breaks
    it, `precision='auto'` detects that and falls back: test_auto_precision_probe)."""
    from selftoktokenizer_b200.capi import Engine
    g = gold(fixture)
    d = C.MID
    sd = synth.synth_state_dict(d, stress=stress)
    x0 = synth.synth_tensor("golden.mid.x0", (4, d.in_channels, d.latent, d.latent), "emb", 1.0)
    tok_ref, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    for precision, tol_v, tol_x in (("bf16x3", 2e-4, 1e-4), ("fp16", 4e-3, 1e-3)):
        eng = Engine(d, sd, device=DEV, precision=precision)
        tok = eng.encode(x0).cpu()
        _check_tokens(tok.numpy(), g["tokens"], g["margin"], f"{fixture} encode")
        ev = max(float(np.abs(eng.dit_velocity(tok_ref, noise, st).cpu().numpy() - g[f"v{st}"]).max()) for st in (0, 49))
        x = eng.decode(tok_ref, noise).cpu().numpy()
        ex = float(np.abs(x - g["pred_x0"]).max())
        print(f"[{fixture} {precision}] B=4: velocity max-abs err {ev:.3e}, 50-step latents {ex:.3e} (finite: {np.isfinite(x).all()})")
        assert np.isfinite(x).all()
        assert ev < tol_v and ex < tol_x
        eng.close()


def test_auto_precision_probe(gold):
    """precision='auto' keeps single-pass fp16 only if a probe on THIS checkpoint agrees with bf16x3; a checkpoint whose
    outlier channels push half-precision operands past the bar gets the fp32-faithful mode."""
    from selftoktokenizer_b200.capi import Engine
    d = C.MID
    eng = Engine(d, synth.synth_state_dict(d), device=DEV, precision="auto")
    print("auto probe (benign checkpoint):", eng.auto_probe)
    assert eng.precision == "fp16" and eng.auto_probe["chosen"] == "fp16" and eng.auto_probe["dev"] <= eng.auto_probe["tol"]
    eng.close()
    sd = synth.synth_state_dict(d, stress=True)
    for name in list(sd):                                  # brutal variant: the outlier rows another x40
        if name.startswith("model.joint_blocks.") and (name.endswith("mlp.fc1.weight") or name.endswith("attn.qkv.weight")):
            w = sd[name]
            rn = w.norm(dim=1)
            w[rn > 10 * rn.median()] *= 40.0
    eng = Engine(d, sd, device=DEV, precision="auto")
    print("auto probe (brutal outliers):", eng.auto_probe)
    assert eng.auto_probe["chosen"] == eng.precision
    assert eng.precision == "bf16x3" and eng.auto_probe["dev"] > eng.auto_probe["tol"]
    g = gold("mid")
    x = eng.decode(torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"]))
    assert torch.isfinite(x).all()
    eng.close()


def test_shape_and_id_checks(tiny_engine):
    """Wrong-resolution latents, short token rows and out-of-range ids fail loudly (ADVICE r1; the reference's
    `codebook[idx]` raises)."""
    from selftoktokenizer_b200.capi import SelftokError
    d = C.TINY
    tok = torch.zeros(2, d.K, dtype=torch.int64)
    noise = torch.zeros(2, d.in_channels, d.latent, d.latent)
    with pytest.raises(SelftokError):
        tiny_engine.encode(torch.zeros(2, d.in_channels, d.latent * 2, d.latent * 2))
    with pytest.raises(SelftokError):
        tiny_engine.decode(tok, torch.zeros(2, d.in_channels, d.latent + 2, d.latent + 2))
    with pytest.raises(SelftokError):
        tiny_engine.decode(tok[:, : d.K - 1], noise)
    with pytest.raises(SelftokError):
        tiny_engine.decode(tok[:1], noise)
    bad = tok.clone()
    bad[1, 3] = d.codebook_size
    with pytest.raises(SelftokError):
        tiny_engine.lookup(bad)                                        # host ids: checked before the launch
    out = tiny_engine.lookup(bad.to(DEV))                              # device ids: NaN row + counter
    assert torch.isnan(out[1, 3]).all() and torch.isfinite(out[0]).all()
    assert tiny_engine.id_errors() == 1 and tiny_engine.id_errors() == 0
    if tiny_engine.precision == "fp16":
        res = torch.empty_like(noise).pin_memory()
        with pytest.raises(SelftokError):
            tiny_engine.decode_host(bad.pin_memory(), noise.pin_memory(), res)
        # the C entry itself (no Python-side check): status SELFTOK_ERR_BAD_ARG after the copy-back
        st = tiny_engine.lib.selftok_decode_host(tiny_engine.h, bad.data_ptr(), noise.data_ptr(), 2, 2, res.data_ptr(), None)
        assert st == -1 and b"token id" in tiny_engine.lib.selftok_last_error()


def test_other_datasize_uses_cropped_positional_grids(tiny_sd, gold):
    """f4: `datasize` != the checkpoint's image_size (a CLI argument of the reference's test.py).  The TINY checkpoint
    (image_size 64) at datasize 96: latent 12, both positional grids centre-cropped to 6 x 6; against the reference's own run."""
    from selftoktokenizer_b200 import SelftokPipeline
    g = gold("tiny_ds96")
    d = dataclasses.replace(C.TINY, latent=12)
    for precision in ("bf16x3", "fp16"):
        pipe = SelftokPipeline(cfg=None, ckpt_path=None, sd3_path=None, datasize=96, device=DEV, state_dict=tiny_sd, dims=d,
                               precision=precision)
        x0 = synth.synth_tensor("golden.tinyds.x0", (2, d.in_channels, 12, 12), "emb", 1.0)
        _check_tokens(pipe.encode_latents(x0).cpu().numpy(), g["tokens"], g["margin"], "datasize 96 encode")
        x = pipe.decode_latents(g["tokens"], noise=torch.from_numpy(g["noise"])).cpu().numpy()
        err = float(np.abs(x - g["pred_x0"]).max())
        print(f"[{precision}] datasize 96 (latent 12) 50-step decode: max-abs err {err:.3e}")
        assert err < TOL[precision]
        pipe.engine.close()


def test_full_renderer_1024_tokens(gold):
    """BASELINE config 4 / f4: ONE renderer pass with 1024 tokens at the full geometry (configs/selftok_renderer_1024tok.yml),
    B = 1, against the reference's own MMDiT_Renderer on the same seeded checkpoint."""
    import os
    from selftoktokenizer_b200.capi import Engine
    g = gold("full_renderer_1024")
    cfg = C.parse_args_from_yaml(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "configs/selftok_renderer_1024tok.yml"))
    d = C.SelftokDims.from_cfg(cfg)
    assert d.K == 1024 and d.renderer and d.k_per_stage == (1024,)
    eng = Engine(d, synth.synth_state_dict(d, device=DEV), device=DEV, precision="auto")
    r = eng.render(torch.from_numpy(g["tokens"])).cpu().numpy()
    err = float(np.abs(r - g["pred_x0"]).max())
    print(f"[{eng.precision}] renderer, 1024 tokens, full geometry: max-abs err {err:.3e} (|x|max {np.abs(g['pred_x0']).max():.2f})")
    assert err < 1e-3
    # the 1024-query encoder on the same engine: deterministic, ids in range, image dependent
    x0 = synth.synth_tensor("golden.full.x0", (2, d.in_channels, d.latent, d.latent), "emb", 1.0)
    tok = eng.encode(x0)
    assert tuple(tok.shape) == (2, 1024) and int(tok.min()) >= 0 and int(tok.max()) < d.codebook_size
    assert torch.equal(tok, eng.encode(x0)) and (tok[0] != tok[1]).float().mean() > 0.3
    eng.close()


def test_prepack_cache_and_model_shell(tiny_sd, gold, tmp_path):
    """f2: checkpoint file -> engine -> prepack cache -> second engine WITHOUT torch.load: identical tokens and latents
    (bitwise); `pipeline.model` keeps the checkpoint interface (state_dict / load_state_dict), EMA decoder selection included."""
    import copy
    from selftoktokenizer_b200 import SelftokPipeline
    from selftoktokenizer_b200.capi import SelftokError
    g = gold("tiny")
    d = C.TINY
    ckpt = dict(tiny_sd)
    ema = {k[len("model."):]: v * 1.01 for k, v in tiny_sd.items() if k.startswith("model.")}     # a different decoder
    ckpt["ema_state_dict"] = ema
    path = str(tmp_path / "tokenizer_ckpt.pth")
    torch.save(ckpt, path)
    cache = str(tmp_path / "cache")
    kw = dict(cfg=None, sd3_path=None, datasize=d.latent * 8, device=DEV, dims=d, precision="fp16")
    p1 = SelftokPipeline(ckpt_path=path, prepack_cache=cache, **kw)
    assert not p1.engine.restored_from_pack and len([f for f in __import__("os").listdir(cache) if f.endswith(".stkpack")]) == 1
    x0 = synth.synth_tensor("golden.tiny.x0", (3, d.in_channels, d.latent, d.latent), "emb", 1.0)
    noise = torch.from_numpy(g["noise"])
    t1, x1 = p1.encode_latents(x0).cpu(), p1.decode_latents(g["tokens"], noise=noise).cpu()
    real_load = torch.load
    try:
        torch.load = lambda *a, **k: (_ for _ in ()).throw(AssertionError("torch.load called although the prepack cache is warm"))
        p2 = SelftokPipeline(ckpt_path=path, prepack_cache=cache, **kw)
    finally:
        torch.load = real_load
    assert p2.engine.restored_from_pack
    assert torch.equal(p2.encode_latents(x0).cpu(), t1) and torch.equal(p2.decode_latents(g["tokens"], noise=noise).cpu(), x1)
    _check_tokens(t1.numpy(), g["tokens"], g["margin"], "prepack encode")
    assert np.abs(x1.numpy() - g["pred_x0"]).max() < TOL["fp16"]
    # the module shell: state_dict round trip and a reload that changes the decoder
    sd = p2.model.state_dict()                                       # read from the checkpoint file on demand
    assert set(k for k in sd if k.startswith("encoder.") or k.startswith("model.")) >= set(synth.state_dict_spec(d))
    sd2 = copy.copy(sd)
    sd2["model.final_layer.linear.bias"] = sd["model.final_layer.linear.bias"] + 0.5
    missing, unexpected = p2.model.load_state_dict(sd2)
    # the reference's own non-parameter buffers (codebook `initted`, `continuous`, ...) are reported, not refused (strict=False)
    assert missing == [] and all(k.startswith("encoder.quantizer.") for k in unexpected), unexpected
    assert not torch.equal(p2.decode_latents(g["tokens"], noise=noise).cpu(), x1)
    with pytest.raises(SelftokError):
        p2.model.load_state_dict({k: v for k, v in sd.items() if k != "model.context_pos_embed"})
    # EMA decoder (SelftokPipeline.py:193-199): another cache key, another result
    p3 = SelftokPipeline(ckpt_path=path, prepack_cache=cache, ema_decoder=True, **kw)
    assert not p3.engine.restored_from_pack
    assert torch.equal(p3.encode_latents(x0).cpu(), t1)
    assert not torch.equal(p3.decode_latents(g["tokens"], noise=noise).cpu(), x1)
    for p in (p1, p2, p3):
        p.engine.close()


def test_guided_sampler_cfg(tiny_engine, gold):
    """f3: classifier-free guidance as RectifiedFlow.sample_one_step implements it (two evaluations per step: conditional with
    context rows blind to the image keys, unconditional = image stream alone at the integer timestep) against the reference's own
    p_sample_loop(..., uncond_scale=2.5)."""
    g, gc = gold("tiny"), gold("tiny_cfg")
    tok, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    x = tiny_engine.decode_cfg(tok, noise, float(gc["cfg_scale"])).cpu().numpy()
    err = float(np.abs(x - gc["pred_x0"]).max())
    print(f"[{tiny_engine.precision}] guided 50-step decode (cfg 2.5): max-abs err {err:.3e}")
    assert err < 2.5 * TOL[tiny_engine.precision]                      # the combination amplifies the per-evaluation error by ~cfg_scale
    # scale 1 collapses to the conditional branch alone -- which is NOT decode(): the guided call site drops context_see_xt
    x1 = tiny_engine.decode_cfg(tok, noise, 1.0, steps=3)
    assert torch.isfinite(x1).all()


@pytest.mark.parametrize("h,B", [(8, 3), (16, 2), (32, 2)])
def test_device_vae_decoder_against_oracle(h, B):
    """f1: the SD3 VAE decoder on the device (implicit-GEMM 3x3 convolutions on the tcgen05 kernel, GroupNorm + SiLU, the
    single-head attention of the middle block) against the pinned restatement of the reference's SDVAE, seeded weights."""
    import vae_oracle as V
    from selftoktokenizer_b200.capi import VaeDecoder
    vsd = synth.synth_vae_state_dict(ch=128, encoder=False)
    z = synth.synth_tensor(f"vae.dev.z{h}", (B, 16, h, h), "emb", 1.0)
    dec = VaeDecoder(vsd, device=DEV)
    out = dec.decode(z).cpu()
    out2 = dec.decode(z).cpu()
    with torch.no_grad():
        ref = V.decode(vsd, z)
    err = float((out - ref).abs().max())
    print(f"device VAE decode latent {h}x{h} B={B}: max-abs err {err:.3e} (|x|max {float(ref.abs().max()):.2f})")
    assert torch.equal(out, out2), "the device VAE must be bit-reproducible"
    assert err < 2e-4
    n = dec.decode(z, norm_ip=True).cpu()
    assert float(n.min()) >= 0.0 and float(n.max()) <= 1.0
    assert float((n - (ref.clamp(-1, 1) + 1) / 2).abs().max()) < 1e-4
    dec.close()


def test_device_vae_encoder_against_reference_fixture(gold):
    """f1, encode side: the SD3 VAE encoder on the device (stride-2 Downsample convolutions as polyphase implicit GEMMs) against
    the REFERENCE's own VAEEncoder output on two seeded 128 x 128 images (tests/golden/vae_enc128.npz), and bit-reproducible."""
    from selftoktokenizer_b200.capi import VaeDecoder
    g = gold("vae_enc128")
    vae = VaeDecoder(synth.synth_vae_state_dict(ch=128), device=DEV)
    x = synth.synth_tensor("golden.vae.x128", (2, 3, 128, 128), "emb", 0.5)
    mean, logvar = vae.encode(x, return_logvar=True)
    mean2 = vae.encode(x)
    mom = torch.cat([mean, logvar], dim=1).cpu().numpy()
    err = float(np.abs(mom - g["moments"]).max())
    print(f"device VAE encode 128x128 B=2: max-abs err vs the reference {err:.3e} (|moments|max {float(np.abs(g['moments']).max()):.2f})")
    assert torch.equal(mean, mean2), "the device VAE must be bit-reproducible"
    assert err < 2e-4
    vae.close()


@pytest.mark.parametrize("H,B", [(256, 2), (512, 1)])
def test_device_vae_encoder_against_oracle(H, B):
    """the same at the shipped image sizes against the pinned restatement (oracle/vae_oracle.py, fp32 on the host)."""
    import vae_oracle as V
    from selftoktokenizer_b200.capi import VaeDecoder
    vsd = synth.synth_vae_state_dict(ch=128)
    vae = VaeDecoder(vsd, device=DEV)
    x = synth.synth_tensor(f"vae.dev.x{H}", (B, 3, H, H), "emb", 0.5)
    mean, logvar = vae.encode(x, return_logvar=True)
    with torch.no_grad():
        ref = V.encode_moments(vsd, x)
    err = float((torch.cat([mean, logvar], dim=1).cpu() - ref).abs().max())
    print(f"device VAE encode {H}x{H} B={B}: max-abs err {err:.3e} (|moments|max {float(ref.abs().max()):.2f})")
    assert err < 2e-4
    # a decoder-only handle refuses to encode, loudly
    dec_only = VaeDecoder(synth.synth_vae_state_dict(ch=128, encoder=False), device=DEV)
    with pytest.raises(Exception):
        dec_only.encode(x)
    dec_only.close()
    vae.close()


def test_pixels_to_tokens_entirely_on_the_device(full_engine):
    """SelftokPipeline.encoding with nothing left on the host: images -> device VAE encoder -> process_in -> Q-Former encoder -> VQ.
    Against the oracle chain on the same images: the VAE latents agree to ~1e-5, so token ids may only differ where the
    reference's own top-1 / top-2 cosine margin is at that rounding level."""
    import vae_oracle as V
    from selftoktokenizer_b200.pipeline import DeviceVAE, SD3LatentFormat
    d = C.FULL
    vsd = synth.synth_vae_state_dict(ch=128)
    spec = synth.state_dict_spec(d)
    sd = {n: synth.synth_tensor(n, sh, k, std) for n, (sh, k, std) in spec.items() if n.startswith("encoder.")}     # host copy for the oracle
    img = synth.synth_tensor("full.images", (2, 3, 256, 256), "emb", 0.5)
    vae = DeviceVAE(vsd, DEV)
    lat = SD3LatentFormat().process_in(vae.encode(img.to(DEV), return_dict=False)[0].mode()).float()
    with torch.no_grad():
        lat_ref = V.latents_from_images(vsd, img)
    lat_err = float((lat.cpu() - lat_ref).abs().max())
    tok = full_engine.encode(lat).cpu().numpy()
    with torch.no_grad():
        _, tok_ref, z_ref = O.encode(sd, d, lat_ref)
    margin = _top2_margin(sd, z_ref)
    mism = tok != tok_ref.numpy()
    print(f"pixels -> tokens on the device: latent max-abs err {lat_err:.3e}; {int(mism.sum())} / {mism.size} ids differ"
          + (f", reference margins there {margin[mism]}" if mism.any() else ""))
    assert lat_err < 2e-4
    assert int(mism.sum()) <= 2 and (not mism.any() or float(margin[mism].max()) < 1e-4)
    vae.decoder.close()


def test_full_pixel_gate_on_device_vae(full_engine, gold):
    """The pixel-boundary parity gate with EVERYTHING after the tokens on the device: 50-step decode (B = 1, full geometry) ->
    process_out -> device VAE decoder -> norm_ip, against the reference's own pixels (tests/golden/full_pixels.npz)."""
    import vae_oracle as V
    from selftoktokenizer_b200.capi import VaeDecoder
    g, ge, gp = gold("full_decode"), gold("full_encode"), gold("full_pixels")
    d = C.FULL
    vsd = synth.synth_vae_state_dict(ch=128, encoder=False)
    dec = VaeDecoder(vsd, device=DEV)
    x = full_engine.decode(torch.from_numpy(ge["tokens"][:1]), torch.from_numpy(g["noise"]))
    px = dec.decode(x / V.SCALE + V.SHIFT, norm_ip=True).cpu().numpy()
    with torch.no_grad():
        x0 = synth.synth_tensor("golden.full.x0", (2, d.in_channels, d.latent, d.latent), "emb", 1.0)[:1]
        gt = V.images_from_latents(vsd, x0).numpy()
    _pixel_gate(px, gp["pixels"], gt, f"full decode {full_engine.precision} + device VAE")
    dec.close()


def test_caller_owned_workspace(tiny_engine, gold):
    """SURVEY 8b: the activation workspace can be the caller's (PyTorch-allocated) block, sized by selftok_workspace_bytes: results
    are bit-identical and the library allocates nothing of its own for it."""
    g = gold("tiny")
    d = C.TINY
    tok, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    x0 = synth.synth_tensor("golden.tiny.x0", (3, d.in_channels, d.latent, d.latent), "emb", 1.0)
    ref_t, ref_x = tiny_engine.encode(x0).cpu(), tiny_engine.decode(tok, noise).cpu()
    own = tiny_engine.device_bytes
    need = tiny_engine.workspace_bytes(3, "decode") + tiny_engine.workspace_bytes(3, "encode")
    assert need > 0
    tiny_engine.use_torch_workspace(3)
    assert tiny_engine.device_bytes < own                             # the library's own blocks were released
    base = tiny_engine.device_bytes
    assert torch.equal(tiny_engine.encode(x0).cpu(), ref_t) and torch.equal(tiny_engine.decode(tok, noise).cpu(), ref_x)
    assert tiny_engine.device_bytes == base                           # nothing allocated behind the caller's back
    # a larger batch than the block was sized for falls back to a library-owned block, transparently
    x5 = synth.synth_tensor("ws.x0", (5, d.in_channels, d.latent, d.latent), "emb", 1.0)
    assert tiny_engine.encode(x5).shape[0] == 5 and tiny_engine.device_bytes > base


def test_roundtrip_driver_script(tmp_path):
    """The reference's test.py on this library (python -m selftoktokenizer_b200.roundtrip): image file -> tokens .npy -> image
    file, shipped 256 / 512-token YAML, seeded synthetic checkpoints (--synthetic), everything incl. both VAE halves on the device."""
    from PIL import Image
    from selftoktokenizer_b200 import roundtrip
    rng = np.random.RandomState(1)
    src = tmp_path / "in.png"
    Image.fromarray(rng.randint(0, 256, (300, 400, 3)).astype(np.uint8)).save(src)
    yml = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "configs", "selftok_256_512tok.yml")
    rc = roundtrip.main(["--yml-path", yml, "--synthetic", "--images", str(src), "--tokens", str(tmp_path / "token.npy"),
                         "--out-prefix", str(tmp_path / "re"), "--device", DEV])
    assert rc == 0
    tok = np.load(tmp_path / "token.npy")
    assert tok.shape == (1, 512) and tok.dtype == np.int64 and tok.min() >= 0 and tok.max() < 32768
    out = np.array(Image.open(tmp_path / "re_0_256.png"))
    assert out.shape == (256, 256, 3) and out.dtype == np.uint8 and out.std() > 0


def test_two_handles_on_two_host_threads(tiny_sd, gold):
    """SURVEY 8b threading: the reference is single-threaded; the C ABI promises more -- one handle per host thread, each on its
    own stream (graph capture is thread-local, the launch counter and last-error are thread-local): two engines driven
    concurrently give bit-identical results to the sequential runs."""
    import threading
    from selftoktokenizer_b200.capi import Engine
    g = gold("tiny")
    d = C.TINY
    tok, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    x0 = synth.synth_tensor("golden.tiny.x0", (3, d.in_channels, d.latent, d.latent), "emb", 1.0)
    engines = [Engine(d, tiny_sd, device=DEV, precision=p) for p in ("fp16", "bf16x3")]
    ref = [(e.encode(x0).cpu(), e.decode(tok, noise).cpu()) for e in engines]
    out, err = [None, None], []

    def work(i):
        try:
            st = torch.cuda.Stream(device=DEV)
            with torch.cuda.stream(st):
                for _ in range(4):
                    t = engines[i].encode(x0)
                    x = engines[i].decode(tok, noise)
                st.synchronize()
                out[i] = (t.cpu(), x.cpu())
        except Exception as exc:  # noqa: BLE001
            err.append(exc)

    th = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not err, err
    for i in range(2):
        assert torch.equal(out[i][0], ref[i][0]) and torch.equal(out[i][1], ref[i][1]), f"engine {i} changed under concurrency"
    for e in engines:
        e.close()


def test_large_batch_is_bitwise_shard_invariant(full_engine):
    """SURVEY 8e: per-image arithmetic must not depend on the batch size or on the position inside the batch.  Batch 80 (not a
    multiple of the bench's 64; 61 440 joint rows, every index path beyond its bench range) against batch 4: ids and 50-step
    latents of the shared images are bit-identical."""
    d = C.FULL
    x0 = synth.synth_tensor("bench.x0.0", (80, d.in_channels, d.latent, d.latent), "emb", 1.0)
    noise = synth.synth_tensor("bench.noise.0", (80, d.in_channels, d.latent, d.latent), "emb", 1.0)
    tok80 = full_engine.encode(x0)
    x80 = full_engine.decode(tok80, noise, steps=6)
    tok4 = full_engine.encode(x0[:4])
    x4 = full_engine.decode(tok4, noise[:4], steps=6)
    tail = full_engine.decode(tok80[76:], noise[76:], steps=6)
    assert torch.equal(tok80[:4].cpu(), tok4.cpu())
    assert torch.equal(x80[:4].cpu(), x4.cpu()), float((x80[:4] - x4).abs().max())
    assert torch.equal(x80[76:].cpu(), tail.cpu())
    assert torch.isfinite(x80).all()
