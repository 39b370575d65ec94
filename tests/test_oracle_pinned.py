"""Pins oracle/selftok_oracle.py (the CPU restatement) against the fixtures that oracle/gen_golden.py produced by
running the UNMODIFIED reference modules."""
import dataclasses
import json
import os

import numpy as np
import pytest
import torch

import selftok_oracle as O
from selftoktokenizer_b200 import config as C, schedule as S, synth

# SURVEY 3.5: per-step visible-token table of the shipped config, recorded from the reference's RectifiedFlow + DiTi_cont
K_TABLE = [511, 510, 508, 507, 505, 504, 502, 500, 499, 497, 496, 491, 486, 481, 476, 472, 467, 462, 457, 452, 448, 440, 433,
           426, 419, 412, 404, 397, 390, 383, 375, 357, 338, 320, 302, 283, 265, 247, 228, 210, 191, 171, 153, 134, 115, 95,
           76, 57, 38, 19]
T_MAPPED = [1000, 980, 960, 940, 920, 900, 880, 860, 840, 820, 800, 780, 760, 740, 720, 700, 680, 660, 640, 620, 600, 580, 560,
            540, 520, 500, 480, 459, 440, 420, 399, 380, 359, 340, 320, 299, 280, 260, 240, 220, 199, 179, 160, 140, 120, 99, 80,
            60, 40, 20]


def test_schedule_tables_full_config(gold):
    tb = S.make_tables(512, C.FULL.stages, C.FULL.k_per_stage, 50)
    assert tb.k.tolist() == K_TABLE
    assert tb.t_mapped.tolist() == T_MAPPED
    assert int((tb.k + 1).sum()) == 17959
    g = gold("full_encode")
    assert np.array_equal(tb.t.numpy(), g["t"])
    assert np.array_equal((tb.t - tb.dt).numpy(), g["t_prev"])          # dt = t - t_prev is exact in fp32 here
    assert np.array_equal(tb.k.numpy(), g["k"])
    assert float(tb.t[1]) == 0.9800000190734863


def test_schedule_tables_tiny(gold):
    g = gold("tiny")
    d = C.TINY
    tb = S.make_tables(d.K, d.stages, d.k_per_stage, 50)
    assert np.array_equal(tb.k.numpy(), g["k"])
    assert np.array_equal(tb.t.numpy(), g["t"])
    assert np.array_equal((tb.t * 1000).numpy(), g["timestep_map"])


@pytest.fixture(scope="module")
def tiny_sd():
    return synth.synth_state_dict(C.TINY)


def test_oracle_encode_matches_reference_fixture(gold, tiny_sd):
    g = gold("tiny")
    d = C.TINY
    x0 = synth.synth_tensor("golden.tiny.x0", (3, d.in_channels, d.latent, d.latent), "emb", 1.0)
    outs_q, tok, z = O.encode(tiny_sd, d, x0)
    assert np.array_equal(tok.numpy(), g["tokens"])
    assert np.abs(z.numpy() - g["z"]).max() < 1e-5
    assert np.abs(outs_q.numpy() - g["outs_q"]).max() < 1e-5
    # the fixture must actually exercise image dependence (SURVEY 8c)
    assert (g["tokens"][0] != g["tokens"][1]).mean() > 0.3


@pytest.mark.parametrize("truncate", [False, True])
def test_oracle_velocity_and_decode_match_reference_fixture(gold, tiny_sd, truncate):
    g = gold("tiny")
    d = C.TINY
    tb = S.make_tables(d.K, d.stages, d.k_per_stage, 50)
    tok = torch.from_numpy(g["tokens"])
    outs_q = O.lookup(tiny_sd, d, tok)
    assert np.abs(outs_q.numpy() - g["outs_q"]).max() < 1e-6
    noise = torch.from_numpy(g["noise"])
    for st in (0, 30, 49):
        v = O.dit_velocity(tiny_sd, d, noise, tb.t_freq[st], outs_q, tb.pos_freq, int(tb.k[st]) + 1, truncate=truncate)
        assert np.abs(v.numpy() - g[f"v{st}"]).max() < 2e-5
    x = O.decode(tiny_sd, d, tok, noise, truncate=truncate)
    assert np.abs(x.numpy() - g["pred_x0"]).max() < 2e-5      # 50 chained steps, fp32


def test_oracle_renderer_matches_reference_fixture(gold):
    g = gold("tiny_renderer")
    d = dataclasses.replace(C.TINY, renderer=True)
    sd = synth.synth_state_dict(d)
    for truncate in (False, True):
        r = O.render(sd, d, torch.from_numpy(g["tokens"]), truncate=truncate)
        assert np.abs(r.numpy() - g["pred_x0"]).max() < 2e-5


def test_oracle_full_encode_matches_reference_fixture(gold):
    """Full geometry, B=2: token ids of the restatement == reference (bit-exact on this host)."""
    g = gold("full_encode")
    d = C.FULL
    spec = synth.state_dict_spec(d)
    sd = {n: synth.synth_tensor(n, sh, k, std) for n, (sh, k, std) in spec.items() if n.startswith("encoder.")}
    x0 = synth.synth_tensor("golden.full.x0", (2, d.in_channels, d.latent, d.latent), "emb", 1.0)
    outs_q, tok, z = O.encode(sd, d, x0)
    mism = tok.numpy() != g["tokens"]
    # any mismatch must be a near-tie (reduction-order noise); on the generating host there are none
    assert mism.mean() <= 0.005 and (g["margin"][mism] < 1e-4).all()
    assert np.abs(z.numpy()[:, :8] - g["z_sample"]).max() < 1e-4
    assert (g["tokens"][0] != g["tokens"][1]).mean() > 0.3


def test_synthetic_weights_are_host_independent():
    """The generator is integer hashing + individually rounded fp32 ops: pin a few values so a silent change
    (which would invalidate every fixture) fails here."""
    t = synth.synth_tensor("encoder.blocks.0.attn.qkv.weight", (192, 64), "w", 0.125)
    assert t.shape == (192, 64)
    ref = [float.fromhex(h) for h in ("0x1.94d7dcp-7", "0x1.4fa070p-6", "-0x1.090e6ap-4", "-0x1.d73e6cp-7")]
    assert t[0, :4].tolist() == ref, t[0, :4]
    cb = synth.synth_tensor("encoder.quantizer._codebook.embed", (1, 1024, 16), "codebook", 1.0)
    assert abs(float(cb[0].norm(dim=-1).mean()) - 1.0) < 1e-6


def test_state_dict_contract_and_encode_match_reference_fixture(gold, tiny_sd):
    """The reference's own modules on the TINY geometry (oracle/gen_golden.py tiny_module): every key of the spec exists in
    their state dict with the same shape, and the restatement's encode gives their tokens and quantised outputs."""
    g = gold("tiny_module")
    ref_shapes = json.loads(str(g["state_dict_shapes"]))
    for name, (shape, _, _) in synth.state_dict_spec(C.TINY).items():
        assert name in ref_shapes and tuple(ref_shapes[name]) == tuple(shape), name
    x0 = synth.synth_tensor("live.x0", (2, 16, 8, 8), "emb", 1.0)
    outs_q, tok, _ = O.encode(tiny_sd, C.TINY, x0)
    assert np.array_equal(tok.numpy(), g["tokens"])
    assert np.abs(outs_q.numpy() - g["outs_q"]).max() < 1e-5


# ------------------------------------------------------------------ plain-C restatement of the index path (oracle/vq_oracle.c)
def _c_oracle():
    import shutil
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    from oracle import c_oracle
    c_oracle.build()
    return c_oracle


def _enc_tensor(d, name):
    sh, kind, std = synth.state_dict_spec(d)[name]
    return synth.synth_tensor(name, sh, kind, std).numpy()


def _check_ids(ids, ref_ids, ref_margin, what):
    bad = np.nonzero(ids != ref_ids)[0]
    for i in bad:                                       # only a rounding-level tie of the reference itself may differ
        assert ref_margin[i] < 1e-6, f"{what}: id mismatch at {i} with reference margin {ref_margin[i]:.3e}"
    if len(bad):
        print(f"{what}: {len(bad)} ids differ, all at reference margins < 1e-6")


def test_c_vq_restatement_matches_reference_fixture_tiny(gold):
    """project_in + l2norm + cosine argmax (first maximum) + gather + final_layer_norm3, in plain C, against what the
    unmodified reference produced from the same pre-VQ features (tests/golden/tiny.npz)."""
    co = _c_oracle()
    g, d = gold("tiny"), C.TINY
    z = g["z"].reshape(-1, g["z"].shape[-1])
    cb = _enc_tensor(d, "encoder.quantizer._codebook.embed")[0]
    ids, _, margin = co.vq(z, _enc_tensor(d, "encoder.quantizer.project_in.weight"),
                           _enc_tensor(d, "encoder.quantizer.project_in.bias"), cb)
    _check_ids(ids, g["tokens"].reshape(-1), g["margin"].reshape(-1), "tiny")
    assert np.abs(margin - g["margin"].reshape(-1)).max() < 1e-6
    out = co.lookup_ln(g["tokens"].reshape(-1), cb, _enc_tensor(d, "encoder.final_layer_norm3.weight"),
                       _enc_tensor(d, "encoder.final_layer_norm3.bias"))
    assert np.abs(out - g["outs_q"].reshape(-1, out.shape[1])).max() < 2e-6


def test_c_vq_restatement_matches_reference_fixture_full(gold):
    """Full geometry (32768 x 16 codebook, 512 -> 16 projection): the fixture keeps the pre-VQ features of the first 8
    tokens of each image."""
    co = _c_oracle()
    g, d = gold("full_encode"), C.FULL
    z = g["z_sample"].reshape(-1, g["z_sample"].shape[-1])
    n = g["z_sample"].shape[1]
    cb = _enc_tensor(d, "encoder.quantizer._codebook.embed")[0]
    ids, _, margin = co.vq(z, _enc_tensor(d, "encoder.quantizer.project_in.weight"),
                           _enc_tensor(d, "encoder.quantizer.project_in.bias"), cb)
    _check_ids(ids, g["tokens"][:, :n].reshape(-1), g["margin"][:, :n].reshape(-1), "full")
    assert np.abs(margin - g["margin"][:, :n].reshape(-1)).max() < 1e-6
    out = co.lookup_ln(g["tokens"].reshape(-1), cb, _enc_tensor(d, "encoder.final_layer_norm3.weight"),
                       _enc_tensor(d, "encoder.final_layer_norm3.bias"))
    assert np.abs(out - g["outs_q"].reshape(-1, out.shape[1])).max() < 2e-6


@pytest.mark.parametrize("name,dims", [("tiny", C.TINY), ("full_encode", C.FULL)])
def test_c_diti_schedule_matches_reference_fixture(gold, name, dims):
    """k_i (visible-token limit per sampler step) as the reference's RectifiedFlow + DiTi_cont produced it."""
    co = _c_oracle()
    g = gold(name)
    k = co.diti_k(g["timestep_map"].astype(np.int64), dims.stages, dims.k_per_stage, dims.K)
    assert (k == g["k"]).all()
    assert (k == S.make_tables(dims.K, dims.stages, dims.k_per_stage).k.numpy()).all()


# ------------------------------------------------------------------ SD3 VAE restatement (oracle/vae_oracle.py)
def test_vae_oracle_matches_reference_fixture(gold):
    """decoder + encoder of the reference's in-tree SDVAE (ch = 32, seeded synthetic weights) as recorded by
    oracle/gen_golden.py vae_tiny."""
    import vae_oracle as V
    g = gold("vae_tiny")
    sd = synth.synth_vae_state_dict(ch=32)
    z = synth.synth_tensor("golden.vae.z", (2, 16, 8, 8), "emb", 1.0)
    x = synth.synth_tensor("golden.vae.x", (2, 3, 64, 64), "emb", 0.5)
    assert np.abs(V.decode(sd, z).numpy() - g["dec"]).max() < 2e-5
    assert np.abs(V.encode_moments(sd, x).numpy() - g["moments"]).max() < 2e-5


def test_vae_oracle_encoder_matches_reference_at_full_width(gold):
    """VAEEncoder at the shipped width (ch = 128) on 128 x 128 images: oracle/gen_golden.py vae_enc128 (the fixture the device
    encoder is checked against in tests/test_parity_gpu.py)."""
    import vae_oracle as V
    g = gold("vae_enc128")
    sd = synth.synth_vae_state_dict(ch=128)
    x = synth.synth_tensor("golden.vae.x128", (2, 3, 128, 128), "emb", 0.5)
    with torch.no_grad():
        mom = V.encode_moments(sd, x).numpy()
    assert mom.shape == (2, 32, 16, 16)
    assert np.abs(mom - g["moments"]).max() < 5e-5


def test_pixel_fixture_is_reference_latents_through_the_vae_oracle(gold):
    """tests/golden/tiny_pixels.npz == images_from_latents(reference pred_x0): the pixel end of SelftokPipeline.decoding
    (process_out -> vae.decode -> norm_ip, SelftokPipeline.py:284-294) restated in vae_oracle."""
    import vae_oracle as V
    g, gp = gold("tiny"), gold("tiny_pixels")
    px = V.images_from_latents(synth.synth_vae_state_dict(ch=128, encoder=False), torch.from_numpy(g["pred_x0"]))
    assert px.min() >= 0 and px.max() <= 1
    assert np.abs(px.numpy() - gp["pixels"]).max() < 2e-5


def test_boundary_helpers_match_reference_fixture(gold):
    """a13: NormalizeToTensor, norm_ip, SD3LatentFormat against what the reference's own definitions
    (SelftokPipeline.py:85-97,135-137; sd3/sd3_impls.py:133-144) returned on the same inputs (oracle/gen_golden.py boundary)."""
    from selftoktokenizer_b200 import pipeline as P
    g = gold("boundary")
    rng = np.random.RandomState(0)
    img = rng.randint(0, 256, size=(24, 40, 3)).astype(np.uint8)
    t = P.NormalizeToTensor()(img)
    assert t.shape == (3, 24, 40) and t.dtype == torch.float32
    assert float(t.min()) >= -1.0 and float(t.max()) <= 1.0
    assert torch.equal(t, torch.from_numpy((img.astype(np.float32) / 127.5 - 1.0).astype(np.float32).transpose(2, 0, 1)))
    grey = P.NormalizeToTensor()(img[:, :, 0])                       # 2-D input gains a channel axis (reshape=True)
    assert grey.shape == (1, 24, 40)
    x = torch.tensor([-3.0, -1.0, 0.0, 0.5, 1.0, 2.0])
    y = x.clone()
    P.norm_ip(y, -1, 1)
    assert torch.equal(y, torch.tensor([0.0, 0.0, 0.5, 0.75, 1.0, 1.0]))
    lat = synth.synth_tensor("golden.boundary.lat", (2, 16, 4, 4), "emb", 1.0)
    f = P.SD3LatentFormat()
    assert torch.allclose(f.process_out(f.process_in(lat)), lat, atol=1e-6)
    assert torch.equal(f.process_in(lat), (lat - 0.0609) * 1.5305)
    assert np.array_equal(t.numpy(), g["normalized"])
    assert np.array_equal(y.numpy(), g["norm_ip"])
    assert np.array_equal(f.process_in(lat).numpy(), g["process_in"]) and np.array_equal(f.process_out(lat).numpy(), g["process_out"])


def test_ema_decoder_state_selection():
    """ema_decoder=True swaps the MMDiT weights for checkpoint['ema_state_dict'] (keys without the 'model.' prefix),
    encoder keys untouched (SelftokPipeline.py:190-199)."""
    from selftoktokenizer_b200.pipeline import _decoder_state
    ck = {"encoder.a": torch.ones(2), "model.w": torch.zeros(3), "model.b": torch.zeros(1), "epoch": 3,
          "ema_state_dict": {"w": torch.full((3,), 7.0), "b": torch.full((1,), 9.0)}}
    plain = _decoder_state(ck, False)
    assert set(plain) == {"encoder.a", "model.w", "model.b"} and float(plain["model.w"][0]) == 0.0
    ema = _decoder_state(ck, True)
    assert set(ema) == {"encoder.a", "model.w", "model.b"}
    assert float(ema["model.w"][0]) == 7.0 and float(ema["model.b"][0]) == 9.0 and float(ema["encoder.a"][0]) == 1.0


def test_config_validation_raises_not_asserts():
    import dataclasses
    with pytest.raises(ValueError):
        dataclasses.replace(C.TINY, k_per_stage=(1, 1, 1, 1, 1)).validate()
    with pytest.raises(ValueError):
        dataclasses.replace(C.TINY, latent=7).validate()
    cfg = C.parse_args_from_yaml(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "configs/selftok_256_512tok.yml"))
    cfg.tokenizer.params.quantizer_config["continuous"] = True
    with pytest.raises(ValueError):
        C.SelftokDims.from_cfg(cfg)
    # datasize overrides the latent side (the reference's CLI argument), the positional grids stay the checkpoint's
    cfg = C.parse_args_from_yaml(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "configs/selftok_256_512tok.yml"))
    d = C.SelftokDims.from_cfg(cfg, datasize=512)
    assert d.latent == 64 and d.enc_pos_max == 64 and d.dit_pos_max == 192 and d.n_img == 1024


def test_mid_fixture_oracle(gold):
    """B = 4 on the mid-size geometry: the restatement reproduces the reference's tokens and 50-step result."""
    g = gold("mid")
    d = C.MID
    sd = synth.synth_state_dict(d)
    x0 = synth.synth_tensor("golden.mid.x0", (4, d.in_channels, d.latent, d.latent), "emb", 1.0)
    _, tok, _ = O.encode(sd, d, x0)
    assert np.array_equal(tok.numpy(), g["tokens"])
    x = O.decode(sd, d, tok, torch.from_numpy(g["noise"]), truncate=True)
    assert np.abs(x.numpy() - g["pred_x0"]).max() < 2e-5


def test_oracle_guided_sampler_matches_reference_fixture(gold, tiny_sd):
    """f3: the restatement of sample_one_step's guided branch + MMDiT.cfg_inference against the reference's own
    p_sample_loop(..., uncond_scale=2.5) (tests/golden/tiny_cfg.npz)."""
    g, gc = gold("tiny"), gold("tiny_cfg")
    x = O.decode_cfg(tiny_sd, C.TINY, torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"]), float(gc["cfg_scale"]))
    assert np.abs(x.numpy() - gc["pred_x0"]).max() < 2e-5
    assert np.abs(gc["pred_x0"] - g["pred_x0"]).max() > 0.05          # the guidance really changes the result
