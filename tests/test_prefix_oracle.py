"""Decode from a token prefix (image b from its first n_b tokens): pins the oracle, applied image by image with
n_vis = min(k_i + 1, n_b), against the fixtures oracle/gen_golden_prefix.py produced with the reference's own
p_sample_loop(..., super_mask = arange(K) < n) and MMDiT_Renderer.forward(..., mask = ...)."""
import dataclasses

import numpy as np
import pytest
import torch

import selftok_oracle as O
from selftoktokenizer_b200 import config as C, schedule as S, synth

TINY_R = dataclasses.replace(C.TINY, renderer=True)


def ctx_rows(k, n_max):
    """Context rows of each step in a batch whose longest prefix is n_max (the engine's rule: the existing truncation to the
    visible prefix k_i + 1, capped at n_max); image b masks the keys [min(rows, n_b), rows)."""
    return [min(int(ki), n_max - 1) + 1 for ki in k]


def test_prefix_context_rows_table():
    tb = S.make_tables(512, C.FULL.stages, C.FULL.k_per_stage, 50)
    k0 = int(tb.k[0])
    assert ctx_rows(tb.k, 512) == [int(x) + 1 for x in tb.k]
    # every n_max >= k_0 + 1 shares one table (one captured graph)
    assert all(ctx_rows(tb.k, n) == ctx_rows(tb.k, k0 + 1) for n in range(k0 + 1, 513))
    # joint rows per 50-step decode of a uniform batch, sum_i (min(k_i + 1, n) + 256)
    rows = {n: sum(r + 256 for r in ctx_rows(tb.k, n)) for n in (32, 64, 128, 256, 512)}
    assert rows == {32: 14388, 64: 15925, 128: 18838, 256: 24019, 512: 30759}


def test_tiny_prefix_fixture_self_check(gold):
    g, gp = gold("tiny"), gold("tiny_prefix")
    n = gp["n"].tolist()
    assert n == [3, 17, 32]
    assert np.array_equal(gp["pred_x0"][2], g["pred_x0"][2])       # n = K is the plain sampler, bit for bit
    for st in (0, 30, 49):
        assert np.array_equal(gp[f"v{st}"][2], g[f"v{st}"][2])
    assert np.abs(gp["pred_x0"][0] - g["pred_x0"][0]).max() > 1e-2  # a 3-token prefix decodes to something else


def _velocity(sd, d, tb, x, step, outs_q, n):
    return torch.cat([O.dit_velocity(sd, d, x[b:b + 1], tb.t_freq[step], outs_q[b:b + 1], tb.pos_freq,
                                     min(int(tb.k[step]) + 1, n[b]), truncate=True) for b in range(len(n))])


def _decode(sd, d, tok, noise, n, steps=50):
    tb = S.make_tables(d.K, d.stages, d.k_per_stage, steps)
    outs_q = O.lookup(sd, d, tok)
    x = noise.float().clone()
    for i in range(steps):
        x = x - tb.dt[i] * _velocity(sd, d, tb, x, i, outs_q, n)
    return x


def _decode_cfg(sd, d, tok, noise, n, cfg_scale, steps=50):
    """O.decode_cfg with the conditional evaluation of image b seeing min(k_i + 1, n_b) context tokens."""
    tb = S.make_tables(d.K, d.stages, d.k_per_stage, steps)
    outs_q = O.lookup(sd, d, tok)
    x = noise.float().clone()
    D, g = d.dit_hidden, d.latent // d.dit_patch
    w = sd["model.x_embedder.proj.weight"].reshape(D, -1)
    for i in range(steps):
        xe = O._linear_impl(O._patchify(x, d.dit_patch), w, sd["model.x_embedder.proj.bias"])
        xe = xe + O._center_crop_pos(sd["model.pos_embed"], d.dit_pos_max, g, g)
        c = O._t_embed(sd, "model.t_embedder", tb.t_freq[i].reshape(1, -1))
        ctx = O.context_embed(sd, outs_q)
        v_c = torch.cat([O._unpatchify(O.joint_blocks(sd, d, ctx[b:b + 1], xe[b:b + 1], c, tb.pos_freq, min(int(tb.k[i]) + 1, n[b]),
                                                      ctx_sees_x=False, truncate=False), d) for b in range(len(n))])
        v_u = O.dit_velocity_uncond(sd, d, x, tb.t_freq_uncond[i])
        x = x - tb.dt[i] * (v_u + cfg_scale * (v_c - v_u))
    return x


def _render(sd, d, tok, n):
    outs_q = O.lookup(sd, d, tok)
    x = (sd["model.mask_token"].expand(1, d.n_img, -1) + sd["model.positional_embedding"]).contiguous()
    c = O._t_embed(sd, "model.t_embedder", S.renderer_t_freq())
    ctx = O.context_embed(sd, outs_q)
    pos_freq = S.make_tables(d.K, d.stages, d.k_per_stage, 1).pos_freq
    return torch.cat([O._unpatchify(O.joint_blocks(sd, d, ctx[b:b + 1], x, c, pos_freq, n[b], ctx_sees_x=False, truncate=True), d)
                      for b in range(len(n))])


def test_oracle_tiny_prefix_matches_reference_fixture(gold):
    g, gp = gold("tiny"), gold("tiny_prefix")
    d, n = C.TINY, gp["n"].tolist()
    sd = synth.synth_state_dict(d)
    tok, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    tb = S.make_tables(d.K, d.stages, d.k_per_stage, 50)
    outs_q = O.lookup(sd, d, tok)
    for st in (0, 30, 49):
        assert np.abs(_velocity(sd, d, tb, noise, st, outs_q, n).numpy() - gp[f"v{st}"]).max() < 2e-5
    assert np.abs(_decode(sd, d, tok, noise, n).numpy() - gp["pred_x0"]).max() < 2e-5
    x = _decode_cfg(sd, d, tok, noise, n, float(gp["cfg_scale"]))
    assert np.abs(x.numpy() - gp["pred_x0_cfg"]).max() < 5e-5


def test_oracle_tiny_renderer_prefix_matches_reference_fixture(gold):
    g, gp = gold("tiny_renderer"), gold("tiny_renderer_prefix")
    d = TINY_R
    r = _render(synth.synth_state_dict(d), d, torch.from_numpy(g["tokens"]), gp["n"].tolist())
    assert np.abs(r.numpy() - gp["pred_x0"]).max() < 2e-5
    assert np.abs(gp["pred_x0"][2] - g["pred_x0"][2]).max() < 2e-5       # n = K


def test_oracle_mid_prefix_matches_reference_fixture(gold):
    g, gp = gold("mid"), gold("mid_prefix")
    d, n = C.MID, gp["n"].tolist()
    x = _decode(synth.synth_state_dict(d), d, torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"]), n)
    assert np.abs(x.numpy() - gp["pred_x0"]).max() < 2e-5
    assert np.array_equal(gp["pred_x0"][3], g["pred_x0"][3])             # n = K


def test_oracle_full_prefix_step_matches_reference_fixture(gold):
    gp, ge = gold("full_prefix_step"), gold("full_encode")
    d, n = C.FULL, gp["n"].tolist()
    sd = synth.synth_state_dict(d)
    tb = S.make_tables(d.K, d.stages, d.k_per_stage, 50)
    outs_q = O.lookup(sd, d, torch.from_numpy(ge["tokens"]))
    x = synth.synth_tensor("golden.full.xt_prefix", (2, d.in_channels, d.latent, d.latent), "emb", 1.0)
    for st in (0, 30):
        assert np.abs(_velocity(sd, d, tb, x, st, outs_q, n).numpy() - gp[f"v{st}"]).max() < 1e-4


def test_oracle_full_renderer_prefix_matches_reference_fixture(gold):
    gp, ge = gold("full_renderer_prefix"), gold("full_encode")
    d = dataclasses.replace(C.FULL, renderer=True)
    r = _render(synth.synth_state_dict(d), d, torch.from_numpy(ge["tokens"]), gp["n"].tolist())
    assert np.abs(r.numpy() - gp["pred_x0"]).max() < 1e-4
