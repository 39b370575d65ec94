"""Decode from a token prefix on the device: the prefix entry points against the reference-generated prefix fixtures, against
the plain entry points (n_b = K), and their batch, id, graph and argument contracts."""
import dataclasses

import numpy as np
import pytest
import torch

from selftoktokenizer_b200 import config as C, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = {"fp32": 2e-4, "bf16x3": 1e-3, "fp16": 1e-3, "bf16": 0.35}
TINY_R = dataclasses.replace(C.TINY, renderer=True)


def _engine(d, precision, sd=None):
    from selftoktokenizer_b200.capi import Engine
    return Engine(d, sd if sd is not None else synth.synth_state_dict(d), device=DEV, precision=precision)


@pytest.fixture(scope="module", params=["fp32", "bf16x3", "fp16", "bf16"])
def tiny_engine(request):
    eng = _engine(C.TINY, request.param)
    yield eng
    eng.close()


def _err(a, b):
    return float(np.abs(a.cpu().numpy() - b).max())


def test_tiny_all_k_prefix_is_the_plain_path_bitwise(tiny_engine, gold):
    g = gold("tiny")
    tok, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    K = C.TINY.K
    for use_graph in (False, True):
        tiny_engine.set_use_graph(use_graph)
        assert torch.equal(tiny_engine.decode(tok, noise, n_tokens=K), tiny_engine.decode(tok, noise))
    assert torch.equal(tiny_engine.decode_cfg(tok, noise, 2.5, n_tokens=[K] * 3), tiny_engine.decode_cfg(tok, noise, 2.5))
    for st in (0, 30, 49):
        assert torch.equal(tiny_engine.dit_velocity(tok, noise, st, n_tokens=K), tiny_engine.dit_velocity(tok, noise, st))


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "fp16", "bf16"])
def test_tiny_renderer_prefix(precision, gold):
    g, gp = gold("tiny_renderer"), gold("tiny_renderer_prefix")
    eng = _engine(TINY_R, precision)
    tok = torch.from_numpy(g["tokens"])
    assert torch.equal(eng.render(tok, n_tokens=TINY_R.K), eng.render(tok))
    err = _err(eng.render(tok, n_tokens=gp["n"]), gp["pred_x0"])
    print(f"[{precision}] renderer, n = {gp['n'].tolist()}: max-abs err {err:.3e}")
    assert err < TOL[precision]
    eng.close()


def test_tiny_prefix_against_reference(tiny_engine, gold):
    g, gp = gold("tiny"), gold("tiny_prefix")
    tol = TOL[tiny_engine.precision]
    tok, noise, n = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"]), gp["n"]
    for st in (0, 30, 49):
        err = _err(tiny_engine.dit_velocity(tok, noise, st, n_tokens=n), gp[f"v{st}"])
        print(f"[{tiny_engine.precision}] prefix velocity step {st}: max-abs err {err:.3e}")
        assert err < tol
    outs = []
    for use_graph in (False, True):
        tiny_engine.set_use_graph(use_graph)
        outs.append(tiny_engine.decode(tok, noise, n_tokens=n))
        err = _err(outs[-1], gp["pred_x0"])
        print(f"[{tiny_engine.precision}] prefix 50-step decode (graph={use_graph}): max-abs err {err:.3e}")
        assert err < tol
    assert torch.equal(outs[0], outs[1])                                  # graph and eager agree bit for bit
    err = _err(tiny_engine.decode_cfg(tok, noise, float(gp["cfg_scale"]), n_tokens=n), gp["pred_x0_cfg"])
    print(f"[{tiny_engine.precision}] prefix guided decode: max-abs err {err:.3e}")
    assert err < 2.5 * tol


def test_tiny_prefix_batch_composition(tiny_engine, gold):
    """Row b of a mixed batch depends only on image b and the batch's longest prefix."""
    g = gold("tiny")
    tok, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    tiny_engine.set_use_graph(True)
    abc = tiny_engine.decode(tok, noise, n_tokens=[3, 17, 32])
    cb = tiny_engine.decode(tok[[2, 1]], noise[[2, 1]], n_tokens=[32, 17])
    assert torch.equal(abc[2], cb[0]) and torch.equal(abc[1], cb[1])
    ab = tiny_engine.dit_velocity(tok[:2], noise[:2], 0, n_tokens=[3, 17])
    ba = tiny_engine.dit_velocity(tok[[1, 0]], noise[[1, 0]], 0, n_tokens=[17, 3])
    assert torch.equal(ab[0], ba[1]) and torch.equal(ab[1], ba[0])


def test_tiny_prefix_ids_after_the_prefix_are_never_read(tiny_engine, gold):
    from selftoktokenizer_b200.capi import SelftokError
    g = gold("tiny")
    tok, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    n = [3, 17, 32]
    ref = tiny_engine.decode(tok, noise, n_tokens=n)
    assert tiny_engine.id_errors() == 0
    hidden = torch.arange(C.TINY.K)[None, :] >= torch.tensor(n)[:, None]
    for fill in (-1, C.TINY.codebook_size):
        t = tok.clone()
        t[hidden] = fill
        assert torch.equal(tiny_engine.decode(t.to(DEV), noise, n_tokens=n), ref)       # device ids
        assert tiny_engine.id_errors() == 0
        assert torch.equal(tiny_engine.decode(t, noise, n_tokens=n), ref)               # host ids: checked inside the prefix only
    bad = tok.clone()
    bad[1, 16] = C.TINY.codebook_size                                                    # inside image 1's prefix of 17
    tiny_engine.decode(bad.to(DEV), noise, n_tokens=n)
    assert tiny_engine.id_errors() > 0
    with pytest.raises(SelftokError):
        tiny_engine.decode(bad, noise, n_tokens=n)


def test_tiny_prefix_graph_replay_refreshes_the_counts(tiny_engine, gold):
    g = gold("tiny")
    tok, noise = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"])
    tiny_engine.set_use_graph(True)
    tiny_engine.decode(tok, noise, n_tokens=[3, 17, 32])
    launches = tiny_engine.last_launch_count
    x_graph = tiny_engine.decode(tok, noise, n_tokens=[32, 5, 9])         # same n_max: the same graph, new counts
    assert tiny_engine.last_launch_count == launches
    tiny_engine.set_use_graph(False)
    assert torch.equal(tiny_engine.decode(tok, noise, n_tokens=[32, 5, 9]), x_graph)
    tiny_engine.set_use_graph(True)


def test_prefix_bad_arguments():
    from selftoktokenizer_b200.capi import SelftokError
    d = C.TINY
    eng = _engine(d, "fp16")
    tok = torch.randint(0, d.codebook_size, (2, d.K))
    noise = torch.randn(2, d.in_channels, d.latent, d.latent)
    for bad in (0, -1, d.K + 1, [1, d.K + 1], 2 ** 40):
        with pytest.raises(SelftokError):
            eng.decode(tok, noise, n_tokens=bad)
        with pytest.raises(SelftokError):
            eng.decode_cfg(tok, noise, 2.5, n_tokens=bad)
        with pytest.raises(SelftokError):
            eng.dit_velocity(tok, noise, 0, n_tokens=bad)
    with pytest.raises(SelftokError):
        eng.decode(tok, noise, n_tokens=[1, 2, 3])                       # one value per image
    with pytest.raises(SelftokError):
        eng.render(tok, n_tokens=4)                                      # not a renderer handle
    eng.close()
    r = _engine(TINY_R, "fp16")
    for bad in (0, d.K + 1):
        with pytest.raises(SelftokError):
            r.render(tok, n_tokens=bad)
    with pytest.raises(SelftokError):
        r.decode(tok, noise, n_tokens=4)                                 # a renderer handle does not decode
    r.close()


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "fp16"])
def test_mid_prefix_against_reference(precision, gold):
    """Holes that cover whole 64-key tiles (image 0 sees 1 of up to 128 context keys): the tile-skip path."""
    g, gp = gold("mid"), gold("mid_prefix")
    d = C.MID
    eng = _engine(d, precision)
    tok, noise, n = torch.from_numpy(g["tokens"]), torch.from_numpy(g["noise"]), gp["n"]
    x = eng.decode(tok, noise, n_tokens=n)
    err = _err(x, gp["pred_x0"])
    print(f"[{precision}] mid prefix 50-step decode n = {n.tolist()}: max-abs err {err:.3e}")
    assert err < TOL[precision]
    assert torch.equal(eng.decode(tok, noise, n_tokens=d.K), eng.decode(tok, noise))
    sub = eng.decode(tok[[3, 0]], noise[[3, 0]], n_tokens=[128, 1])
    assert torch.equal(sub[0], x[3]) and torch.equal(sub[1], x[0])
    eng.close()


@pytest.fixture(scope="module")
def full_sd():
    return synth.synth_state_dict(C.FULL, device=DEV)


@pytest.mark.parametrize("precision", ["bf16x3", "fp16"])
def test_full_prefix_velocity_against_reference(precision, full_sd, gold):
    gp, ge = gold("full_prefix_step"), gold("full_encode")
    d = C.FULL
    eng = _engine(d, precision, full_sd)
    tok = torch.from_numpy(ge["tokens"])
    x = synth.synth_tensor("golden.full.xt_prefix", (2, d.in_channels, d.latent, d.latent), "emb", 1.0)
    for st in (0, 30):
        err = _err(eng.dit_velocity(tok, x, st, n_tokens=gp["n"]), gp[f"v{st}"])
        print(f"[{precision}] full-geometry prefix velocity step {st}, n = {gp['n'].tolist()}: max-abs err {err:.3e}")
        assert err < 1e-3
    eng.close()


# one renderer pass does not average out operand rounding as the 50-step sampler does: single-pass half operands sit at the
# edge of 1e-3 at this geometry with or without a prefix (the plain renderer is held to the same 2.5e-3 in fp16)
@pytest.mark.parametrize("precision,tol", [("bf16x3", 1e-3), ("fp16", 2.5e-3)])
def test_full_renderer_prefix_against_reference(precision, tol, gold):
    gp, ge = gold("full_renderer_prefix"), gold("full_encode")
    d = dataclasses.replace(C.FULL, renderer=True)
    eng = _engine(d, precision, synth.synth_state_dict(d, device=DEV))
    err = _err(eng.render(torch.from_numpy(ge["tokens"]), n_tokens=gp["n"]), gp["pred_x0"])
    print(f"[{precision}] full-geometry renderer, n = {gp['n'].tolist()}: max-abs err {err:.3e}")
    assert err < tol
    eng.close()
