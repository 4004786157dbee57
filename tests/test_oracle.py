"""Pins the oracle (oracle/reference_path.py) — CPU only, no GPU needed.

1. Against the committed golden fixtures (outputs of the unmodified reference, tests/golden/make_golden.py):
   forward logits, loss, every parameter gradient, the in-place weight masking side effect, deterministic
   unconditional / conditional samples (bit-identical pixels) and the 7x7 receptive-field patterns.
2. Bit-for-bit against a 3-step Adam trajectory of the reference (losses, gradient norms, final weights),
   replayed single-threaded as it was recorded.

Tolerance between fixtures and oracle is 1e-5 relative (not bit-exact) only because the fixture was produced
with 1 thread and the box that replays it may sum in a different order; samples are compared exactly.
"""

import os

import pytest
import torch

from oracle import reference_path as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MODELS = ["pixel_cnn", "gated_pixel_cnn", "pixel_snail", "image_gpt"]


def close(a, b, rtol=1e-5, atol=1e-6):
    tol = atol + rtol * max(1.0, b.abs().max().item())
    return (a - b).abs().max().item() <= tol


def load(name):
    return torch.load(os.path.join(GOLD, name), weights_only=False)


@pytest.mark.parametrize("model", MODELS)
def test_model_forward_loss_grads_match_reference_fixture(model):
    fx = load(f"model_{model}.pt")
    logits, loss, grads, state = O.loss_and_grads(model, fx["state_before"], fx["x"], fx["cfg"])
    assert close(logits, fx["logits"]), (logits - fx["logits"]).abs().max()
    assert abs(loss.item() - fx["loss"].item()) <= 1e-5 * abs(fx["loss"].item())
    assert set(grads) == set(fx["grads"]), set(grads) ^ set(fx["grads"])
    for k, g in fx["grads"].items():
        assert close(grads[k], g, rtol=1e-4), (k, (grads[k] - g).abs().max().item())
    # CausalConv2d zeroes masked taps of the Parameter in place (reference nn/convolution.py:42)
    for k, v in fx["state_after"].items():
        if k in state and v.is_floating_point():
            assert torch.equal(state[k], v), k


@pytest.mark.parametrize("model", MODELS)
def test_model_sampling_is_bit_identical_to_reference_fixture(model):
    fx = load(f"model_{model}.pt")
    n, c, h, w = fx["x"].shape
    u = list(fx["sample_uniforms"])
    s = O.sample(model, fx["state_before"], fx["cfg"], O.uniform_sample_fn(u), n_samples=n, shape=(c, h, w))
    assert torch.equal(s, fx["sample"])
    cs = O.sample(model, fx["state_before"], fx["cfg"], O.uniform_sample_fn(u), conditioned_on=fx["cond"])
    assert torch.equal(cs, fx["cond_sample"])
    # reference models/tests.py:92-95 — pixels >= 0 are left untouched
    assert torch.equal(cs[:, :, : h // 2], fx["cond"][:, :, : h // 2])


def test_causal_conv_fixtures():
    fx = load("nn_blocks.pt")
    for tag in ["conv3x3A", "conv3x3B", "conv7x7A", "conv3x5B"]:
        f = fx[tag]
        kh, kw = f["weight_before"].shape[-2:]
        assert torch.equal(O.causal_mask(kh, kw, f["mask_center"]).expand_as(f["mask"]), f["mask"]), tag
        x = f["x"].clone().requires_grad_(True)
        w = f["weight_before"].clone().requires_grad_(True)
        b = f["bias"].clone().requires_grad_(True)
        y, wm = O.causal_conv2d(x, w, b, f["mask_center"], f["padding"])
        dx, dw, db = torch.autograd.grad(y, [x, w, b], f["dy"])
        assert torch.equal(wm.detach(), f["weight_after"]), tag
        assert close(y, f["y"]) and close(dx, f["dx"]) and close(dw, f["dw"], rtol=1e-4) and close(db, f["db"], rtol=1e-4), tag
        # masked taps still receive gradient (dense wgrad), SURVEY.md §7.3-3
        assert (dw * (1 - f["mask"])).abs().sum() > 0, tag


def test_gated_layernorm_attention_posenc_fixtures():
    fx = load("nn_blocks.pt")
    for tag, act in [("gated_tanh", torch.tanh), ("gated_identity", lambda z: z)]:
        f = fx[tag]
        x = f["x"].clone().requires_grad_(True)
        y = O.gated_activation(x, act)
        (dx,) = torch.autograd.grad(y, [x], f["dy"])
        assert close(y, f["y"]) and close(dx, f["dx"]), tag
    f = fx["layernorm"]
    x = f["x"].clone().requires_grad_(True)
    gm = f["gamma"].clone().requires_grad_(True)
    bt = f["beta"].clone().requires_grad_(True)
    y = O.nchw_layer_norm(x, gm, bt)
    dx, dg, db = torch.autograd.grad(y, [x, gm, bt], f["dy"])
    assert close(y, f["y"]) and close(dx, f["dx"]) and close(dg, f["dgamma"], rtol=1e-4) and close(db, f["dbeta"], rtol=1e-4)
    for tag in ["attn_causal_mh", "attn_strict_extra", "attn_defaults"]:
        f = fx[tag]
        kw = f["kwargs"]
        p = {"a." + k: v.clone().requires_grad_(True) for k, v in f["state"].items()}
        x = f["x"].clone().requires_grad_(True)
        extra = None if f["extra"] is None else f["extra"].clone().requires_grad_(True)
        embed = kw.get("embed_channels") or kw["in_channels"]
        out_c = kw.get("out_channels") or kw["in_channels"]
        y = O.causal_attention(x, p, "a.", kw.get("n_heads", 1), embed, out_c, kw.get("mask_center", False), extra)
        assert close(y, f["y"]), tag
        wrt = {"x": x, **({"extra": extra} if extra is not None else {}), **{k[2:]: v for k, v in p.items()}}
        gs = torch.autograd.grad(y, list(wrt.values()), f["dy"])
        for (k, _), g in zip(wrt.items(), gs):
            assert close(g, f["grads"][k], rtol=1e-4), (tag, k)
        if kw.get("mask_center"):
            # first position has no keys: output is exactly the projection bias (SURVEY.md Appendix A)
            assert torch.equal(y[:, :, 0, 0], p["a._proj.bias"].detach().expand(y.shape[0], -1))
    assert torch.equal(O.image_positional_encoding(fx["posenc"]["shape"]), fx["posenc"]["value"])


def test_receptive_fields_match_reference():
    """Known-answer causality patterns (SURVEY.md §4): output pixel (3,3) of a 7x7 input."""
    fx = load("receptive_fields.pt")
    ctor_cfg = {
        "pixel_cnn": None, "gated_pixel_cnn": None, "pixel_snail": None, "image_gpt": {"n_attention_heads": 2},
    }
    expect_full = torch.zeros(7, 7)
    expect_full[:3] = 1
    expect_full[3, :3] = 1
    for name in MODELS:
        assert fx[name][3, 3] == 0 and fx[name][4:].sum() == 0, name
    for name in ["pixel_cnn", "gated_pixel_cnn", "pixel_snail"]:
        assert torch.equal(fx[name], expect_full), name
    blind = expect_full.clone()
    blind[2, 6] = 0  # 3x3 mask-A blind spot of ImageGPT's input conv
    assert torch.equal(fx["image_gpt"], blind)
    assert ctor_cfg  # causality of the oracle itself is checked by the bit-exact probe below


# ------------------------------------------------------------------------------------------------
# Bit-exact checks
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", MODELS)
def test_oracle_bitwise_vs_reference_adam_trajectory(model):
    """Three training steps of the oracle reproduce the reference's losses, gradient norms and final weights bit for
    bit.  Single-threaded like the fixture: Adam turns a gradient that is rounding noise (e.g. the key bias of softmax
    attention) into a full +-lr step, so any change of summation order shows up in the weights."""
    fx = load(f"model_{model}.pt")
    tr = load("adam_trajectory.pt")[model]
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        ts = O.TrainState(model, fx["state_before"], fx["cfg"], lr=tr["lr"])
        g = torch.Generator().manual_seed(tr["data_seed"])
        for step in range(3):
            x = torch.rand(fx["x"].shape, generator=g)
            o_loss, o_norm = ts.step(x)
            assert o_loss == tr["losses"][step] and o_norm == tr["norms"][step], (step, o_loss, tr["losses"][step])
    finally:
        torch.set_num_threads(threads)
    assert {k for k, v in ts.p.items() if v.requires_grad} <= set(tr["state"])
    for k, v in tr["state"].items():
        if k in ts.p:
            assert torch.equal(ts.p[k].detach(), v), k


def test_oracle_bitwise_causality_probe():
    """Overwriting every pixel at/after (r,c) leaves forward(x)[:, :, r, c] bit-identical (SURVEY.md §7.3-7)."""
    for model in MODELS:
        fx = load(f"model_{model}.pt")
        x = fx["x"].clone()
        base = O.forward(model, O.trainable(fx["state_before"]), x, fx["cfg"]).detach()
        r, c = 4, 3
        x2 = x.clone()
        x2[:, :, r, c:] = -1
        x2[:, :, r + 1:, :] = -1
        out = O.forward(model, O.trainable(fx["state_before"]), x2, fx["cfg"]).detach()
        assert torch.equal(out[:, :, r, c], base[:, :, r, c]), model


def test_linear_causal_attention_matches_reference_fixture():
    """The oracle's LinearCausalAttention against outputs / gradients of the reference itself (nn/attention.py:209-275)."""
    from oracle import reference_path as O

    fx = torch.load(os.path.join(GOLD, "nn_linear_attention.pt"), weights_only=False)
    for tag, f in fx.items():
        kw = f["kwargs"]
        embed = kw.get("embed_channels") or kw["in_channels"]
        outc = kw.get("out_channels") or kw["in_channels"]
        pt = O.trainable(f["state"])
        x = f["x"].clone().requires_grad_(True)
        y = O.linear_causal_attention(x, pt, "", kw.get("n_heads", 1), embed, outc)
        y.backward(f["dy"])
        assert torch.allclose(y, f["y"], rtol=1e-5, atol=1e-5), tag
        assert torch.allclose(x.grad, f["grads"]["x"], rtol=1e-4, atol=1e-5), tag
        for k, v in pt.items():
            assert torch.allclose(v.grad, f["grads"][k], rtol=1e-4, atol=1e-4), (tag, k)
