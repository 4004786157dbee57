"""Generates the golden fixtures in this directory by running the UNMODIFIED reference.

Needs a checkout of the reference (EugenHotaj/pytorch-generative):
    python tests/golden/make_golden.py <path to the pytorch-generative checkout>
The reference's own tests hold no numeric vectors for this path (SURVEY.md §8c), so these fixtures —
outputs of the reference itself on seeded inputs — are what pins the oracle (oracle/reference_path.py)
and, through it, the CUDA path.  Each fixture is a small torch .pt dict; the tests read only these files,
never the reference itself.

Fixtures
  model_<name>.pt : cfg, state_dict (default init under manual_seed + N(0, 0.05) noise so that biases,
                    LayerNorm affine and `_pos` are non-trivial), x, logits, loss, grads of every
                    parameter, state after forward (masked CausalConv2d weights), an unconditional sample
                    and a conditional sample drawn with pre-generated uniforms in raster order.
  nn_blocks.pt    : CausalConv2d (3x3 A/B, 7x7 A, rectangular 3x5), GatedActivation (tanh / identity),
                    NCHWLayerNorm, CausalAttention (strict / non-strict, extra input, multi-head):
                    outputs and all gradients.
  nn_linear_attention.pt : LinearCausalAttention (one head; two heads with embed != out channels): output, all gradients.
  receptive_fields.pt : debug.compute_receptive_field-style 7x7 causality patterns of the four models.
  adam_trajectory.pt : three recipe training steps of each model from its model_<name>.pt weights: loss and
                    gradient norm of every step, floating-point state after the last step.
"""

import os
import sys
import warnings

import torch

HERE = os.path.dirname(os.path.abspath(__file__))

MODEL_CFGS = {
    "pixel_cnn": dict(cls="PixelCNN", shape=(2, 1, 8, 8), binarized=True,
                      kwargs=dict(in_channels=1, out_channels=1, n_residual=2, residual_channels=8, head_channels=8)),
    "gated_pixel_cnn": dict(cls="GatedPixelCNN", shape=(2, 3, 8, 8), binarized=False,
                            kwargs=dict(in_channels=3, out_channels=3, n_gated=2, gated_channels=8, head_channels=8)),
    "pixel_snail": dict(cls="PixelSNAIL", shape=(2, 3, 8, 8), binarized=False,
                        kwargs=dict(in_channels=3, out_channels=3, n_channels=16, n_pixel_snail_blocks=2,
                                    n_residual_blocks=1, attention_key_channels=4, attention_value_channels=8)),
    "image_gpt": dict(cls="ImageGPT", shape=(2, 3, 8, 8), binarized=False,
                      kwargs=dict(in_channels=3, out_channels=3, in_size=8, n_transformer_blocks=2,
                                  n_attention_heads=2, n_embedding_channels=32)),
}


def synthetic_batch(shape, binarized, seed):
    g = torch.Generator().manual_seed(seed)
    if binarized:  # dynamically-binarized-MNIST stand-in (reference datasets.py:16-17)
        return torch.bernoulli(torch.full(shape, 0.5), generator=g)
    return torch.randint(0, 256, shape, generator=g).float() / 255  # ToTensor range (datasets.py:170)


def perturb_(model, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for prm in model.parameters():
            prm.add_(torch.randn(prm.shape, generator=g) * 0.05)


def loss_fn(x, preds):
    b = x.shape[0]
    l = torch.nn.functional.binary_cross_entropy_with_logits(preds.reshape(b, -1), x.reshape(b, -1), reduction="none")
    return l.sum(dim=1).mean()


def make_model_fixture(pg, name, spec):
    torch.manual_seed(0)
    uniforms = None

    def sample_fn(logits):
        return (next(uniforms) < torch.sigmoid(logits)).float()

    model = getattr(pg.models, spec["cls"])(sample_fn=sample_fn, **spec["kwargs"])
    perturb_(model, 1)
    x = synthetic_batch(spec["shape"], spec["binarized"], 2)
    state_before = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model.zero_grad()
    logits = model(x)
    loss = loss_fn(x, logits)
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
    state_after = {k: v.detach().clone() for k, v in model.state_dict().items()}
    n, c, h, w = spec["shape"]
    g = torch.Generator().manual_seed(3)
    u = [torch.rand(n, c, generator=g) for _ in range(h * w)]
    uniforms = iter(u)
    sample = model.sample(n_samples=n)
    cond = x.clone()
    cond[:, :, h // 2:, :] = -1
    uniforms = iter(u)
    cond_sample = model.sample(conditioned_on=cond)
    return dict(name=name, cls=spec["cls"], cfg=spec["kwargs"], x=x, state_before=state_before,
                state_after=state_after, logits=logits.detach().contiguous(), loss=loss.detach(), grads=grads,
                sample_uniforms=torch.stack(u), sample=sample, cond=cond, cond_sample=cond_sample)


def _grads(out, tensors):
    g = torch.Generator().manual_seed(9)
    dy = torch.randn(out.shape, generator=g)
    gs = torch.autograd.grad(out, tensors, dy)
    return dy, [t.detach().clone() for t in gs]


def make_nn_fixture(pg):
    fx = {}
    g = torch.Generator().manual_seed(4)
    # CausalConv2d variants
    for tag, (mc, cin, cout, ks, pad) in {
        "conv3x3A": (True, 3, 16, 3, 1), "conv3x3B": (False, 8, 8, 3, 1), "conv7x7A": (True, 1, 16, 7, 3),
        "conv3x5B": (False, 2, 4, (3, 5), (1, 2)),
    }.items():
        torch.manual_seed(5)
        m = pg.nn.CausalConv2d(mc, in_channels=cin, out_channels=cout, kernel_size=ks, padding=pad)
        x = torch.randn(2, cin, 8, 8, generator=g, requires_grad=True)
        w0 = m.weight.detach().clone()
        y = m(x)
        dy, (dx, dw, db) = _grads(y, [x, m.weight, m.bias])
        fx[tag] = dict(mask_center=mc, padding=pad, x=x.detach(), weight_before=w0, weight_after=m.weight.detach().clone(),
                       bias=m.bias.detach().clone(), mask=m.mask.clone(), y=y.detach(), dy=dy, dx=dx, dw=dw, db=db)
    # GatedActivation
    for tag, act in {"gated_tanh": torch.tanh, "gated_identity": torch.nn.Identity()}.items():
        m = pg.nn.GatedActivation(activation_fn=act)
        x = torch.randn(2, 16, 8, 8, generator=g, requires_grad=True)
        y = m(x)
        dy, (dx,) = _grads(y, [x])
        fx[tag] = dict(x=x.detach(), y=y.detach(), dy=dy, dx=dx)
    # NCHWLayerNorm
    torch.manual_seed(6)
    m = pg.nn.NCHWLayerNorm(32)
    with torch.no_grad():
        m.weight.add_(torch.randn(32, generator=g) * 0.3)
        m.bias.add_(torch.randn(32, generator=g) * 0.3)
    x = (torch.randn(2, 32, 8, 8, generator=g) * 3 + 1).requires_grad_(True)
    y = m(x)
    dy, (dx, dgm, dbt) = _grads(y, [x, m.weight, m.bias])
    fx["layernorm"] = dict(x=x.detach(), gamma=m.weight.detach().clone(), beta=m.bias.detach().clone(),
                           y=y.detach().contiguous(), dy=dy, dx=dx, dgamma=dgm, dbeta=dbt)
    # CausalAttention variants
    for tag, kw in {
        "attn_causal_mh": dict(in_channels=32, n_heads=2, embed_channels=32, out_channels=32, mask_center=False),
        "attn_strict_extra": dict(in_channels=18, n_heads=1, embed_channels=4, out_channels=8, mask_center=True,
                                  extra_input_channels=3),
        "attn_defaults": dict(in_channels=16),
    }.items():
        torch.manual_seed(7)
        m = pg.nn.CausalAttention(**kw)
        x = torch.randn(2, kw["in_channels"], 8, 8, generator=g, requires_grad=True)
        extra = None
        if kw.get("extra_input_channels"):
            extra = torch.randn(2, kw["extra_input_channels"], 8, 8, generator=g, requires_grad=True)
        y = m(x, extra) if extra is not None else m(x)
        wrt = [x] + ([extra] if extra is not None else []) + list(m.parameters())
        dy, gs = _grads(y, wrt)
        names = ["x"] + (["extra"] if extra is not None else []) + [n for n, _ in m.named_parameters()]
        fx[tag] = dict(kwargs=kw, x=x.detach(), extra=None if extra is None else extra.detach(),
                       state={k: v.detach().clone() for k, v in m.state_dict().items()}, y=y.detach(), dy=dy,
                       grads=dict(zip(names, gs)))
    # image_positional_encoding
    fx["posenc"] = dict(shape=(2, 3, 8, 6), value=pg.nn.image_positional_encoding((2, 3, 8, 6)).clone())
    return fx


def make_receptive_fields(pg):
    """Gradient-based causality patterns on 7x7 single-channel inputs for output pixel (3,3)
    (reference debug.py:7-21, restated so the input is seeded)."""
    out = {}
    ctors = {
        "pixel_cnn": lambda: pg.models.PixelCNN(1, 1, n_residual=2, residual_channels=4, head_channels=4),
        "gated_pixel_cnn": lambda: pg.models.GatedPixelCNN(1, 1, n_gated=2, gated_channels=4, head_channels=4),
        "pixel_snail": lambda: pg.models.PixelSNAIL(1, 1, n_channels=8, n_pixel_snail_blocks=1, n_residual_blocks=1,
                                                    attention_key_channels=2, attention_value_channels=4),
        "image_gpt": lambda: pg.models.ImageGPT(1, 1, in_size=7, n_transformer_blocks=1, n_attention_heads=2,
                                                n_embedding_channels=8),
    }
    for name, ctor in ctors.items():
        torch.manual_seed(8)
        model = ctor()
        img = torch.randn(1, 1, 7, 7, generator=torch.Generator().manual_seed(8), requires_grad=True)
        model(img)[0, 0, 3, 3].mean().backward()
        out[name] = (img.grad.abs()[0, 0] > 0).float()
    return out


def make_linear_attention_fixture(pg):
    """LinearCausalAttention (reference nn/attention.py:209-275): two head geometries, outputs and all gradients."""
    out = {}
    for tag, kwargs, shape in [("one_head", dict(in_channels=8), (2, 8, 5, 6)),
                               ("two_heads", dict(in_channels=6, n_heads=2, embed_channels=8, out_channels=12), (2, 6, 4, 7))]:
        torch.manual_seed(11)
        m = pg.nn.LinearCausalAttention(**kwargs)
        g = torch.Generator().manual_seed(12)
        x = torch.randn(shape, generator=g).requires_grad_(True)
        y = m(x)
        dy = torch.randn(y.shape, generator=g)
        y.backward(dy)
        out[tag] = dict(kwargs=kwargs, state={k: v.detach().clone() for k, v in m.state_dict().items()}, x=x.detach().clone(),
                        y=y.detach().clone(), dy=dy, grads=dict(x=x.grad.clone(), **{k: p.grad.clone() for k, p in m.named_parameters()}))
    return out


def make_adam_trajectory(pg):
    """Trainer._train_one_batch (reference trainer.py:173-193) three times per model, from the model fixture's weights,
    on uniform batches drawn from one seeded generator: zero_grad, forward, recipe loss, backward,
    clip_grad_norm_(1e50), Adam, MultiplicativeLR."""
    out = {}
    for name, spec in MODEL_CFGS.items():
        fx = torch.load(os.path.join(HERE, f"model_{name}.pt"), weights_only=False)
        model = getattr(pg.models, spec["cls"])(**spec["kwargs"])
        model.load_state_dict(fx["state_before"])
        lr = 5e-3 if name == "image_gpt" else 1e-3
        opt = torch.optim.Adam(model.parameters(), lr=lr)
        sched = torch.optim.lr_scheduler.MultiplicativeLR(opt, lr_lambda=lambda _: 0.999977)
        g = torch.Generator().manual_seed(11)
        losses, norms = [], []
        for _ in range(3):
            x = torch.rand(fx["x"].shape, generator=g)
            opt.zero_grad()
            loss = loss_fn(x, model(x))
            loss.backward()
            norm = torch.nn.utils.clip_grad_norm_(model.parameters(), 1e50)
            opt.step()
            sched.step()
            losses.append(loss.item())
            norms.append(norm.item())
        state = {k: v.detach().clone() for k, v in model.state_dict().items() if v.is_floating_point()}
        out[name] = dict(lr=lr, data_seed=11, losses=losses, norms=norms, state=state)
    return out


def main():
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "pytorch_generative")):
        sys.exit("usage: make_golden.py <path to the pytorch-generative checkout>")
    sys.path.insert(0, os.path.abspath(sys.argv[1]))
    warnings.filterwarnings("ignore")
    torch.set_num_threads(1)  # deterministic summation order for the fixtures
    import pytorch_generative as pg

    for name, spec in MODEL_CFGS.items():
        fx = make_model_fixture(pg, name, spec)
        torch.save(fx, os.path.join(HERE, f"model_{name}.pt"))
        print(f"model_{name}.pt  loss={fx['loss'].item():.6f}  |logits|max={fx['logits'].abs().max().item():.4f}")
    torch.save(make_nn_fixture(pg), os.path.join(HERE, "nn_blocks.pt"))
    torch.save(make_receptive_fields(pg), os.path.join(HERE, "receptive_fields.pt"))
    print("nn_blocks.pt, receptive_fields.pt written")
    torch.save(make_linear_attention_fixture(pg), os.path.join(HERE, "nn_linear_attention.pt"))
    print("nn_linear_attention.pt written")
    torch.save(make_adam_trajectory(pg), os.path.join(HERE, "adam_trajectory.pt"))
    print("adam_trajectory.pt written")


if __name__ == "__main__":
    main()
