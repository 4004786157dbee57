"""CPU restatement of the reference's autoregressive-image hot path.  TEST INFRASTRUCTURE ONLY.

This file is the oracle (task §③): a plain-torch, CPU, fp32, *functional* restatement of what
EugenHotaj/pytorch-generative computes on the path named by BASELINE.json's north_star.  Only
`tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` legs may import
it; the product (`pytorch_generative_b200`) never does — its ops raise when the CUDA library is
missing.

Where the arithmetic lives: the reference delegates every op to PyTorch (third-party, absent from
/root/reference; requirements.txt pins only `torch>=1.5.1`).  This image has torch 2.11.0, the same
library the reference runs on here, so the restatement calls the same ATen ops (conv2d, layer_norm,
matmul, softmax, ...) in the same order as the reference call sites cited on each function; weights
come in as a state_dict with the reference's own key names, so a reference checkpoint is the input.

Pinning: the reference's tests hold no golden vectors for this path (SURVEY.md §8c: "parity
unpinned" upstream).  The oracle is therefore pinned against outputs of the reference itself, run in
a reference checkout: `tests/golden/make_golden.py` imports the reference, runs seeded tiny configs of
all four models and the four nn blocks (and a 3-step Adam trajectory of each model), and commits
inputs/outputs under tests/golden/; `tests/test_oracle.py` checks this file against those fixtures.
"""

import math

import torch
import torch.nn.functional as F

# --------------------------------------------------------------------------------------------------
# nn building blocks
# --------------------------------------------------------------------------------------------------


def causal_mask(kh, kw, mask_center):
    """0/1 tap mask of CausalConv2d — reference nn/convolution.py:35-38.

    Rows above the centre row are live; in the centre row the columns left of the centre are live,
    plus the centre itself unless `mask_center`.
    """
    m = torch.zeros(kh, kw)
    m[: kh // 2, :] = 1
    m[kh // 2, : kw // 2 + (0 if mask_center else 1)] = 1
    return m


def causal_conv2d(x, weight, bias, mask_center, padding):
    """CausalConv2d.forward — reference nn/convolution.py:41-43 (weight *= mask; conv2d).

    Returns (y, masked_weight); the reference overwrites the Parameter in place, the oracle returns the
    masked tensor so callers can check that side effect too.  Gradients flow to `weight` densely,
    exactly as in the reference where the mask multiply is outside autograd.
    """
    kh, kw = weight.shape[-2:]
    mask = causal_mask(kh, kw, mask_center).to(weight.dtype)
    with torch.no_grad():
        weight.mul_(mask)
    return F.conv2d(x, weight, bias, padding=padding), weight


def gated_activation(x, activation=torch.tanh):
    """GatedActivation.forward — reference nn/convolution.py:62-66."""
    c = x.shape[1]
    assert c % 2 == 0, "x must have an even number of channels."
    half = c // 2
    return activation(x[:, :half]) * torch.sigmoid(x[:, half:])


def nchw_layer_norm(x, gamma, beta, eps=1e-5):
    """NCHWLayerNorm.forward — reference nn/convolution.py:72-75 (LayerNorm over C of an NCHW tensor)."""
    y = F.layer_norm(x.permute(0, 2, 3, 1), (x.shape[1],), gamma, beta, eps)
    return y.permute(0, 3, 1, 2)


def image_positional_encoding(shape):
    """(N, 2, H, W) row/column coordinates in [-.5, .5) — reference nn/attention.py:49-57."""
    n, _, h, w = shape
    base = torch.zeros(n, 1, h, w)
    rows = torch.arange(-0.5, 0.5, 1 / h).view(1, 1, h, 1) + base
    cols = torch.arange(-0.5, 0.5, 1 / w).view(1, 1, 1, w) + base
    return torch.cat((rows, cols), dim=1)


def causal_attention(x, p, prefix, n_heads, embed_channels, out_channels, mask_center, extra_x=None):
    """CausalAttention.forward — reference nn/attention.py:120-161.

    q = 1x1(x); [k|v] = 1x1(cat(x, extra_x)); heads are contiguous channel blocks, sequence index is
    row*W+col; scores / sqrt(dk) are masked with tril(diagonal=-mask_center), soft-maxed, masked entries
    re-zeroed (the all-masked first row of a strict mask becomes zeros), then `_proj`.
    """
    n, _, h, w = x.shape
    s = h * w

    def heads(t):
        return t.view(n, n_heads, t.shape[1] // n_heads, s).transpose(2, 3)

    q = heads(F.conv2d(x, p[prefix + "_q.weight"], p[prefix + "_q.bias"]))
    kv_in = x if extra_x is None else torch.cat((x, extra_x), dim=1)
    kv = F.conv2d(kv_in, p[prefix + "_kv.weight"], p[prefix + "_kv.bias"])
    k, v = kv.split([embed_channels, out_channels], dim=1)
    k, v = heads(k), heads(v)
    allowed = torch.tril(torch.ones(s, s), diagonal=-int(mask_center)).view(1, 1, s, s)
    scores = (q @ k.transpose(2, 3)) / math.sqrt(k.shape[-1])
    scores = scores.masked_fill(allowed == 0, float("-inf"))
    weights = F.softmax(scores, dim=-1).masked_fill(allowed == 0, 0)
    out = (weights @ v).transpose(2, 3).contiguous().view(n, -1, h, w)
    return F.conv2d(out, p[prefix + "_proj.weight"], p[prefix + "_proj.bias"])


def linear_causal_attention(x, p, prefix, n_heads, embed_channels, out_channels, feature_fn=None):
    """LinearCausalAttention.forward — reference nn/attention.py:252-275 with the sequential numerator of
    `_UnnormalizedLinearCausalAttention` (:168-180) written as the same running sum (autograd differentiates the loop; the
    reference's hand-written backward :182-199 computes the same gradients).  The normaliser keeps the reference's
    `K.cumsum(1)` over dimension 1 of the [N, heads, L, d] tensors."""
    feature_fn = feature_fn or (lambda t: F.elu(t) + 1)
    n, _, h, w = x.shape

    def heads(t):
        return t.view(n, n_heads, t.shape[1] // n_heads, -1).transpose(2, 3)

    q = heads(F.conv2d(x, p[prefix + "_query.weight"], p[prefix + "_query.bias"]))
    kv = F.conv2d(x, p[prefix + "_kv.weight"], p[prefix + "_kv.bias"])
    k, v = kv.split([embed_channels, out_channels], dim=1)
    k, v = heads(k), heads(v)
    q, k = feature_fn(q), feature_fn(k)
    den = 1 / (torch.einsum("nlhi,nlhi->nlh", q, k.cumsum(1)) + 1e-10)
    rows, state = [], 0
    for i in range(v.shape[2]):
        state = state + k[:, :, i:i + 1].transpose(2, 3) @ v[:, :, i:i + 1]
        rows.append(q[:, :, i:i + 1] @ state)
    num = torch.cat(rows, dim=2)
    out = num * den.unsqueeze(-1)
    return out.transpose(2, 3).contiguous().view(n, -1, h, w)


# --------------------------------------------------------------------------------------------------
# Model stacks (state_dict keys are the reference's, SURVEY.md §8b)
# --------------------------------------------------------------------------------------------------


def _conv(x, p, name, padding=0):
    return F.conv2d(x, p[name + ".weight"], p[name + ".bias"], padding=padding)


def _count(p, prefix):
    """Number of consecutive integer-indexed children `prefix.{i}.` present in the state dict."""
    idx = set()
    for k in p:
        if k.startswith(prefix + "."):
            idx.add(int(k[len(prefix) + 1:].split(".")[0]))
    return len(idx)


def pixel_cnn_forward(p, x):
    """PixelCNN.forward — reference models/autoregressive/pixel_cnn.py:106-110 with the block at 52-53.

    7x7 type-A input conv; n residual blocks ReLU-1x1-ReLU-causal3x3(B)-ReLU-1x1 each applied as
    x + block(x) where block(x) itself is x + net(x) (so x <- 2x + net(x)); head ReLU-1x1-ReLU-1x1.
    """
    x, _ = causal_conv2d(x, p["_input.weight"], p["_input.bias"], True, 3)
    for i in range(_count(p, "_causal_layers")):
        pre = f"_causal_layers.{i}._net."
        t = _conv(F.relu(x), p, pre + "1")
        t, _ = causal_conv2d(F.relu(t), p[pre + "3.weight"], p[pre + "3.bias"], False, 1)
        t = _conv(F.relu(t), p, pre + "5")
        x = x + (x + t)
    x = _conv(F.relu(x), p, "_head.1")
    return _conv(F.relu(x), p, "_head.3")


def _gated_layer(p, pre, v_in, h_in, k, causal):
    """GatedPixelCNNLayer.forward — reference models/autoregressive/gated_pixel_cnn.py:112-130."""
    _, _, h, w = v_in.shape
    pad = (k - 1) // 2
    v = _conv(v_in, p, pre + "_vstack_1xN", padding=(0, pad))
    v = _conv(v, p, pre + "_vstack_Nx1", padding=(pad + 1, 0))[:, :, :h, :]
    link = _conv(v, p, pre + "_link")
    v = gated_activation(v + _conv(v_in, p, pre + "_vstack_1x1"))
    hs = link + _conv(h_in, p, pre + "_hstack_1xN", padding=(0, pad + int(causal)))[:, :, :, :w]
    hs = gated_activation(hs)
    skip = _conv(hs, p, pre + "_hstack_skip")
    hs = _conv(hs, p, pre + "_hstack_residual")
    if not causal:
        hs = hs + h_in
    return v, hs, skip


def gated_pixel_cnn_forward(p, x):
    """GatedPixelCNN.forward — reference gated_pixel_cnn.py:185-190 (k=7 causal input layer, k=3 layers)."""
    v, h, skips = _gated_layer(p, "_input.", x, x, 7, True)
    for i in range(_count(p, "_gated_layers")):
        v, h, skip = _gated_layer(p, f"_gated_layers.{i}.", v, h, 3, False)
        skips = skips + skip
    t = _conv(F.relu(skips), p, "_head.1")
    return _conv(F.relu(t), p, "_head.3")


def _snail_residual(p, pre, x):
    """ResidualBlock.forward — reference models/autoregressive/pixel_snail.py:52-56."""
    _, _, h, w = x.shape
    t = F.elu(_conv(F.elu(x), p, pre + "_input_conv", padding=1))[:, :, :h, :w]
    t = _conv(t, p, pre + "_output_conv", padding=1)[:, :, :h, :w]
    return x + gated_activation(t, lambda z: z)


def pixel_snail_forward(p, x):
    """PixelSNAIL.forward — reference pixel_snail.py:182-187 with the block at 103-119."""
    img = x
    x, _ = causal_conv2d(x, p["_input.weight"], p["_input.bias"], True, 1)
    key_ch = p["_pixel_snail_blocks.0._attention._q.weight"].shape[0]
    val_ch = p["_pixel_snail_blocks.0._attention._proj.weight"].shape[0]
    for i in range(_count(p, "_pixel_snail_blocks")):
        pre = f"_pixel_snail_blocks.{i}."
        res = x
        for j in range(_count(p, pre + "_residual")):
            res = _snail_residual(p, f"{pre}_residual.{j}.", res)
        pos = image_positional_encoding(img.shape)
        attn = causal_attention(torch.cat((pos, res), dim=1), p, pre + "_attention.", 1, key_ch, val_ch, True, img)
        res = F.elu(_conv(F.elu(res), p, pre + "_residual_out"))
        attn = F.elu(_conv(F.elu(attn), p, pre + "_attention_out"))
        x = x + F.elu(_conv(F.elu(res + attn), p, pre + "_out"))
    return _conv(_conv(x, p, "_output.0"), p, "_output.1")


def image_gpt_forward(p, x, n_heads):
    """ImageGPT.forward — reference models/autoregressive/image_gpt.py:105-109 with the block at 50-52.

    x <- causal3x3_A(x + pos); each block h = x + attn(ln1(x)), out = h + mlp(ln2(h)) is applied as
    x <- x + out (double residual); logits = 1x1(ln(x)).
    """
    x, _ = causal_conv2d(x + p["_pos"], p["_input.weight"], p["_input.bias"], True, 1)
    c = x.shape[1]
    for i in range(_count(p, "_transformer")):
        pre = f"_transformer.{i}."
        a = nchw_layer_norm(x, p[pre + "_ln1.weight"], p[pre + "_ln1.bias"])
        h = x + causal_attention(a, p, pre + "_attn.", n_heads, c, c, False)
        m = nchw_layer_norm(h, p[pre + "_ln2.weight"], p[pre + "_ln2.bias"])
        m = _conv(F.gelu(_conv(m, p, pre + "_out.0")), p, pre + "_out.2")
        x = x + (h + m)
    return _conv(nchw_layer_norm(x, p["_ln.weight"], p["_ln.bias"]), p, "_out")


FORWARDS = {
    "pixel_cnn": lambda p, x, cfg: pixel_cnn_forward(p, x),
    "gated_pixel_cnn": lambda p, x, cfg: gated_pixel_cnn_forward(p, x),
    "pixel_snail": lambda p, x, cfg: pixel_snail_forward(p, x),
    "image_gpt": lambda p, x, cfg: image_gpt_forward(p, x, cfg["n_attention_heads"]),
}


def forward(model, p, x, cfg=None):
    return FORWARDS[model](p, x, cfg or {})


# --------------------------------------------------------------------------------------------------
# Parameter layout of the four constructors (state-dict keys and shapes, torch default initialisers)
# --------------------------------------------------------------------------------------------------
def init_state(model, cfg, seed=0):
    """A freshly initialised state dict of `model` with the reference's keys and shapes (SURVEY.md §8b) and the same
    torch initialisers its constructors use (nn.Conv2d / nn.LayerNorm defaults, `_pos` zeros): what
    `Model(**cfg).state_dict()` returns in the reference (pixel_cnn.py:59-104, gated_pixel_cnn.py:136-183,
    pixel_snail.py:130-180, image_gpt.py:64-103).  Used by the CPU timing arm, which must not import the product."""
    torch.manual_seed(seed)
    sd = {}

    def conv(name, cin, cout, k=1):
        m = torch.nn.Conv2d(cin, cout, k)
        sd[name + ".weight"], sd[name + ".bias"] = m.weight.detach().clone(), m.bias.detach().clone()

    def causal(name, cin, cout, k, mask_center):
        conv(name, cin, cout, k)
        kh, kw = sd[name + ".weight"].shape[-2:]
        sd[name + ".mask"] = causal_mask(kh, kw, mask_center).expand_as(sd[name + ".weight"]).clone()

    def ln(name, c):
        sd[name + ".weight"], sd[name + ".bias"] = torch.ones(c), torch.zeros(c)

    def attention(pre, cin, embed, out, extra=0):
        conv(pre + "_q", cin, embed)
        conv(pre + "_kv", cin + extra, embed + out)
        conv(pre + "_proj", out, out)

    if model == "pixel_cnn":
        c, res = cfg["in_channels"], cfg.get("residual_channels", 128)
        causal("_input", c, 2 * res, 7, True)
        for i in range(cfg.get("n_residual", 15)):
            pre = f"_causal_layers.{i}._net."
            conv(pre + "1", 2 * res, res)
            causal(pre + "3", res, res, 3, False)
            conv(pre + "5", res, 2 * res)
        conv("_head.1", 2 * res, cfg.get("head_channels", 32))
        conv("_head.3", cfg.get("head_channels", 32), cfg["out_channels"])
    elif model == "gated_pixel_cnn":
        g = cfg.get("gated_channels", 128)

        def layer(pre, cin, k):
            conv(pre + "_vstack_1xN", cin, g, (1, k))
            conv(pre + "_vstack_Nx1", g, 2 * g, (k // 2 + 1, 1))
            conv(pre + "_vstack_1x1", cin, 2 * g)
            conv(pre + "_link", 2 * g, 2 * g)
            conv(pre + "_hstack_1xN", cin, 2 * g, (1, k // 2 + 1))
            conv(pre + "_hstack_residual", g, g)
            conv(pre + "_hstack_skip", g, g)

        layer("_input.", cfg["in_channels"], 7)
        for i in range(cfg.get("n_gated", 10)):
            layer(f"_gated_layers.{i}.", g, 3)
        conv("_head.1", g, cfg.get("head_channels", 32))
        conv("_head.3", cfg.get("head_channels", 32), cfg["out_channels"])
    elif model == "pixel_snail":
        c, img = cfg.get("n_channels", 64), cfg["in_channels"]
        key, val = cfg.get("attention_key_channels", 4), cfg.get("attention_value_channels", 32)
        causal("_input", img, c, 3, True)
        for i in range(cfg.get("n_pixel_snail_blocks", 8)):
            pre = f"_pixel_snail_blocks.{i}."
            for j in range(cfg.get("n_residual_blocks", 2)):
                conv(f"{pre}_residual.{j}._input_conv", c, c, 2)
                conv(f"{pre}_residual.{j}._output_conv", c, 2 * c, 2)
            attention(pre + "_attention.", c + 2, key, val, extra=img)
            conv(pre + "_residual_out", c, c)
            conv(pre + "_attention_out", val, c)
            conv(pre + "_out", c, c)
        conv("_output.0", c, c // 2)
        conv("_output.1", c // 2, cfg["out_channels"])
    elif model == "image_gpt":
        c, s = cfg.get("n_embedding_channels", 16), cfg.get("in_size", 28)
        sd["_pos"] = torch.zeros(1, cfg["in_channels"], s, s)
        causal("_input", cfg["in_channels"], c, 3, True)
        for i in range(cfg.get("n_transformer_blocks", 8)):
            pre = f"_transformer.{i}."
            ln(pre + "_ln1", c)
            ln(pre + "_ln2", c)
            attention(pre + "_attn.", c, c, c)
            conv(pre + "_out.0", c, 4 * c)
            conv(pre + "_out.2", 4 * c, c)
        ln("_ln", c)
        conv("_out", c, cfg["out_channels"])
    else:
        raise ValueError(model)
    return sd


# --------------------------------------------------------------------------------------------------
# Recipe loss, training step, sampling
# --------------------------------------------------------------------------------------------------


def recipe_loss(x, preds):
    """loss_fn of every recipe — reference image_gpt.py:158-162 (`reshape`, since the reference's `.view`
    raises on its own channels-last 3-channel logits, SURVEY.md §7.3-5)."""
    b = x.shape[0]
    loss = F.binary_cross_entropy_with_logits(preds.reshape(b, -1), x.reshape(b, -1), reduction="none")
    return loss.sum(dim=1).mean()


def trainable(p):
    """Clones a state dict into leaf tensors; floating-point entries that are Parameters in the
    reference (everything except the `mask` buffers and `_c/_h/_w`) require grad."""
    out = {}
    for k, v in p.items():
        t = v.detach().clone()
        if t.is_floating_point() and not k.endswith("mask"):
            t.requires_grad_(True)
        out[k] = t
    return out


def loss_and_grads(model, p, x, cfg=None):
    """One forward + recipe loss + backward.  Returns (logits, loss, {name: grad}, masked state)."""
    pt = trainable(p)
    logits = forward(model, pt, x, cfg)
    loss = recipe_loss(x, logits)
    loss.backward()
    grads = {k: v.grad for k, v in pt.items() if v.requires_grad and v.grad is not None}
    return logits.detach(), loss.detach(), grads, {k: v.detach() for k, v in pt.items()}


class TrainState:
    """Trainer._train_one_batch restated — reference trainer.py:173-193: zero_grad, forward, loss,
    backward, clip_grad_norm_(params, 1e50) (always computed for the grad_norm metric), Adam step,
    MultiplicativeLR step, two .item() reads."""

    def __init__(self, model, p, cfg=None, lr=1e-3, lr_gamma=0.999977):
        self.model, self.cfg = model, cfg
        self.p = trainable(p)
        self.params = [v for v in self.p.values() if v.requires_grad]
        self.opt = torch.optim.Adam(self.params, lr=lr)
        self.sched = torch.optim.lr_scheduler.MultiplicativeLR(self.opt, lr_lambda=lambda _: lr_gamma)

    def step(self, x):
        self.opt.zero_grad()
        loss = recipe_loss(x, forward(self.model, self.p, x, self.cfg))
        loss.backward()
        norm = torch.nn.utils.clip_grad_norm_(self.params, 1e50)
        self.opt.step()
        self.sched.step()
        return loss.item(), norm.item()


@torch.no_grad()
def sample(model, p, cfg, sample_fn, n_samples=None, conditioned_on=None, shape=None):
    """AutoregressiveModel.sample — reference models/base.py:97-120: raster scan, one full forward per
    pixel, all channels of a pixel drawn together, only entries < 0 are overwritten."""
    if conditioned_on is None:
        c, h, w = shape
        conditioned_on = torch.ones(n_samples, c, h, w) * -1
    else:
        conditioned_on = conditioned_on.clone()
    n, c, h, w = conditioned_on.shape
    for row in range(h):
        for col in range(w):
            out = forward(model, p, conditioned_on, cfg)[:, :, row, col]
            out = sample_fn(out).view(n, c)
            cur = conditioned_on[:, :, row, col]
            conditioned_on[:, :, row, col] = torch.where(cur < 0, out, cur)
    return conditioned_on


def uniform_sample_fn(uniforms):
    """Deterministic Bernoulli draw used for bit-identical sampling parity (SURVEY.md §7.3-7): consumes
    one pre-drawn uniform tensor [n, c] per pixel in raster order."""
    it = iter(uniforms)

    def fn(logits):
        return (next(it).to(logits.device) < torch.sigmoid(logits)).float()

    return fn
