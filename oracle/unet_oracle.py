"""TEST INFRASTRUCTURE ONLY — CPU fp32 restatement of the reference's denoising UNet forward.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may import this.
It is a functional walk over a reference-keyed state dict (no nn.Modules), pinned against the UNMODIFIED
reference by tests/test_oracle_cpu.py (test_*_matches_reference_golden*) through the committed fixtures under
tests/golden/ (generated from the reference by tests/golden/make_golden*.py).

Each function cites the reference lines it restates (paths relative to /root/reference).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F


def sinusoid(t: torch.Tensor, dim: int) -> torch.Tensor:
    """lvdm/models/utils_diffusion.py:8-28 (cos first, then sin; zero pad for odd dim)."""
    half = dim // 2
    freqs = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=torch.float32) / half).to(t.device)
    a = t[:, None].float() * freqs[None]
    e = torch.cat([a.cos(), a.sin()], dim=-1)
    if dim % 2:
        e = torch.cat([e, torch.zeros_like(e[:, :1])], dim=-1)
    return e


class SD:
    """State-dict view with a key prefix."""

    def __init__(self, sd, prefix=""):
        self.sd, self.prefix = sd, prefix

    def __call__(self, name):
        return self.sd[self.prefix + name].float()

    def has(self, name):
        return (self.prefix + name) in self.sd

    def sub(self, name):
        return SD(self.sd, self.prefix + name)


def group_norm(x, p: SD, eps):
    return F.group_norm(x, 32, p("weight"), p("bias"), eps)


def res_block(p: SD, x, emb, B, temporal_conv=True):
    """openaimodel3d.py:210-236 (ResBlock._forward) + :272-279 (TemporalConvBlock)."""
    h = F.conv2d(F.silu(group_norm(x, p.sub("in_layers.0."), 1e-5)), p("in_layers.2.weight"), p("in_layers.2.bias"),
                 padding=1)
    e = F.linear(F.silu(emb), p("emb_layers.1.weight"), p("emb_layers.1.bias"))
    h = h + e[:, :, None, None]
    h = F.conv2d(F.silu(group_norm(h, p.sub("out_layers.0."), 1e-5)), p("out_layers.3.weight"),
                 p("out_layers.3.bias"), padding=1)
    if p.has("skip_connection.weight"):
        x = F.conv2d(x, p("skip_connection.weight"), p("skip_connection.bias"))
    h = x + h
    if temporal_conv and p.has("temopral_conv.conv1.0.weight"):
        n, c, hh, ww = h.shape
        v = h.reshape(B, n // B, c, hh, ww).permute(0, 2, 1, 3, 4)          # b c t h w
        y = v
        for i, ci in ((1, 2), (2, 3), (3, 3), (4, 3)):
            q = p.sub(f"temopral_conv.conv{i}.")
            y = F.conv3d(F.silu(group_norm(y, q.sub("0."), 1e-5)), q(f"{ci}.weight"), q(f"{ci}.bias"),
                         padding=(1, 0, 0))
        v = v + y
        h = v.permute(0, 2, 1, 3, 4).reshape(n, c, hh, ww)
    return h


# "einsum": the explicit softmax(q k^T) v of CrossAttention.forward (the numerics oracle: fp32 softmax, fixed op order).
# "sdpa":   F.scaled_dot_product_attention = what CrossAttention.efficient_forward (attention.py:146-209, xformers
#           installed) amounts to on a GPU: fused flash kernels, no materialised scores.  Only bench.py's library
#           baseline switches to it (the fair "best library path" to beat, SURVEY 8c).
ATTENTION_IMPL = "einsum"


def attention_core(q, k, v, heads):
    """attention.py:101-125: softmax(q k^T / sqrt(d)) v per head; q [b, n, h*d]."""
    b, n, inner = q.shape
    d = inner // heads
    qh = q.reshape(b, n, heads, d).transpose(1, 2)
    kh = k.reshape(b, -1, heads, d).transpose(1, 2)
    vh = v.reshape(b, -1, heads, d).transpose(1, 2)
    if ATTENTION_IMPL == "sdpa":
        return F.scaled_dot_product_attention(qh, kh, vh).transpose(1, 2).reshape(b, n, inner)
    s = (qh @ kh.transpose(-1, -2)) * d ** -0.5
    o = s.softmax(dim=-1) @ vh
    return o.transpose(1, 2).reshape(b, n, inner)


def cross_attention(p: SD, x, context, heads, text_len=77):
    """attention.py:81-144 (CrossAttention.forward).  context None -> self attention."""
    q = F.linear(x, p("to_q.weight"))
    if context is None:
        k = F.linear(x, p("to_k.weight"))
        v = F.linear(x, p("to_v.weight"))
        out = attention_core(q, k, v, heads)
    else:
        txt = context[:, :text_len]
        out = attention_core(q, F.linear(txt, p("to_k.weight")), F.linear(txt, p("to_v.weight")), heads)
        if p.has("to_k_ip.weight"):
            img = context[:, text_len:]
            out = out + 1.0 * attention_core(q, F.linear(img, p("to_k_ip.weight")), F.linear(img, p("to_v_ip.weight")),
                                             heads)
    return F.linear(out, p("to_out.0.weight"), p("to_out.0.bias"))


def layer_norm(x, p: SD):
    return F.layer_norm(x, (x.shape[-1],), p("weight"), p("bias"), 1e-5)


def transformer_block(p: SD, x, context, heads):
    """attention.py:242-246 (BasicTransformerBlock._forward) + :415-442 (GEGLU feed-forward, erf gelu)."""
    x = cross_attention(p.sub("attn1."), layer_norm(x, p.sub("norm1.")), None, heads) + x
    x = cross_attention(p.sub("attn2."), layer_norm(x, p.sub("norm2.")), context, heads) + x
    h = F.linear(layer_norm(x, p.sub("norm3.")), p("ff.net.0.proj.weight"), p("ff.net.0.proj.bias"))
    a, g = h.chunk(2, dim=-1)
    return F.linear(a * F.gelu(g), p("ff.net.2.weight"), p("ff.net.2.bias")) + x


def spatial_transformer(p: SD, x, context, heads):
    """attention.py:294-310 (SpatialTransformer.forward), use_linear and conv projections."""
    n, c, hh, ww = x.shape
    h = group_norm(x, p.sub("norm."), 1e-6)
    w_in, w_out = p("proj_in.weight"), p("proj_out.weight")
    h = h.permute(0, 2, 3, 1).reshape(n, hh * ww, c)
    h = F.linear(h, w_in.reshape(w_in.shape[0], -1), p("proj_in.bias"))
    h = transformer_block(p.sub("transformer_blocks.0."), h, context, heads)
    h = F.linear(h, w_out.reshape(w_out.shape[0], -1), p("proj_out.bias"))
    return h.reshape(n, hh, ww, c).permute(0, 3, 1, 2) + x


def temporal_transformer(p: SD, x, B, heads):
    """attention.py:365-412 (TemporalTransformer.forward, only_self_att: attn1 and attn2 are both self-attn)."""
    n, c, hh, ww = x.shape
    T = n // B
    v = x.reshape(B, T, c, hh, ww).permute(0, 2, 1, 3, 4)                    # b c t h w
    h = group_norm(v, p.sub("norm."), 1e-6)
    h = h.permute(0, 3, 4, 2, 1).reshape(B * hh * ww, T, c)                  # (b h w) t c
    w_in, w_out = p("proj_in.weight"), p("proj_out.weight")
    h = F.linear(h, w_in.reshape(w_in.shape[0], -1), p("proj_in.bias"))
    h = transformer_block(p.sub("transformer_blocks.0."), h, None, heads)
    h = F.linear(h, w_out.reshape(w_out.shape[0], -1), p("proj_out.bias"))
    h = h.reshape(B, hh, ww, T, c).permute(0, 3, 4, 1, 2).reshape(n, c, hh, ww)
    return h + x


def run_layers(p: SD, layers, h, emb, context, B, lay):
    """openaimodel3d.py:36-48 (TimestepEmbedSequential.forward)."""
    for i, l in enumerate(layers):
        q = p.sub(f"{i}.")
        if l.kind == "conv_in":
            h = F.conv2d(h, q("weight"), q("bias"), padding=1)
        elif l.kind == "res":
            h = res_block(q, h, emb, B, lay.temporal_conv)
        elif l.kind == "st":
            h = spatial_transformer(q, h, context, l.heads)
        elif l.kind == "tt":
            h = temporal_transformer(q, h, B, l.heads)
        elif l.kind == "down":
            h = F.conv2d(h, q("op.weight"), q("op.bias"), stride=2, padding=1)
        elif l.kind == "up":
            h = F.conv2d(F.interpolate(h, scale_factor=2, mode="nearest"), q("conv.weight"), q("conv.bias"), padding=1)
        else:
            raise ValueError(l.kind)
    return h


@torch.no_grad()
def unet_forward(sd, lay, x, timesteps, context, fs=None, prefix=""):
    """openaimodel3d.py:548-603 (UNetModel.forward).  x [B, C, T, H, W] -> [B, out, T, H, W], fp32."""
    p = SD(sd, prefix)
    B, _, T, H, W = x.shape
    mc = lay.model_channels

    def mlp(name, e):
        return F.linear(F.silu(F.linear(e, p(f"{name}.0.weight"), p(f"{name}.0.bias"))), p(f"{name}.2.weight"),
                        p(f"{name}.2.bias"))

    emb = mlp("time_embed", sinusoid(timesteps, mc))
    if context.shape[1] == 77 + T * 16:
        txt = context[:, :77].repeat_interleave(T, dim=0)
        img = context[:, 77:].reshape(B * T, 16, context.shape[-1])
        ctx = torch.cat([txt, img], dim=1)
    else:
        ctx = context.repeat_interleave(T, dim=0)
    emb = emb.repeat_interleave(T, dim=0)
    if lay.fs_condition:
        if fs is None:
            fs = torch.full((B,), lay.default_fs, dtype=torch.long, device=x.device)
        emb = emb + mlp("fps_embedding", sinusoid(fs, mc)).repeat_interleave(T, dim=0)
    h = x.float().permute(0, 2, 1, 3, 4).reshape(B * T, -1, H, W)
    skips = []
    for bi, (pref, layers) in enumerate(lay.input_blocks):
        h = run_layers(p.sub(pref + "."), layers, h, emb, ctx, B, lay)
        if bi == 0 and lay.init_attn:
            h = run_layers(p.sub("init_attn."), lay.init_attn, h, emb, ctx, B, lay)
        skips.append(h)
    h = run_layers(p.sub("middle_block."), lay.middle_block, h, emb, ctx, B, lay)
    for pref, layers in lay.output_blocks:
        h = torch.cat([h, skips.pop()], dim=1)
        h = run_layers(p.sub(pref + "."), layers, h, emb, ctx, B, lay)
    y = F.conv2d(F.silu(group_norm(h, p.sub("out.0."), 1e-5)), p("out.2.weight"), p("out.2.bias"), padding=1)
    return y.reshape(B, T, -1, H, W).permute(0, 2, 1, 3, 4)
