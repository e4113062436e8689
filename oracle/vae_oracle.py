"""TEST INFRASTRUCTURE ONLY — CPU fp32 restatement of the dual-reference video decoder (and the encoder that
produces its hidden states).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
reference leg may import this.  Pinned against the unmodified reference by tests/test_oracle_cpu.py
(test_*_matches_reference_golden*) and tests/golden/.  Paths cited are relative to the reference repository's root.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .unet_oracle import SD, group_norm


def swish(x):
    return x * torch.sigmoid(x)


def resnet2d(p: SD, x):
    """lvdm/models/autoencoder_dualref.py:72-92 (ResnetBlock.forward, temb=None)."""
    h = F.conv2d(swish(group_norm(x, p.sub("norm1."), 1e-6)), p("conv1.weight"), p("conv1.bias"), padding=1)
    h = F.conv2d(swish(group_norm(h, p.sub("norm2."), 1e-6)), p("conv2.weight"), p("conv2.bias"), padding=1)
    if p.has("nin_shortcut.weight"):
        x = F.conv2d(x, p("nin_shortcut.weight"), p("nin_shortcut.bias"))
    return x + h


def video_res_block(p: SD, x, T):
    """autoencoder_dualref.py:892-911 (VideoResBlock.forward) + :672-698 (3-D ResBlock, skip_t_emb)."""
    x = resnet2d(p, x)
    n, c, hh, ww = x.shape
    v = x.reshape(n // T, T, c, hh, ww).permute(0, 2, 1, 3, 4)               # b c t h w
    q = p.sub("time_stack.")
    h = F.conv3d(F.silu(group_norm(v, q.sub("in_layers.0."), 1e-5)), q("in_layers.2.weight"), q("in_layers.2.bias"),
                 padding=(1, 0, 0))
    h = F.conv3d(F.silu(group_norm(h, q.sub("out_layers.0."), 1e-5)), q("out_layers.3.weight"),
                 q("out_layers.3.bias"), padding=(1, 0, 0))
    vt = v + h
    alpha = torch.sigmoid(p("mix_factor"))
    out = alpha * vt + (1.0 - alpha) * v
    return out.permute(0, 2, 1, 3, 4).reshape(n, c, hh, ww)


def mid_attention(p: SD, x):
    """autoencoder_dualref.py:172-206 (MemoryEfficientAttnBlock): single head, d = C."""
    n, c, hh, ww = x.shape
    h = group_norm(x, p.sub("norm."), 1e-6)
    q = F.conv2d(h, p("q.weight"), p("q.bias")).flatten(2).transpose(1, 2)
    k = F.conv2d(h, p("k.weight"), p("k.bias")).flatten(2).transpose(1, 2)
    v = F.conv2d(h, p("v.weight"), p("v.bias")).flatten(2).transpose(1, 2)
    o = F.scaled_dot_product_attention(q[:, None], k[:, None], v[:, None])[:, 0]
    o = o.transpose(1, 2).reshape(n, c, hh, ww)
    return x + F.conv2d(o, p("proj_out.weight"), p("proj_out.bias"))


def fusion_attention(p: SD, x, ctx, heads=8):
    """autoencoder_dualref.py:270-341: every frame attends to the tokens of BOTH reference frames."""
    n, c, hh, ww = x.shape
    h = group_norm(x, p.sub("norm."), 1e-6).flatten(2).transpose(1, 2)        # n (hw) c
    q = F.linear(h, p("to_q.weight"))
    b, cc, l, ch, cw = ctx.shape
    assert b == 1, "reference semantics are only defined for one clip per decode call (SURVEY App. C.3)"
    c2 = ctx.permute(0, 2, 3, 4, 1).reshape(1, l * ch * cw, cc)                # [ref0 tokens ; ref1 tokens]
    k = F.linear(c2, p("to_k.weight")).expand(n, -1, -1)
    v = F.linear(c2, p("to_v.weight")).expand(n, -1, -1)
    d = q.shape[-1] // heads

    def split(t):
        return t.reshape(t.shape[0], t.shape[1], heads, d).transpose(1, 2)

    o = F.scaled_dot_product_attention(split(q), split(k), split(v))
    o = o.transpose(1, 2).reshape(n, hh * ww, heads * d)
    o = F.linear(o, p("to_out.0.weight"), p("to_out.0.bias"))
    return x + o.transpose(1, 2).reshape(n, c, hh, ww)


def combiner(p: SD, x, ctx):
    """autoencoder_dualref.py:357-368: 1x1 conv of the two reference maps added to first / last frame."""
    c2 = F.conv2d(ctx[0].permute(1, 0, 2, 3), p("conv.weight"), p("conv.bias"))   # [2, C, h, w]
    x = x.clone()
    x[0] = x[0] + c2[0]
    x[-1] = x[-1] + c2[1]
    return x


@torch.no_grad()
def decode(sd, lay, z, ref_context, prefix="first_stage_model.decoder."):
    """autoencoder.py:112-116 (post_quant_conv skipped because kwargs are passed) +
    autoencoder_dualref.py:489-527 (Decoder.forward) for ONE chunk of T = z.shape[0] latents of one clip.
    z [T, 4, h, w] (already divided by scale_factor), ref_context: 5 maps [1, C, 2, H_l, W_l]."""
    p = SD(sd, prefix)
    T = z.shape[0]
    h = F.conv2d(z.float(), p("conv_in.weight"), p("conv_in.bias"), padding=1)
    h = video_res_block(p.sub("mid.block_1."), h, T)
    h = mid_attention(p.sub("mid.attn_1."), h)
    h = video_res_block(p.sub("mid.block_2."), h, T)
    for i_level in reversed(range(lay.num_resolutions)):
        lv = lay.levels[i_level]
        for j in range(len(lv["blocks"])):
            h = video_res_block(p.sub(f"up.{i_level}.block.{j}."), h, T)
        if ref_context is not None:
            q = p.sub(f"attn_refinement.{i_level}.")
            ctx = ref_context[i_level].float()
            h = fusion_attention(q, h, ctx) if lv["refine"] == "fusion" else combiner(q, h, ctx)
        if lv["upsample"]:
            q = p.sub(f"up.{i_level}.upsample.")
            h = F.conv2d(F.interpolate(h, scale_factor=2, mode="nearest"), q("conv.weight"), q("conv.bias"), padding=1)
    h = swish(group_norm(h, p.sub("norm_out."), 1e-6))
    if ref_context is not None:
        h = combiner(p.sub(f"attn_refinement.{lay.num_resolutions}."), h, ref_context[-1].float())
    h = F.conv2d(h, p("conv_out.weight"), p("conv_out.bias"), padding=1)          # AE3DConv :929-935
    v = h.reshape(1, T, *h.shape[1:]).permute(0, 2, 1, 3, 4)
    v = F.conv3d(v, p("conv_out.time_mix_conv.weight"), p("conv_out.time_mix_conv.bias"), padding=(1, 0, 0))
    return v.permute(0, 2, 1, 3, 4).reshape(T, -1, h.shape[-2], h.shape[-1])


@torch.no_grad()
def decode_first_stage(sd, lay, z, ref_context, scale_factor=0.18215, chunk=16,
                       prefix="first_stage_model.decoder."):
    """ddpm3d.py:647-683 (decode_core, perframe_ae=True): z [1, 4, T, h, w] -> [1, 3, T, 8h, 8w]."""
    b, c, t, hh, ww = z.shape
    assert b == 1, "B > 1 is defined as B independent B = 1 runs (SURVEY §8e)"
    zz = z.permute(0, 2, 1, 3, 4).reshape(b * t, c, hh, ww) * (1.0 / scale_factor)
    outs = [decode(sd, lay, zz[i:i + chunk], ref_context, prefix) for i in range(0, zz.shape[0], chunk)]
    out = torch.cat(outs, dim=0)
    return out.reshape(b, t, *out.shape[1:]).permute(0, 2, 1, 3, 4)


@torch.no_grad()
def encode_hidden(sd, lay, x, prefix="first_stage_model.encoder."):
    """lvdm/modules/networks/ae_modules.py:432-475 (Encoder.forward, return_hidden_states=True).
    x [N, 3, H, W] -> (h [N, 2*z, H/8, W/8] before quant_conv, [5 hidden maps])."""
    p = SD(sd, prefix)
    h = F.conv2d(x.float(), p("conv_in.weight"), p("conv_in.bias"), padding=1)
    first = h
    hidden = []
    for i, lv in enumerate(lay.levels):
        for j in range(len(lv["blocks"])):
            h = resnet2d(p.sub(f"down.{i}.block.{j}."), h)
        hidden.append(h)
        if lv["downsample"]:
            q = p.sub(f"down.{i}.downsample.")
            h = F.conv2d(F.pad(h, (0, 1, 0, 1)), q("conv.weight"), q("conv.bias"), stride=2)
    hidden.append(first)
    h = resnet2d(p.sub("mid.block_1."), h)
    h = mid_attention(p.sub("mid.attn_1."), h)
    h = resnet2d(p.sub("mid.block_2."), h)
    h = swish(group_norm(h, p.sub("norm_out."), 1e-6))
    return F.conv2d(h, p("conv_out.weight"), p("conv_out.bias"), padding=1), hidden
