"""ORACLE (test infrastructure only — never imported by the product path).

CPU fp32 restatement of the reference denoiser forward, written functionally over a plain
``state_dict``.  Every contraction/normalisation is the same ATen op the reference calls
(SURVEY.md §8c lists the call sites), in the same order, so on the same torch build this
matches the reference module bit-for-bit or to fp32 rounding; ``oracle/make_golden.py`` pins it
against the real reference (imported from /root/reference in the build container) and writes the
fixtures in ``tests/golden``.

Parity status: the reference has NO tests/golden vectors of its own ("parity unpinned" by the
reference); it is pinned here against outputs of the reference itself run in the build container
(fixtures + generating script committed).

Reference map (all under /root/reference):
  unet forward            unet1d/unet_1d_condition.py:743-1037
  timestep embedding      unet1d/embeddings.py:24-64, 157-218
  text-time embedding     unet1d/embeddings.py:421-434, 499-546
  ResnetBlock2D           unet1d/resnet.py:591-641
  Down/Upsample2D         unet1d/resnet.py:214-223, 138-173
  Transformer2DModel      unet1d/transformer_1d.py:256-295
  BasicTransformerBlock   unet1d/attention.py:130-203 ; GEGLU :280-301 ; FeedForward :252-255
  Attention (SDPA)        unet1d/attention_processor.py:971-1052 ; mask prep :309-336
  Diffusion_Encoder       model.py:403-415 ; sequence_mask modules/commons.py:149-153
"""
from __future__ import annotations

import math
from typing import Callable, Dict, Optional

import torch
import torch.nn.functional as F

from ns2vc_b200.arch import UNetConfig, build_plan


def sequence_mask(length: torch.Tensor, max_length: int) -> torch.Tensor:
    # modules/commons.py:149-153
    x = torch.arange(max_length, dtype=length.dtype, device=length.device)
    return x.unsqueeze(0) < length.unsqueeze(1)


def timestep_embedding(timesteps: torch.Tensor, dim: int, flip_sin_to_cos: bool, freq_shift: float) -> torch.Tensor:
    # embeddings.py:24-64
    half = dim // 2
    exponent = -math.log(10000) * torch.arange(0, half, dtype=torch.float32)
    exponent = exponent / (half - freq_shift)
    emb = torch.exp(exponent)
    emb = timesteps[:, None].float() * emb[None, :]
    emb = torch.cat([torch.sin(emb), torch.cos(emb)], dim=-1)
    if flip_sin_to_cos:
        emb = torch.cat([emb[:, half:], emb[:, :half]], dim=-1)
    if dim % 2 == 1:
        emb = F.pad(emb, (0, 1, 0, 0))
    return emb


def text_time_embedding(sd, p: str, ehs: torch.Tensor, num_heads: int) -> torch.Tensor:
    # embeddings.py:421-434 (TextTimeEmbedding) and :499-546 (AttentionPooling)
    x = F.layer_norm(ehs, (ehs.shape[-1],), sd[p + ".norm1.weight"], sd[p + ".norm1.bias"], 1e-5)
    bs, length, width = x.shape
    dph = width // num_heads

    def shape(t):
        t = t.view(bs, -1, num_heads, dph).transpose(1, 2)
        t = t.reshape(bs * num_heads, -1, dph).transpose(1, 2)
        return t

    class_token = x.mean(dim=1, keepdim=True) + sd[p + ".pool.positional_embedding"]
    x = torch.cat([class_token, x], dim=1)
    q = shape(F.linear(class_token, sd[p + ".pool.q_proj.weight"], sd[p + ".pool.q_proj.bias"]))
    k = shape(F.linear(x, sd[p + ".pool.k_proj.weight"], sd[p + ".pool.k_proj.bias"]))
    v = shape(F.linear(x, sd[p + ".pool.v_proj.weight"], sd[p + ".pool.v_proj.bias"]))
    scale = 1 / math.sqrt(math.sqrt(dph))
    weight = torch.einsum("bct,bcs->bts", q * scale, k * scale)
    weight = torch.softmax(weight.float(), dim=-1).type(weight.dtype)
    a = torch.einsum("bts,bcs->bct", weight, v)
    a = a.reshape(bs, -1, 1).transpose(1, 2)[:, 0, :]
    a = F.linear(a, sd[p + ".proj.weight"], sd[p + ".proj.bias"])
    return F.layer_norm(a, (a.shape[-1],), sd[p + ".norm2.weight"], sd[p + ".norm2.bias"], 1e-5)


def resnet_block(sd, p: str, x: torch.Tensor, temb: torch.Tensor, groups: int, eps: float, scale_shift: bool):
    # resnet.py:591-641
    h = F.group_norm(x, groups, sd[p + ".norm1.weight"], sd[p + ".norm1.bias"], eps)
    h = F.silu(h)
    h = F.conv1d(h, sd[p + ".conv1.weight"], sd[p + ".conv1.bias"], padding=1)
    t = F.linear(F.silu(temb), sd[p + ".time_emb_proj.weight"], sd[p + ".time_emb_proj.bias"])[:, :, None]
    if not scale_shift:
        h = h + t
    h = F.group_norm(h, groups, sd[p + ".norm2.weight"], sd[p + ".norm2.bias"], eps)
    if scale_shift:
        scale, shift = torch.chunk(t, 2, dim=1)
        h = h * (1 + scale) + shift
    h = F.silu(h)
    h = F.conv1d(h, sd[p + ".conv2.weight"], sd[p + ".conv2.bias"], padding=1)
    if (p + ".conv_shortcut.weight") in sd:
        x = F.conv1d(x, sd[p + ".conv_shortcut.weight"], sd[p + ".conv_shortcut.bias"])
    return (x + h) / 1.0


def attention(sd, p: str, hs: torch.Tensor, ehs: Optional[torch.Tensor], mask_bias: Optional[torch.Tensor], heads: int):
    # attention_processor.py:971-1052 (AttnProcessor2_0)
    B = hs.shape[0]
    q = F.linear(hs, sd[p + ".to_q.weight"])
    src = hs if ehs is None else ehs
    k = F.linear(src, sd[p + ".to_k.weight"])
    v = F.linear(src, sd[p + ".to_v.weight"])
    dh = k.shape[-1] // heads
    q = q.view(B, -1, heads, dh).transpose(1, 2)
    k = k.view(B, -1, heads, dh).transpose(1, 2)
    v = v.view(B, -1, heads, dh).transpose(1, 2)
    am = None
    if mask_bias is not None:
        # prepare_attention_mask (:309-336): [B,1,S] -> repeat_interleave(heads) -> view(B,heads,1,S)
        am = mask_bias.repeat_interleave(heads, dim=0).view(B, heads, -1, mask_bias.shape[-1])
    o = F.scaled_dot_product_attention(q, k, v, attn_mask=am, dropout_p=0.0, is_causal=False)
    o = o.transpose(1, 2).reshape(B, -1, heads * dh)
    return F.linear(o, sd[p + ".to_out.0.weight"], sd[p + ".to_out.0.bias"])


def transformer(sd, p: str, x: torch.Tensor, ehs: torch.Tensor, mask_bias, groups: int, heads: int):
    # transformer_1d.py:256-295 with one BasicTransformerBlock (attention.py:130-203)
    res = x
    h = F.group_norm(x, groups, sd[p + ".norm.weight"], sd[p + ".norm.bias"], 1e-6)
    h = F.conv1d(h, sd[p + ".proj_in.weight"], sd[p + ".proj_in.bias"])
    h = h.permute(0, 2, 1)
    b = p + ".transformer_blocks.0"
    C = h.shape[-1]
    n = F.layer_norm(h, (C,), sd[b + ".norm1.weight"], sd[b + ".norm1.bias"], 1e-5)
    h = attention(sd, b + ".attn1", n, None, None, heads) + h
    n = F.layer_norm(h, (C,), sd[b + ".norm2.weight"], sd[b + ".norm2.bias"], 1e-5)
    h = attention(sd, b + ".attn2", n, ehs, mask_bias, heads) + h
    n = F.layer_norm(h, (C,), sd[b + ".norm3.weight"], sd[b + ".norm3.bias"], 1e-5)
    # GEGLU (attention.py:299-301): value, gate = chunk(2); value * gelu(gate)   [erf gelu]
    g = F.linear(n, sd[b + ".ff.net.0.proj.weight"], sd[b + ".ff.net.0.proj.bias"])
    val, gate = g.chunk(2, dim=-1)
    g = val * F.gelu(gate)
    h = F.linear(g, sd[b + ".ff.net.2.weight"], sd[b + ".ff.net.2.bias"]) + h
    h = h.permute(0, 2, 1).contiguous()
    h = F.conv1d(h, sd[p + ".proj_out.weight"], sd[p + ".proj_out.bias"])
    return h + res


def unet_forward(sd: Dict[str, torch.Tensor], cfg: UNetConfig, sample: torch.Tensor, timestep: torch.Tensor,
                 ehs: torch.Tensor, ehs_mask: Optional[torch.Tensor] = None,
                 tap: Optional[Callable[[str, torch.Tensor], None]] = None) -> torch.Tensor:
    """sample [B,Cin,T] fp32, timestep [B] (int or fractional float), ehs [B,S,xdim],
    ehs_mask bool [B,S] (True = keep).  Returns [B,Cout,T].  ``tap(name, tensor)`` observes
    intermediate activations (channel-major, as in the reference)."""
    tap = tap or (lambda n, t: None)
    groups, heads = cfg.norm_num_groups, cfg.num_heads
    ss = cfg.resnet_time_scale_shift == "scale_shift"
    mask_bias = None
    if ehs_mask is not None:
        # unet_1d_condition.py:816-818
        mask_bias = ((1 - ehs_mask.to(sample.dtype)) * -10000.0).unsqueeze(1)
    timesteps = timestep
    if not torch.is_tensor(timesteps):
        timesteps = torch.tensor([timesteps], dtype=torch.float64 if isinstance(timestep, float) else torch.int64)
    elif timesteps.ndim == 0:
        timesteps = timesteps[None]
    timesteps = timesteps.expand(sample.shape[0])
    t_emb = timestep_embedding(timesteps, cfg.block_out_channels[0], cfg.flip_sin_to_cos, cfg.freq_shift)
    t_emb = t_emb.to(sample.dtype)
    emb = F.linear(t_emb, sd["time_embedding.linear_1.weight"], sd["time_embedding.linear_1.bias"])
    emb = F.silu(emb)
    emb = F.linear(emb, sd["time_embedding.linear_2.weight"], sd["time_embedding.linear_2.bias"])
    if cfg.addition_embed_type == "text":
        aug = text_time_embedding(sd, "add_embedding", ehs, cfg.addition_embed_type_num_heads)
        tap("aug_emb", aug)
        emb = emb + aug
    tap("emb", emb)

    h = F.conv1d(sample, sd["conv_in.weight"], sd["conv_in.bias"], padding=1)
    tap("conv_in", h)
    skips = []
    for op in build_plan(cfg):
        if op.kind == "push":
            skips.append(h)
        elif op.kind == "pop_cat":
            h = torch.cat([h, skips.pop()], dim=1)
        elif op.kind == "resnet":
            h = resnet_block(sd, op.prefix, h, emb, groups, cfg.norm_eps, ss)
            tap(op.prefix, h)
        elif op.kind == "xformer":
            h = transformer(sd, op.prefix, h, ehs, mask_bias, groups, heads)
            tap(op.prefix, h)
        elif op.kind == "down":
            h = F.conv1d(h, sd[op.prefix + ".conv.weight"], sd[op.prefix + ".conv.bias"], stride=2, padding=1)
            tap(op.prefix, h)
        elif op.kind == "up":
            # forced-size nearest upsample to the next skip's length (unet_1d_condition.py:789-797,
            # 1009-1010; resnet.py:160)
            h = F.interpolate(h, size=skips[-1].shape[2:], mode="nearest")
            h = F.conv1d(h, sd[op.prefix + ".conv.weight"], sd[op.prefix + ".conv.bias"], padding=1)
            tap(op.prefix, h)
    h = F.group_norm(h, groups, sd["conv_norm_out.weight"], sd["conv_norm_out.bias"], cfg.norm_eps)
    h = F.silu(h)
    return F.conv1d(h, sd["conv_out.weight"], sd["conv_out.bias"], padding=1)


def denoiser_forward(sd, cfg: UNetConfig, x: torch.Tensor, content_TBC: torch.Tensor, prompt_SBC: torch.Tensor,
                     prompt_lengths: torch.Tensor, t: torch.Tensor, tap=None) -> torch.Tensor:
    """Diffusion_Encoder.forward (model.py:403-415): x [B,100,T], content [T,B,256],
    prompt [S,B,256], prompt_lengths int64 [B], t [B]."""
    assert not torch.isnan(x).any()
    prompt = prompt_SBC.permute(1, 0, 2)
    content = content_TBC.permute(1, 2, 0)
    xin = torch.cat([x, content], dim=1)
    mask = sequence_mask(prompt_lengths, prompt.shape[1]).to(torch.bool)
    return unet_forward(sd, cfg, xin, t, prompt, mask, tap=tap)
