"""ORACLE (test infrastructure, not product code): pure-PyTorch restatement of the diffusers v0.27.2 building blocks
that the Ctrl-Adapter hot path calls into.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference`` legs may import
anything under ``oracle/``; the product package ``ctrl_adapter_b200`` never does.

PARITY STATUS: diffusers is a third-party dependency of the reference that is NOT vendored under /root/reference and
is not installable here (SURVEY.md section 8c), so the arithmetic in this file is restated from the published
v0.27.2 sources ("parity unpinned" for this layer: no upstream golden vectors exist).  The reference's OWN modules
(model/*.py, controlnet/*.py) are executed on top of these blocks through ``oracle/diffusers_shim`` to generate the
golden vectors under tests/golden/, which pins the in-repo layer of the path.

Module / parameter names follow diffusers so that state-dict keys are identical (SURVEY.md Appendix B).
Each class cites the reference call site that reaches it.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch
import torch.nn.functional as F
from torch import nn


# ------------------------------------------------------------------------------------------------
# embeddings  (reached from model/adapter_spatial_temporal.py:56-66,207-208,263-265; controlnet/controlnet.py:257-263)
# ------------------------------------------------------------------------------------------------
def get_timestep_embedding(timesteps: torch.Tensor, embedding_dim: int, flip_sin_to_cos: bool = False,
                           downscale_freq_shift: float = 1, scale: float = 1, max_period: int = 10000):
    assert timesteps.dim() == 1
    half_dim = embedding_dim // 2
    exponent = -math.log(max_period) * torch.arange(0, half_dim, dtype=torch.float32, device=timesteps.device)
    exponent = exponent / (half_dim - downscale_freq_shift)
    # fp32 exp / sin / cos are not correctly rounded and differ between CPU vector units: they are evaluated in fp64 and
    # rounded once, so the fp32 embedding (and every golden vector downstream of it) is the same on every machine
    emb = torch.exp(exponent.double()).float()
    emb = timesteps[:, None].float() * emb[None, :]
    emb = scale * emb
    emb = torch.cat([torch.sin(emb.double()), torch.cos(emb.double())], dim=-1).float()
    if flip_sin_to_cos:
        emb = torch.cat([emb[:, half_dim:], emb[:, :half_dim]], dim=-1)
    if embedding_dim % 2 == 1:
        emb = F.pad(emb, (0, 1, 0, 0))
    return emb


class Timesteps(nn.Module):
    def __init__(self, num_channels: int, flip_sin_to_cos: bool, downscale_freq_shift: float):
        super().__init__()
        self.num_channels = num_channels
        self.flip_sin_to_cos = flip_sin_to_cos
        self.downscale_freq_shift = downscale_freq_shift

    def forward(self, timesteps):
        return get_timestep_embedding(timesteps, self.num_channels, flip_sin_to_cos=self.flip_sin_to_cos,
                                      downscale_freq_shift=self.downscale_freq_shift)


class TimestepEmbedding(nn.Module):
    def __init__(self, in_channels: int, time_embed_dim: int, act_fn: str = "silu", out_dim: int = None,
                 post_act_fn: Optional[str] = None, cond_proj_dim=None, sample_proj_bias=True):
        super().__init__()
        self.linear_1 = nn.Linear(in_channels, time_embed_dim, sample_proj_bias)
        self.cond_proj = nn.Linear(cond_proj_dim, in_channels, bias=False) if cond_proj_dim is not None else None
        assert act_fn in ("silu", "swish")
        self.act = nn.SiLU()
        time_embed_dim_out = out_dim if out_dim is not None else time_embed_dim
        self.linear_2 = nn.Linear(time_embed_dim, time_embed_dim_out, sample_proj_bias)
        self.post_act = None

    def forward(self, sample, condition=None):
        if condition is not None:
            sample = sample + self.cond_proj(condition)
        # get_timestep_embedding returns fp32 and the reference's adapter passes it on uncast: float64 parity runs
        # need it in the layer's dtype (a no-op in fp32, and what autocast does anyway)
        sample = self.linear_1(sample.to(self.linear_1.weight.dtype))
        sample = self.act(sample)
        sample = self.linear_2(sample)
        return sample


# ------------------------------------------------------------------------------------------------
# attention / feed-forward / transformer blocks
# (reached from model/adapter_spatial_temporal.py:108-130,271,280 and from the ControlNet / UNet Transformer2DModel)
# ------------------------------------------------------------------------------------------------
class Attention(nn.Module):
    """diffusers Attention with AttnProcessor2_0 (F.scaled_dot_product_attention, no mask, no norm, no residual)."""

    def __init__(self, query_dim: int, cross_attention_dim: Optional[int] = None, heads: int = 8, dim_head: int = 64,
                 dropout: float = 0.0, bias: bool = False, upcast_attention: bool = False, out_bias: bool = True):
        super().__init__()
        self.inner_dim = dim_head * heads
        self.heads = heads
        self.dim_head = dim_head
        self.scale = dim_head ** -0.5
        cross = cross_attention_dim if cross_attention_dim is not None else query_dim
        self.to_q = nn.Linear(query_dim, self.inner_dim, bias=bias)
        self.to_k = nn.Linear(cross, self.inner_dim, bias=bias)
        self.to_v = nn.Linear(cross, self.inner_dim, bias=bias)
        self.to_out = nn.ModuleList([nn.Linear(self.inner_dim, query_dim, bias=out_bias), nn.Dropout(dropout)])

    def forward(self, hidden_states, encoder_hidden_states=None, attention_mask=None):
        b = hidden_states.shape[0]
        q = self.to_q(hidden_states)
        ctx = hidden_states if encoder_hidden_states is None else encoder_hidden_states
        k = self.to_k(ctx)
        v = self.to_v(ctx)
        hd = self.inner_dim // self.heads
        q = q.view(b, -1, self.heads, hd).transpose(1, 2)
        k = k.view(b, -1, self.heads, hd).transpose(1, 2)
        v = v.view(b, -1, self.heads, hd).transpose(1, 2)
        h = F.scaled_dot_product_attention(q, k, v, attn_mask=attention_mask, dropout_p=0.0, is_causal=False)
        h = h.transpose(1, 2).reshape(b, -1, self.heads * hd).to(q.dtype)
        h = self.to_out[0](h)
        h = self.to_out[1](h)
        return h


class GEGLU(nn.Module):
    def __init__(self, dim_in: int, dim_out: int, bias: bool = True):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out * 2, bias=bias)

    def forward(self, hidden_states):
        hidden_states, gate = self.proj(hidden_states).chunk(2, dim=-1)
        return hidden_states * F.gelu(gate)


class FeedForward(nn.Module):
    def __init__(self, dim: int, dim_out: Optional[int] = None, mult: int = 4, dropout: float = 0.0,
                 activation_fn: str = "geglu", final_dropout: bool = False, inner_dim=None, bias: bool = True):
        super().__init__()
        if inner_dim is None:
            inner_dim = int(dim * mult)
        dim_out = dim_out if dim_out is not None else dim
        assert activation_fn in ("geglu", "gelu")
        act = GEGLU(dim, inner_dim, bias=bias) if activation_fn == "geglu" else _GELUProj(dim, inner_dim, bias=bias)
        self.net = nn.ModuleList([act, nn.Dropout(dropout), nn.Linear(inner_dim, dim_out, bias=bias)])

    def forward(self, hidden_states):
        for m in self.net:
            hidden_states = m(hidden_states)
        return hidden_states


class _GELUProj(nn.Module):
    """diffusers activations.GELU (approximate="none"): Linear followed by exact erf GELU."""

    def __init__(self, dim_in: int, dim_out: int, bias: bool = True):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out, bias=bias)

    def forward(self, hidden_states):
        return F.gelu(self.proj(hidden_states))


class BasicTransformerBlock(nn.Module):
    def __init__(self, dim: int, num_attention_heads: int, attention_head_dim: int, dropout=0.0,
                 cross_attention_dim: Optional[int] = None, activation_fn: str = "geglu", attention_bias: bool = False,
                 only_cross_attention: bool = False, double_self_attention: bool = False, upcast_attention: bool = False,
                 norm_elementwise_affine: bool = True, norm_type: str = "layer_norm", norm_eps: float = 1e-5,
                 final_dropout: bool = False, attention_type: str = "default", **_unused):
        super().__init__()
        self.only_cross_attention = only_cross_attention
        self.norm1 = nn.LayerNorm(dim, elementwise_affine=norm_elementwise_affine, eps=norm_eps)
        self.attn1 = Attention(query_dim=dim, heads=num_attention_heads, dim_head=attention_head_dim, dropout=dropout,
                               bias=attention_bias,
                               cross_attention_dim=cross_attention_dim if only_cross_attention else None,
                               upcast_attention=upcast_attention)
        if cross_attention_dim is not None or double_self_attention:
            self.norm2 = nn.LayerNorm(dim, norm_eps, norm_elementwise_affine)
            self.attn2 = Attention(query_dim=dim,
                                   cross_attention_dim=cross_attention_dim if not double_self_attention else None,
                                   heads=num_attention_heads, dim_head=attention_head_dim, dropout=dropout,
                                   bias=attention_bias, upcast_attention=upcast_attention)
        else:
            self.norm2 = None
            self.attn2 = None
        self.norm3 = nn.LayerNorm(dim, norm_eps, norm_elementwise_affine)
        self.ff = FeedForward(dim, dropout=dropout, activation_fn=activation_fn, final_dropout=final_dropout)

    def forward(self, hidden_states, attention_mask=None, encoder_hidden_states=None, encoder_attention_mask=None,
                timestep=None, cross_attention_kwargs=None, class_labels=None, added_cond_kwargs=None):
        norm_hidden_states = self.norm1(hidden_states)
        attn_output = self.attn1(norm_hidden_states,
                                 encoder_hidden_states=encoder_hidden_states if self.only_cross_attention else None,
                                 attention_mask=attention_mask)
        hidden_states = attn_output + hidden_states
        if self.attn2 is not None:
            norm_hidden_states = self.norm2(hidden_states)
            attn_output = self.attn2(norm_hidden_states, encoder_hidden_states=encoder_hidden_states,
                                     attention_mask=encoder_attention_mask)
            hidden_states = attn_output + hidden_states
        norm_hidden_states = self.norm3(hidden_states)
        ff_output = self.ff(norm_hidden_states)
        hidden_states = ff_output + hidden_states
        return hidden_states


class TemporalBasicTransformerBlock(nn.Module):
    def __init__(self, dim: int, time_mix_inner_dim: int, num_attention_heads: int, attention_head_dim: int,
                 cross_attention_dim: Optional[int] = None):
        super().__init__()
        self.is_res = dim == time_mix_inner_dim
        self.norm_in = nn.LayerNorm(dim)
        self.ff_in = FeedForward(dim, dim_out=time_mix_inner_dim, activation_fn="geglu")
        self.norm1 = nn.LayerNorm(time_mix_inner_dim)
        self.attn1 = Attention(query_dim=time_mix_inner_dim, heads=num_attention_heads, dim_head=attention_head_dim,
                               cross_attention_dim=None)
        if cross_attention_dim is not None:
            self.norm2 = nn.LayerNorm(time_mix_inner_dim)
            self.attn2 = Attention(query_dim=time_mix_inner_dim, cross_attention_dim=cross_attention_dim,
                                   heads=num_attention_heads, dim_head=attention_head_dim)
        else:
            self.norm2 = None
            self.attn2 = None
        self.norm3 = nn.LayerNorm(time_mix_inner_dim)
        self.ff = FeedForward(time_mix_inner_dim, activation_fn="geglu")

    def forward(self, hidden_states, num_frames: int, encoder_hidden_states=None):
        batch_frames, seq_length, channels = hidden_states.shape
        batch_size = batch_frames // num_frames
        hidden_states = hidden_states[None, :].reshape(batch_size, num_frames, seq_length, channels)
        hidden_states = hidden_states.permute(0, 2, 1, 3)
        hidden_states = hidden_states.reshape(batch_size * seq_length, num_frames, channels)
        residual = hidden_states
        hidden_states = self.norm_in(hidden_states)
        hidden_states = self.ff_in(hidden_states)
        if self.is_res:
            hidden_states = hidden_states + residual
        norm_hidden_states = self.norm1(hidden_states)
        attn_output = self.attn1(norm_hidden_states, encoder_hidden_states=None)
        hidden_states = attn_output + hidden_states
        if self.attn2 is not None:
            norm_hidden_states = self.norm2(hidden_states)
            attn_output = self.attn2(norm_hidden_states, encoder_hidden_states=encoder_hidden_states)
            hidden_states = attn_output + hidden_states
        norm_hidden_states = self.norm3(hidden_states)
        ff_output = self.ff(norm_hidden_states)
        if self.is_res:
            hidden_states = ff_output + hidden_states
        else:
            hidden_states = ff_output
        hidden_states = hidden_states[None, :].reshape(batch_size, seq_length, num_frames, channels)
        hidden_states = hidden_states.permute(0, 2, 1, 3)
        hidden_states = hidden_states.reshape(batch_size * num_frames, seq_length, channels)
        return hidden_states


# ------------------------------------------------------------------------------------------------
# resnets, samplers, blender  (reached from model/resnet_block_2d.py:11-25,141,149; adapter_spatial_temporal.py:96-104,134-152)
# ------------------------------------------------------------------------------------------------
class Upsample2D(nn.Module):
    def __init__(self, channels: int, use_conv: bool = False, use_conv_transpose: bool = False,
                 out_channels: Optional[int] = None, name: str = "conv", kernel_size=None, padding=1, bias=True,
                 interpolate=True, **_unused):
        super().__init__()
        assert not use_conv_transpose
        self.channels = channels
        self.out_channels = out_channels or channels
        self.use_conv = use_conv
        self.name = name
        self.interpolate = interpolate
        self.conv = None
        if use_conv:
            conv = nn.Conv2d(self.channels, self.out_channels, kernel_size=3 if kernel_size is None else kernel_size,
                             padding=padding, bias=bias)
            if name == "conv":
                self.conv = conv
            else:
                self.Conv2d_0 = conv

    def forward(self, hidden_states, output_size=None, *args, **kwargs):
        assert hidden_states.shape[1] == self.channels
        dtype = hidden_states.dtype
        if dtype == torch.bfloat16:
            hidden_states = hidden_states.to(torch.float32)
        if hidden_states.shape[0] >= 64:
            hidden_states = hidden_states.contiguous()
        if self.interpolate:
            if output_size is None:
                hidden_states = F.interpolate(hidden_states, scale_factor=2.0, mode="nearest")
            else:
                hidden_states = F.interpolate(hidden_states, size=output_size, mode="nearest")
        if dtype == torch.bfloat16:
            hidden_states = hidden_states.to(dtype)
        if self.use_conv:
            hidden_states = self.conv(hidden_states) if self.name == "conv" else self.Conv2d_0(hidden_states)
        return hidden_states


class Downsample2D(nn.Module):
    def __init__(self, channels: int, use_conv: bool = False, out_channels: Optional[int] = None, padding: int = 1,
                 name: str = "conv", kernel_size=3, bias=True, **_unused):
        super().__init__()
        self.channels = channels
        self.out_channels = out_channels or channels
        self.use_conv = use_conv
        self.padding = padding
        self.name = name
        if use_conv:
            conv = nn.Conv2d(self.channels, self.out_channels, kernel_size=kernel_size, stride=2, padding=padding, bias=bias)
        else:
            assert self.channels == self.out_channels
            conv = nn.AvgPool2d(kernel_size=2, stride=2)
        if name == "conv":
            self.Conv2d_0 = conv
            self.conv = conv
        elif name == "Conv2d_0":
            self.conv = conv
        else:
            self.conv = conv

    def forward(self, hidden_states, *args, **kwargs):
        assert hidden_states.shape[1] == self.channels
        if self.use_conv and self.padding == 0:
            hidden_states = F.pad(hidden_states, (0, 1, 0, 1), mode="constant", value=0)
        return self.conv(hidden_states)


class ResnetBlock2D(nn.Module):
    """diffusers ResnetBlock2D ("default" time embedding norm).  The reference's copy model/resnet_block_2d.py:30-221
    is this block plus the ``output_size`` argument forwarded to the up-sampler (:179-184); both behaviours are here."""

    def __init__(self, *, in_channels: int, out_channels: Optional[int] = None, conv_shortcut: bool = False,
                 dropout: float = 0.0, temb_channels: int = 512, groups: int = 32, groups_out: Optional[int] = None,
                 pre_norm: bool = True, eps: float = 1e-6, non_linearity: str = "swish", skip_time_act: bool = False,
                 time_embedding_norm: str = "default", kernel=None, output_scale_factor: float = 1.0,
                 use_in_shortcut: Optional[bool] = None, up: bool = False, down: bool = False,
                 conv_shortcut_bias: bool = True, conv_2d_out_channels: Optional[int] = None):
        super().__init__()
        assert time_embedding_norm == "default" and kernel is None
        self.in_channels = in_channels
        out_channels = in_channels if out_channels is None else out_channels
        self.out_channels = out_channels
        self.up = up
        self.down = down
        self.output_scale_factor = output_scale_factor
        self.skip_time_act = skip_time_act
        if groups_out is None:
            groups_out = groups
        self.norm1 = nn.GroupNorm(num_groups=groups, num_channels=in_channels, eps=eps, affine=True)
        self.conv1 = nn.Conv2d(in_channels, out_channels, kernel_size=3, stride=1, padding=1)
        self.time_emb_proj = nn.Linear(temb_channels, out_channels) if temb_channels is not None else None
        self.norm2 = nn.GroupNorm(num_groups=groups_out, num_channels=out_channels, eps=eps, affine=True)
        self.dropout = nn.Dropout(dropout)
        conv_2d_out_channels = conv_2d_out_channels or out_channels
        self.conv2 = nn.Conv2d(out_channels, conv_2d_out_channels, kernel_size=3, stride=1, padding=1)
        self.nonlinearity = nn.SiLU()
        self.upsample = self.downsample = None
        if self.up:
            self.upsample = Upsample2D(in_channels, use_conv=False)
        elif self.down:
            self.downsample = Downsample2D(in_channels, use_conv=False, padding=1, name="op")
        self.use_in_shortcut = self.in_channels != conv_2d_out_channels if use_in_shortcut is None else use_in_shortcut
        self.conv_shortcut = None
        if self.use_in_shortcut:
            self.conv_shortcut = nn.Conv2d(in_channels, conv_2d_out_channels, kernel_size=1, stride=1, padding=0,
                                           bias=conv_shortcut_bias)

    def forward(self, input_tensor, temb, output_size=None, *args, **kwargs):
        hidden_states = input_tensor
        hidden_states = self.norm1(hidden_states)
        hidden_states = self.nonlinearity(hidden_states)
        if self.upsample is not None:
            if hidden_states.shape[0] >= 64:
                input_tensor = input_tensor.contiguous()
                hidden_states = hidden_states.contiguous()
            if output_size is None:
                input_tensor = self.upsample(input_tensor)
                hidden_states = self.upsample(hidden_states)
            else:
                input_tensor = self.upsample(input_tensor, output_size)
                hidden_states = self.upsample(hidden_states, output_size)
        elif self.downsample is not None:
            input_tensor = self.downsample(input_tensor)
            hidden_states = self.downsample(hidden_states)
        hidden_states = self.conv1(hidden_states)
        if self.time_emb_proj is not None:
            if not self.skip_time_act:
                temb = self.nonlinearity(temb)
            temb = self.time_emb_proj(temb)[:, :, None, None]
        if temb is not None:
            hidden_states = hidden_states + temb
        hidden_states = self.norm2(hidden_states)
        hidden_states = self.nonlinearity(hidden_states)
        hidden_states = self.dropout(hidden_states)
        hidden_states = self.conv2(hidden_states)
        if self.conv_shortcut is not None:
            input_tensor = self.conv_shortcut(input_tensor)
        return (input_tensor + hidden_states) / self.output_scale_factor


class TemporalResnetBlock(nn.Module):
    def __init__(self, in_channels: int, out_channels: Optional[int] = None, temb_channels: int = 512, eps: float = 1e-6):
        super().__init__()
        self.in_channels = in_channels
        out_channels = in_channels if out_channels is None else out_channels
        self.out_channels = out_channels
        kernel_size = (3, 1, 1)
        padding = [k // 2 for k in kernel_size]
        self.norm1 = nn.GroupNorm(num_groups=32, num_channels=in_channels, eps=eps, affine=True)
        self.conv1 = nn.Conv3d(in_channels, out_channels, kernel_size=kernel_size, stride=1, padding=padding)
        self.time_emb_proj = nn.Linear(temb_channels, out_channels) if temb_channels is not None else None
        self.norm2 = nn.GroupNorm(num_groups=32, num_channels=out_channels, eps=eps, affine=True)
        self.dropout = nn.Dropout(0.0)
        self.conv2 = nn.Conv3d(out_channels, out_channels, kernel_size=kernel_size, stride=1, padding=padding)
        self.nonlinearity = nn.SiLU()
        self.use_in_shortcut = self.in_channels != out_channels
        self.conv_shortcut = None
        if self.use_in_shortcut:
            self.conv_shortcut = nn.Conv3d(in_channels, out_channels, kernel_size=1, stride=1, padding=0)

    def forward(self, input_tensor, temb):
        hidden_states = input_tensor
        hidden_states = self.norm1(hidden_states)
        hidden_states = self.nonlinearity(hidden_states)
        hidden_states = self.conv1(hidden_states)
        if self.time_emb_proj is not None:
            temb = self.nonlinearity(temb)
            temb = self.time_emb_proj(temb)[:, :, :, None, None]
            temb = temb.permute(0, 2, 1, 3, 4)
            hidden_states = hidden_states + temb
        hidden_states = self.norm2(hidden_states)
        hidden_states = self.nonlinearity(hidden_states)
        hidden_states = self.dropout(hidden_states)
        hidden_states = self.conv2(hidden_states)
        if self.conv_shortcut is not None:
            input_tensor = self.conv_shortcut(input_tensor)
        return input_tensor + hidden_states


class AlphaBlender(nn.Module):
    strategies = ["learned", "fixed", "learned_with_images"]

    def __init__(self, alpha: float, merge_strategy: str = "learned_with_images",
                 switch_spatial_to_temporal_mix: bool = False):
        super().__init__()
        self.merge_strategy = merge_strategy
        self.switch_spatial_to_temporal_mix = switch_spatial_to_temporal_mix
        assert merge_strategy in self.strategies
        if merge_strategy == "fixed":
            self.register_buffer("mix_factor", torch.Tensor([alpha]))
        else:
            self.register_parameter("mix_factor", nn.Parameter(torch.Tensor([alpha])))

    def get_alpha(self, image_only_indicator, ndims: int):
        if self.merge_strategy == "fixed":
            alpha = self.mix_factor
        elif self.merge_strategy == "learned":
            alpha = torch.sigmoid(self.mix_factor)
        else:
            alpha = torch.where(image_only_indicator.bool(), torch.ones(1, 1, device=image_only_indicator.device),
                                torch.sigmoid(self.mix_factor)[..., None])
            if ndims == 5:
                alpha = alpha[:, None, :, None, None]
            elif ndims == 3:
                alpha = alpha.reshape(-1)[:, None, None]
            else:
                raise ValueError(f"Unexpected ndims {ndims}")
        return alpha

    def forward(self, x_spatial, x_temporal, image_only_indicator=None):
        alpha = self.get_alpha(image_only_indicator, x_spatial.ndim)
        alpha = alpha.to(x_spatial.dtype)
        if self.switch_spatial_to_temporal_mix:
            alpha = 1.0 - alpha
        return alpha * x_spatial + (1.0 - alpha) * x_temporal


# ------------------------------------------------------------------------------------------------
# Transformer2DModel and the 2-D UNet blocks (ControlNet: controlnet/controlnet.py:371-424; SDXL UNet: stock diffusers)
# ------------------------------------------------------------------------------------------------
class Transformer2DModel(nn.Module):
    def __init__(self, num_attention_heads: int = 16, attention_head_dim: int = 88, in_channels: Optional[int] = None,
                 num_layers: int = 1, cross_attention_dim: Optional[int] = None, norm_num_groups: int = 32,
                 use_linear_projection: bool = False, only_cross_attention: bool = False, upcast_attention: bool = False,
                 attention_type: str = "default", **_unused):
        super().__init__()
        self.use_linear_projection = use_linear_projection
        inner_dim = num_attention_heads * attention_head_dim
        self.in_channels = in_channels
        self.norm = nn.GroupNorm(num_groups=norm_num_groups, num_channels=in_channels, eps=1e-6, affine=True)
        if use_linear_projection:
            self.proj_in = nn.Linear(in_channels, inner_dim)
        else:
            self.proj_in = nn.Conv2d(in_channels, inner_dim, kernel_size=1, stride=1, padding=0)
        self.transformer_blocks = nn.ModuleList([
            BasicTransformerBlock(inner_dim, num_attention_heads, attention_head_dim, cross_attention_dim=cross_attention_dim,
                                  only_cross_attention=only_cross_attention, upcast_attention=upcast_attention)
            for _ in range(num_layers)])
        if use_linear_projection:
            self.proj_out = nn.Linear(inner_dim, in_channels)
        else:
            self.proj_out = nn.Conv2d(inner_dim, in_channels, kernel_size=1, stride=1, padding=0)

    def forward(self, hidden_states, encoder_hidden_states=None, **_kw):
        batch, _, height, width = hidden_states.shape
        residual = hidden_states
        hidden_states = self.norm(hidden_states)
        if not self.use_linear_projection:
            hidden_states = self.proj_in(hidden_states)
            inner_dim = hidden_states.shape[1]
            hidden_states = hidden_states.permute(0, 2, 3, 1).reshape(batch, height * width, inner_dim)
        else:
            inner_dim = hidden_states.shape[1]
            hidden_states = hidden_states.permute(0, 2, 3, 1).reshape(batch, height * width, inner_dim)
            hidden_states = self.proj_in(hidden_states)
        for block in self.transformer_blocks:
            hidden_states = block(hidden_states, encoder_hidden_states=encoder_hidden_states)
        if not self.use_linear_projection:
            hidden_states = hidden_states.reshape(batch, height, width, inner_dim).permute(0, 3, 1, 2).contiguous()
            hidden_states = self.proj_out(hidden_states)
        else:
            hidden_states = self.proj_out(hidden_states)
            hidden_states = hidden_states.reshape(batch, height, width, inner_dim).permute(0, 3, 1, 2).contiguous()
        return (hidden_states + residual,)


def _as_list(v, n):
    return list(v) if isinstance(v, (list, tuple)) else [v] * n


class DownBlock2D(nn.Module):
    has_cross_attention = False

    def __init__(self, in_channels: int, out_channels: int, temb_channels: int, num_layers: int = 1,
                 resnet_eps: float = 1e-6, resnet_groups: int = 32, output_scale_factor: float = 1.0,
                 add_downsample: bool = True, downsample_padding: int = 1, **_unused):
        super().__init__()
        self.resnets = nn.ModuleList([
            ResnetBlock2D(in_channels=in_channels if i == 0 else out_channels, out_channels=out_channels,
                          temb_channels=temb_channels, eps=resnet_eps, groups=resnet_groups,
                          output_scale_factor=output_scale_factor) for i in range(num_layers)])
        self.downsamplers = None
        if add_downsample:
            self.downsamplers = nn.ModuleList([Downsample2D(out_channels, use_conv=True, out_channels=out_channels,
                                                            padding=downsample_padding, name="op")])

    def forward(self, hidden_states, temb=None, **_kw):
        output_states = ()
        for resnet in self.resnets:
            hidden_states = resnet(hidden_states, temb)
            output_states = output_states + (hidden_states,)
        if self.downsamplers is not None:
            for d in self.downsamplers:
                hidden_states = d(hidden_states)
            output_states = output_states + (hidden_states,)
        return hidden_states, output_states


class CrossAttnDownBlock2D(nn.Module):
    has_cross_attention = True

    def __init__(self, in_channels: int, out_channels: int, temb_channels: int, num_layers: int = 1,
                 transformer_layers_per_block=1, resnet_eps: float = 1e-6, resnet_groups: int = 32,
                 num_attention_heads: int = 1, cross_attention_dim: int = 1280, output_scale_factor: float = 1.0,
                 downsample_padding: int = 1, add_downsample: bool = True, use_linear_projection: bool = False,
                 only_cross_attention: bool = False, upcast_attention: bool = False, **_unused):
        super().__init__()
        tl = _as_list(transformer_layers_per_block, num_layers)
        self.num_attention_heads = num_attention_heads
        resnets, attentions = [], []
        for i in range(num_layers):
            resnets.append(ResnetBlock2D(in_channels=in_channels if i == 0 else out_channels, out_channels=out_channels,
                                         temb_channels=temb_channels, eps=resnet_eps, groups=resnet_groups,
                                         output_scale_factor=output_scale_factor))
            attentions.append(Transformer2DModel(num_attention_heads, out_channels // num_attention_heads,
                                                 in_channels=out_channels, num_layers=tl[i],
                                                 cross_attention_dim=cross_attention_dim, norm_num_groups=resnet_groups,
                                                 use_linear_projection=use_linear_projection,
                                                 only_cross_attention=only_cross_attention,
                                                 upcast_attention=upcast_attention))
        self.attentions = nn.ModuleList(attentions)
        self.resnets = nn.ModuleList(resnets)
        self.downsamplers = None
        if add_downsample:
            self.downsamplers = nn.ModuleList([Downsample2D(out_channels, use_conv=True, out_channels=out_channels,
                                                            padding=downsample_padding, name="op")])

    def forward(self, hidden_states, temb=None, encoder_hidden_states=None, **_kw):
        output_states = ()
        for resnet, attn in zip(self.resnets, self.attentions):
            hidden_states = resnet(hidden_states, temb)
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states)[0]
            output_states = output_states + (hidden_states,)
        if self.downsamplers is not None:
            for d in self.downsamplers:
                hidden_states = d(hidden_states)
            output_states = output_states + (hidden_states,)
        return hidden_states, output_states


class UNetMidBlock2DCrossAttn(nn.Module):
    has_cross_attention = True

    def __init__(self, in_channels: int, temb_channels: int, num_layers: int = 1, transformer_layers_per_block=1,
                 resnet_eps: float = 1e-6, resnet_groups: int = 32, num_attention_heads: int = 1,
                 output_scale_factor: float = 1.0, cross_attention_dim: int = 1280, use_linear_projection: bool = False,
                 upcast_attention: bool = False, **_unused):
        super().__init__()
        tl = _as_list(transformer_layers_per_block, num_layers)
        resnets = [ResnetBlock2D(in_channels=in_channels, out_channels=in_channels, temb_channels=temb_channels,
                                 eps=resnet_eps, groups=resnet_groups, output_scale_factor=output_scale_factor)]
        attentions = []
        for i in range(num_layers):
            attentions.append(Transformer2DModel(num_attention_heads, in_channels // num_attention_heads,
                                                 in_channels=in_channels, num_layers=tl[i],
                                                 cross_attention_dim=cross_attention_dim, norm_num_groups=resnet_groups,
                                                 use_linear_projection=use_linear_projection,
                                                 upcast_attention=upcast_attention))
            resnets.append(ResnetBlock2D(in_channels=in_channels, out_channels=in_channels, temb_channels=temb_channels,
                                         eps=resnet_eps, groups=resnet_groups, output_scale_factor=output_scale_factor))
        self.attentions = nn.ModuleList(attentions)
        self.resnets = nn.ModuleList(resnets)

    def forward(self, hidden_states, temb=None, encoder_hidden_states=None, **_kw):
        hidden_states = self.resnets[0](hidden_states, temb)
        for attn, resnet in zip(self.attentions, self.resnets[1:]):
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states)[0]
            hidden_states = resnet(hidden_states, temb)
        return hidden_states


class UpBlock2D(nn.Module):
    has_cross_attention = False

    def __init__(self, in_channels: int, prev_output_channel: int, out_channels: int, temb_channels: int,
                 num_layers: int = 1, resnet_eps: float = 1e-6, resnet_groups: int = 32,
                 output_scale_factor: float = 1.0, add_upsample: bool = True, **_unused):
        super().__init__()
        resnets = []
        for i in range(num_layers):
            res_skip_channels = in_channels if (i == num_layers - 1) else out_channels
            resnet_in_channels = prev_output_channel if i == 0 else out_channels
            resnets.append(ResnetBlock2D(in_channels=resnet_in_channels + res_skip_channels, out_channels=out_channels,
                                         temb_channels=temb_channels, eps=resnet_eps, groups=resnet_groups,
                                         output_scale_factor=output_scale_factor))
        self.resnets = nn.ModuleList(resnets)
        self.upsamplers = None
        if add_upsample:
            self.upsamplers = nn.ModuleList([Upsample2D(out_channels, use_conv=True, out_channels=out_channels)])

    def forward(self, hidden_states, res_hidden_states_tuple, temb=None, upsample_size=None, **_kw):
        for resnet in self.resnets:
            res_hidden_states = res_hidden_states_tuple[-1]
            res_hidden_states_tuple = res_hidden_states_tuple[:-1]
            hidden_states = torch.cat([hidden_states, res_hidden_states], dim=1)
            hidden_states = resnet(hidden_states, temb)
        if self.upsamplers is not None:
            for u in self.upsamplers:
                hidden_states = u(hidden_states, upsample_size)
        return hidden_states


class CrossAttnUpBlock2D(nn.Module):
    has_cross_attention = True

    def __init__(self, in_channels: int, out_channels: int, prev_output_channel: int, temb_channels: int,
                 num_layers: int = 1, transformer_layers_per_block=1, resnet_eps: float = 1e-6, resnet_groups: int = 32,
                 num_attention_heads: int = 1, cross_attention_dim: int = 1280, output_scale_factor: float = 1.0,
                 add_upsample: bool = True, use_linear_projection: bool = False, only_cross_attention: bool = False,
                 upcast_attention: bool = False, **_unused):
        super().__init__()
        tl = _as_list(transformer_layers_per_block, num_layers)
        resnets, attentions = [], []
        for i in range(num_layers):
            res_skip_channels = in_channels if (i == num_layers - 1) else out_channels
            resnet_in_channels = prev_output_channel if i == 0 else out_channels
            resnets.append(ResnetBlock2D(in_channels=resnet_in_channels + res_skip_channels, out_channels=out_channels,
                                         temb_channels=temb_channels, eps=resnet_eps, groups=resnet_groups,
                                         output_scale_factor=output_scale_factor))
            attentions.append(Transformer2DModel(num_attention_heads, out_channels // num_attention_heads,
                                                 in_channels=out_channels, num_layers=tl[i],
                                                 cross_attention_dim=cross_attention_dim, norm_num_groups=resnet_groups,
                                                 use_linear_projection=use_linear_projection,
                                                 only_cross_attention=only_cross_attention,
                                                 upcast_attention=upcast_attention))
        self.attentions = nn.ModuleList(attentions)
        self.resnets = nn.ModuleList(resnets)
        self.upsamplers = None
        if add_upsample:
            self.upsamplers = nn.ModuleList([Upsample2D(out_channels, use_conv=True, out_channels=out_channels)])

    def forward(self, hidden_states, res_hidden_states_tuple, temb=None, encoder_hidden_states=None,
                upsample_size=None, **_kw):
        for resnet, attn in zip(self.resnets, self.attentions):
            res_hidden_states = res_hidden_states_tuple[-1]
            res_hidden_states_tuple = res_hidden_states_tuple[:-1]
            hidden_states = torch.cat([hidden_states, res_hidden_states], dim=1)
            hidden_states = resnet(hidden_states, temb)
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states)[0]
        if self.upsamplers is not None:
            for u in self.upsamplers:
                hidden_states = u(hidden_states, upsample_size)
        return hidden_states


def get_down_block(down_block_type: str, num_layers: int, in_channels: int, out_channels: int, temb_channels: int,
                   add_downsample: bool, resnet_eps: float, resnet_act_fn: str = "silu",
                   transformer_layers_per_block=1, num_attention_heads=None, resnet_groups=None,
                   cross_attention_dim=None, downsample_padding=None, use_linear_projection=False,
                   only_cross_attention=False, upcast_attention=False, attention_head_dim=None, **_unused):
    if attention_head_dim is None:
        attention_head_dim = num_attention_heads
    if down_block_type == "DownBlock2D":
        return DownBlock2D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                           temb_channels=temb_channels, add_downsample=add_downsample, resnet_eps=resnet_eps,
                           resnet_groups=resnet_groups, downsample_padding=downsample_padding)
    if down_block_type == "CrossAttnDownBlock2D":
        return CrossAttnDownBlock2D(num_layers=num_layers, transformer_layers_per_block=transformer_layers_per_block,
                                    in_channels=in_channels, out_channels=out_channels, temb_channels=temb_channels,
                                    add_downsample=add_downsample, resnet_eps=resnet_eps, resnet_groups=resnet_groups,
                                    downsample_padding=downsample_padding, cross_attention_dim=cross_attention_dim,
                                    num_attention_heads=num_attention_heads, use_linear_projection=use_linear_projection,
                                    only_cross_attention=only_cross_attention, upcast_attention=upcast_attention)
    raise ValueError(f"{down_block_type} does not exist.")


def get_up_block(up_block_type: str, num_layers: int, in_channels: int, out_channels: int, prev_output_channel: int,
                 temb_channels: int, add_upsample: bool, resnet_eps: float, transformer_layers_per_block=1,
                 num_attention_heads=None, resnet_groups=None, cross_attention_dim=None, use_linear_projection=False,
                 only_cross_attention=False, upcast_attention=False, **_unused):
    if up_block_type == "UpBlock2D":
        return UpBlock2D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                         prev_output_channel=prev_output_channel, temb_channels=temb_channels, add_upsample=add_upsample,
                         resnet_eps=resnet_eps, resnet_groups=resnet_groups)
    if up_block_type == "CrossAttnUpBlock2D":
        return CrossAttnUpBlock2D(num_layers=num_layers, transformer_layers_per_block=transformer_layers_per_block,
                                  in_channels=in_channels, out_channels=out_channels,
                                  prev_output_channel=prev_output_channel, temb_channels=temb_channels,
                                  add_upsample=add_upsample, resnet_eps=resnet_eps, resnet_groups=resnet_groups,
                                  cross_attention_dim=cross_attention_dim, num_attention_heads=num_attention_heads,
                                  use_linear_projection=use_linear_projection, only_cross_attention=only_cross_attention,
                                  upcast_attention=upcast_attention)
    raise ValueError(f"{up_block_type} does not exist.")


# ------------------------------------------------------------------------------------------------
# 3-D (video) blocks of diffusers v0.27.2 used by I2VGenXLUNet
# (reference: /root/reference/i2vgen_xl/models/unets/unet_i2vgen_xl.py:30-38 imports them from
#  diffusers.models.unets.unet_3d_blocks / transformers.transformer_temporal / resnet)
# ------------------------------------------------------------------------------------------------
class GELUProj(nn.Module):
    """diffusers activations.GELU: Linear followed by exact (erf) GELU."""

    def __init__(self, dim_in: int, dim_out: int, bias: bool = True):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out, bias=bias)

    def forward(self, hidden_states):
        return F.gelu(self.proj(hidden_states))


class FeedForwardGELU(nn.Module):
    """FeedForward(activation_fn="gelu", inner_dim=...) as used by I2VGenXLTransformerTemporalEncoder."""

    def __init__(self, dim: int, inner_dim: int, dim_out: Optional[int] = None, bias: bool = True):
        super().__init__()
        dim_out = dim_out if dim_out is not None else dim
        self.net = nn.ModuleList([GELUProj(dim, inner_dim, bias=bias), nn.Dropout(0.0), nn.Linear(inner_dim, dim_out, bias=bias)])

    def forward(self, hidden_states):
        for m in self.net:
            hidden_states = m(hidden_states)
        return hidden_states


class TemporalConvLayer(nn.Module):
    """4 x (GroupNorm -> SiLU -> [Dropout] -> Conv3d (3,1,1)) with identity skip; last conv zero-initialised."""

    def __init__(self, in_dim: int, out_dim: Optional[int] = None, dropout: float = 0.0, norm_num_groups: int = 32):
        super().__init__()
        out_dim = out_dim or in_dim
        self.in_dim, self.out_dim = in_dim, out_dim
        self.conv1 = nn.Sequential(nn.GroupNorm(norm_num_groups, in_dim), nn.SiLU(),
                                   nn.Conv3d(in_dim, out_dim, (3, 1, 1), padding=(1, 0, 0)))
        self.conv2 = nn.Sequential(nn.GroupNorm(norm_num_groups, out_dim), nn.SiLU(), nn.Dropout(dropout),
                                   nn.Conv3d(out_dim, in_dim, (3, 1, 1), padding=(1, 0, 0)))
        self.conv3 = nn.Sequential(nn.GroupNorm(norm_num_groups, out_dim), nn.SiLU(), nn.Dropout(dropout),
                                   nn.Conv3d(out_dim, in_dim, (3, 1, 1), padding=(1, 0, 0)))
        self.conv4 = nn.Sequential(nn.GroupNorm(norm_num_groups, out_dim), nn.SiLU(), nn.Dropout(dropout),
                                   nn.Conv3d(out_dim, in_dim, (3, 1, 1), padding=(1, 0, 0)))
        nn.init.zeros_(self.conv4[-1].weight)
        nn.init.zeros_(self.conv4[-1].bias)

    def forward(self, hidden_states, num_frames: int = 1):
        hidden_states = hidden_states[None, :].reshape((-1, num_frames) + hidden_states.shape[1:]).permute(0, 2, 1, 3, 4)
        identity = hidden_states
        hidden_states = self.conv1(hidden_states)
        hidden_states = self.conv2(hidden_states)
        hidden_states = self.conv3(hidden_states)
        hidden_states = self.conv4(hidden_states)
        hidden_states = identity + hidden_states
        hidden_states = hidden_states.permute(0, 2, 1, 3, 4).reshape(
            (hidden_states.shape[0] * hidden_states.shape[2], -1) + hidden_states.shape[3:])
        return hidden_states


class TransformerTemporalModel(nn.Module):
    """Frame-axis transformer: GroupNorm (5-D statistics) -> proj_in -> BasicTransformerBlock(double self-attention)
    over (batch*h*w, frames, c) -> proj_out -> + residual."""

    def __init__(self, num_attention_heads: int = 16, attention_head_dim: int = 88, in_channels: Optional[int] = None,
                 out_channels: Optional[int] = None, num_layers: int = 1, dropout: float = 0.0, norm_num_groups: int = 32,
                 cross_attention_dim: Optional[int] = None, attention_bias: bool = False,
                 double_self_attention: bool = True, **_unused):
        super().__init__()
        inner_dim = num_attention_heads * attention_head_dim
        self.in_channels = in_channels
        self.norm = nn.GroupNorm(num_groups=norm_num_groups, num_channels=in_channels, eps=1e-6, affine=True)
        self.proj_in = nn.Linear(in_channels, inner_dim)
        self.transformer_blocks = nn.ModuleList([
            BasicTransformerBlock(inner_dim, num_attention_heads, attention_head_dim, dropout=dropout,
                                  cross_attention_dim=cross_attention_dim, attention_bias=attention_bias,
                                  double_self_attention=double_self_attention) for _ in range(num_layers)])
        self.proj_out = nn.Linear(inner_dim, in_channels)

    def forward(self, hidden_states, encoder_hidden_states=None, num_frames: int = 1, **_kw):
        batch_frames, channel, height, width = hidden_states.shape
        batch_size = batch_frames // num_frames
        residual = hidden_states
        hidden_states = hidden_states[None, :].reshape(batch_size, num_frames, channel, height, width)
        hidden_states = hidden_states.permute(0, 2, 1, 3, 4)
        hidden_states = self.norm(hidden_states)
        hidden_states = hidden_states.permute(0, 3, 4, 2, 1).reshape(batch_size * height * width, num_frames, channel)
        hidden_states = self.proj_in(hidden_states)
        for block in self.transformer_blocks:
            hidden_states = block(hidden_states, encoder_hidden_states=encoder_hidden_states)
        hidden_states = self.proj_out(hidden_states)
        hidden_states = (hidden_states[None, None, :].reshape(batch_size, height, width, num_frames, channel)
                         .permute(0, 3, 4, 1, 2).contiguous())
        hidden_states = hidden_states.reshape(batch_frames, channel, height, width)
        return (hidden_states + residual,)


class DownBlock3D(nn.Module):
    has_cross_attention = False

    def __init__(self, in_channels, out_channels, temb_channels, num_layers=1, resnet_eps=1e-6, resnet_groups=32,
                 output_scale_factor=1.0, add_downsample=True, downsample_padding=1, **_unused):
        super().__init__()
        self.resnets = nn.ModuleList([ResnetBlock2D(in_channels=in_channels if i == 0 else out_channels,
                                                    out_channels=out_channels, temb_channels=temb_channels,
                                                    eps=resnet_eps, groups=resnet_groups,
                                                    output_scale_factor=output_scale_factor) for i in range(num_layers)])
        self.temp_convs = nn.ModuleList([TemporalConvLayer(out_channels, out_channels, dropout=0.1,
                                                           norm_num_groups=resnet_groups) for _ in range(num_layers)])
        self.downsamplers = None
        if add_downsample:
            self.downsamplers = nn.ModuleList([Downsample2D(out_channels, use_conv=True, out_channels=out_channels,
                                                            padding=downsample_padding, name="op")])

    def forward(self, hidden_states, temb=None, num_frames=1, **_kw):
        output_states = ()
        for resnet, temp_conv in zip(self.resnets, self.temp_convs):
            hidden_states = resnet(hidden_states, temb)
            hidden_states = temp_conv(hidden_states, num_frames=num_frames)
            output_states += (hidden_states,)
        if self.downsamplers is not None:
            for d in self.downsamplers:
                hidden_states = d(hidden_states)
            output_states += (hidden_states,)
        return hidden_states, output_states


class CrossAttnDownBlock3D(nn.Module):
    has_cross_attention = True

    def __init__(self, in_channels, out_channels, temb_channels, num_layers=1, resnet_eps=1e-6, resnet_groups=32,
                 num_attention_heads=1, cross_attention_dim=1280, output_scale_factor=1.0, downsample_padding=1,
                 add_downsample=True, use_linear_projection=False, only_cross_attention=False, upcast_attention=False,
                 **_unused):
        super().__init__()
        self.num_attention_heads = num_attention_heads
        resnets, temp_convs, attentions, temp_attentions = [], [], [], []
        for i in range(num_layers):
            resnets.append(ResnetBlock2D(in_channels=in_channels if i == 0 else out_channels, out_channels=out_channels,
                                         temb_channels=temb_channels, eps=resnet_eps, groups=resnet_groups,
                                         output_scale_factor=output_scale_factor))
            temp_convs.append(TemporalConvLayer(out_channels, out_channels, dropout=0.1, norm_num_groups=resnet_groups))
            # NB positional order (heads, head_dim) = (out_channels // num_attention_heads, num_attention_heads)
            attentions.append(Transformer2DModel(out_channels // num_attention_heads, num_attention_heads,
                                                 in_channels=out_channels, num_layers=1,
                                                 cross_attention_dim=cross_attention_dim, norm_num_groups=resnet_groups,
                                                 use_linear_projection=use_linear_projection,
                                                 only_cross_attention=only_cross_attention,
                                                 upcast_attention=upcast_attention))
            temp_attentions.append(TransformerTemporalModel(out_channels // num_attention_heads, num_attention_heads,
                                                            in_channels=out_channels, num_layers=1,
                                                            cross_attention_dim=cross_attention_dim,
                                                            norm_num_groups=resnet_groups))
        self.resnets = nn.ModuleList(resnets)
        self.temp_convs = nn.ModuleList(temp_convs)
        self.attentions = nn.ModuleList(attentions)
        self.temp_attentions = nn.ModuleList(temp_attentions)
        self.downsamplers = None
        if add_downsample:
            self.downsamplers = nn.ModuleList([Downsample2D(out_channels, use_conv=True, out_channels=out_channels,
                                                            padding=downsample_padding, name="op")])

    def forward(self, hidden_states, temb=None, encoder_hidden_states=None, num_frames=1, **_kw):
        output_states = ()
        for resnet, temp_conv, attn, temp_attn in zip(self.resnets, self.temp_convs, self.attentions, self.temp_attentions):
            hidden_states = resnet(hidden_states, temb)
            hidden_states = temp_conv(hidden_states, num_frames=num_frames)
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states)[0]
            hidden_states = temp_attn(hidden_states, num_frames=num_frames)[0]
            output_states += (hidden_states,)
        if self.downsamplers is not None:
            for d in self.downsamplers:
                hidden_states = d(hidden_states)
            output_states += (hidden_states,)
        return hidden_states, output_states


class UNetMidBlock3DCrossAttn(nn.Module):
    has_cross_attention = True

    def __init__(self, in_channels, temb_channels, num_layers=1, resnet_eps=1e-6, resnet_groups=32,
                 num_attention_heads=1, output_scale_factor=1.0, cross_attention_dim=1280, use_linear_projection=True,
                 upcast_attention=False, **_unused):
        super().__init__()
        resnets = [ResnetBlock2D(in_channels=in_channels, out_channels=in_channels, temb_channels=temb_channels,
                                 eps=resnet_eps, groups=resnet_groups, output_scale_factor=output_scale_factor)]
        temp_convs = [TemporalConvLayer(in_channels, in_channels, dropout=0.1, norm_num_groups=resnet_groups)]
        attentions, temp_attentions = [], []
        for _ in range(num_layers):
            attentions.append(Transformer2DModel(in_channels // num_attention_heads, num_attention_heads,
                                                 in_channels=in_channels, num_layers=1,
                                                 cross_attention_dim=cross_attention_dim, norm_num_groups=resnet_groups,
                                                 use_linear_projection=use_linear_projection,
                                                 upcast_attention=upcast_attention))
            temp_attentions.append(TransformerTemporalModel(in_channels // num_attention_heads, num_attention_heads,
                                                            in_channels=in_channels, num_layers=1,
                                                            cross_attention_dim=cross_attention_dim,
                                                            norm_num_groups=resnet_groups))
            resnets.append(ResnetBlock2D(in_channels=in_channels, out_channels=in_channels, temb_channels=temb_channels,
                                         eps=resnet_eps, groups=resnet_groups, output_scale_factor=output_scale_factor))
            temp_convs.append(TemporalConvLayer(in_channels, in_channels, dropout=0.1, norm_num_groups=resnet_groups))
        self.resnets = nn.ModuleList(resnets)
        self.temp_convs = nn.ModuleList(temp_convs)
        self.attentions = nn.ModuleList(attentions)
        self.temp_attentions = nn.ModuleList(temp_attentions)

    def forward(self, hidden_states, temb=None, encoder_hidden_states=None, num_frames=1, **_kw):
        hidden_states = self.resnets[0](hidden_states, temb)
        hidden_states = self.temp_convs[0](hidden_states, num_frames=num_frames)
        for attn, temp_attn, resnet, temp_conv in zip(self.attentions, self.temp_attentions, self.resnets[1:],
                                                      self.temp_convs[1:]):
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states)[0]
            hidden_states = temp_attn(hidden_states, num_frames=num_frames)[0]
            hidden_states = resnet(hidden_states, temb)
            hidden_states = temp_conv(hidden_states, num_frames=num_frames)
        return hidden_states


class UpBlock3D(nn.Module):
    has_cross_attention = False

    def __init__(self, in_channels, prev_output_channel, out_channels, temb_channels, num_layers=1, resnet_eps=1e-6,
                 resnet_groups=32, output_scale_factor=1.0, add_upsample=True, **_unused):
        super().__init__()
        resnets, temp_convs = [], []
        for i in range(num_layers):
            res_skip_channels = in_channels if (i == num_layers - 1) else out_channels
            resnet_in_channels = prev_output_channel if i == 0 else out_channels
            resnets.append(ResnetBlock2D(in_channels=resnet_in_channels + res_skip_channels, out_channels=out_channels,
                                         temb_channels=temb_channels, eps=resnet_eps, groups=resnet_groups,
                                         output_scale_factor=output_scale_factor))
            temp_convs.append(TemporalConvLayer(out_channels, out_channels, dropout=0.1, norm_num_groups=resnet_groups))
        self.resnets = nn.ModuleList(resnets)
        self.temp_convs = nn.ModuleList(temp_convs)
        self.upsamplers = None
        if add_upsample:
            self.upsamplers = nn.ModuleList([Upsample2D(out_channels, use_conv=True, out_channels=out_channels)])

    def forward(self, hidden_states, res_hidden_states_tuple, temb=None, upsample_size=None, num_frames=1, **_kw):
        for resnet, temp_conv in zip(self.resnets, self.temp_convs):
            res_hidden_states = res_hidden_states_tuple[-1]
            res_hidden_states_tuple = res_hidden_states_tuple[:-1]
            hidden_states = torch.cat([hidden_states, res_hidden_states], dim=1)
            hidden_states = resnet(hidden_states, temb)
            hidden_states = temp_conv(hidden_states, num_frames=num_frames)
        if self.upsamplers is not None:
            for u in self.upsamplers:
                hidden_states = u(hidden_states, upsample_size)
        return hidden_states


class CrossAttnUpBlock3D(nn.Module):
    has_cross_attention = True

    def __init__(self, in_channels, out_channels, prev_output_channel, temb_channels, num_layers=1, resnet_eps=1e-6,
                 resnet_groups=32, num_attention_heads=1, cross_attention_dim=1280, output_scale_factor=1.0,
                 add_upsample=True, use_linear_projection=False, only_cross_attention=False, upcast_attention=False,
                 **_unused):
        super().__init__()
        resnets, temp_convs, attentions, temp_attentions = [], [], [], []
        for i in range(num_layers):
            res_skip_channels = in_channels if (i == num_layers - 1) else out_channels
            resnet_in_channels = prev_output_channel if i == 0 else out_channels
            resnets.append(ResnetBlock2D(in_channels=resnet_in_channels + res_skip_channels, out_channels=out_channels,
                                         temb_channels=temb_channels, eps=resnet_eps, groups=resnet_groups,
                                         output_scale_factor=output_scale_factor))
            temp_convs.append(TemporalConvLayer(out_channels, out_channels, dropout=0.1, norm_num_groups=resnet_groups))
            attentions.append(Transformer2DModel(out_channels // num_attention_heads, num_attention_heads,
                                                 in_channels=out_channels, num_layers=1,
                                                 cross_attention_dim=cross_attention_dim, norm_num_groups=resnet_groups,
                                                 use_linear_projection=use_linear_projection,
                                                 only_cross_attention=only_cross_attention,
                                                 upcast_attention=upcast_attention))
            temp_attentions.append(TransformerTemporalModel(out_channels // num_attention_heads, num_attention_heads,
                                                            in_channels=out_channels, num_layers=1,
                                                            cross_attention_dim=cross_attention_dim,
                                                            norm_num_groups=resnet_groups))
        self.resnets = nn.ModuleList(resnets)
        self.temp_convs = nn.ModuleList(temp_convs)
        self.attentions = nn.ModuleList(attentions)
        self.temp_attentions = nn.ModuleList(temp_attentions)
        self.upsamplers = None
        if add_upsample:
            self.upsamplers = nn.ModuleList([Upsample2D(out_channels, use_conv=True, out_channels=out_channels)])

    def forward(self, hidden_states, res_hidden_states_tuple, temb=None, encoder_hidden_states=None,
                upsample_size=None, num_frames=1, **_kw):
        for resnet, temp_conv, attn, temp_attn in zip(self.resnets, self.temp_convs, self.attentions, self.temp_attentions):
            res_hidden_states = res_hidden_states_tuple[-1]
            res_hidden_states_tuple = res_hidden_states_tuple[:-1]
            hidden_states = torch.cat([hidden_states, res_hidden_states], dim=1)
            hidden_states = resnet(hidden_states, temb)
            hidden_states = temp_conv(hidden_states, num_frames=num_frames)
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states)[0]
            hidden_states = temp_attn(hidden_states, num_frames=num_frames)[0]
        if self.upsamplers is not None:
            for u in self.upsamplers:
                hidden_states = u(hidden_states, upsample_size)
        return hidden_states


def get_down_block_3d(down_block_type, num_layers, in_channels, out_channels, temb_channels, add_downsample, resnet_eps,
                      resnet_act_fn="silu", num_attention_heads=None, resnet_groups=None, cross_attention_dim=None,
                      downsample_padding=None, dual_cross_attention=False, use_linear_projection=True,
                      only_cross_attention=False, upcast_attention=False, **_unused):
    """unet_3d_blocks.get_down_block (note the 3-D default use_linear_projection=True)."""
    if down_block_type == "DownBlock3D":
        return DownBlock3D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                           temb_channels=temb_channels, add_downsample=add_downsample, resnet_eps=resnet_eps,
                           resnet_groups=resnet_groups, downsample_padding=downsample_padding)
    if down_block_type == "CrossAttnDownBlock3D":
        return CrossAttnDownBlock3D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                                    temb_channels=temb_channels, add_downsample=add_downsample, resnet_eps=resnet_eps,
                                    resnet_groups=resnet_groups, downsample_padding=downsample_padding,
                                    cross_attention_dim=cross_attention_dim, num_attention_heads=num_attention_heads,
                                    use_linear_projection=use_linear_projection,
                                    only_cross_attention=only_cross_attention, upcast_attention=upcast_attention)
    raise ValueError(f"{down_block_type} does not exist.")


def get_up_block_3d(up_block_type, num_layers, in_channels, out_channels, prev_output_channel, temb_channels,
                    add_upsample, resnet_eps, resnet_act_fn="silu", num_attention_heads=None, resnet_groups=None,
                    cross_attention_dim=None, dual_cross_attention=False, use_linear_projection=True,
                    only_cross_attention=False, upcast_attention=False, **_unused):
    if up_block_type == "UpBlock3D":
        return UpBlock3D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                         prev_output_channel=prev_output_channel, temb_channels=temb_channels, add_upsample=add_upsample,
                         resnet_eps=resnet_eps, resnet_groups=resnet_groups)
    if up_block_type == "CrossAttnUpBlock3D":
        return CrossAttnUpBlock3D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                                  prev_output_channel=prev_output_channel, temb_channels=temb_channels,
                                  add_upsample=add_upsample, resnet_eps=resnet_eps, resnet_groups=resnet_groups,
                                  cross_attention_dim=cross_attention_dim, num_attention_heads=num_attention_heads,
                                  use_linear_projection=use_linear_projection,
                                  only_cross_attention=only_cross_attention, upcast_attention=upcast_attention)
    raise ValueError(f"{up_block_type} does not exist.")


# ------------------------------------------------------------------------------------------------
# Spatio-temporal (Stable Video Diffusion) blocks: diffusers v0.27.2 models/resnet.py::SpatioTemporalResBlock,
# models/transformers/transformer_temporal.py::TransformerSpatioTemporalModel and the *SpatioTemporal blocks of
# models/unets/unet_3d_blocks.py, reached from svd/models/unets/unet_spatio_temporal_condition.py:13,168-235.
# Restated from the published v0.27.2 semantics (diffusers is not vendored by the reference): parity unpinned for this
# layer, like the rest of this file.  The eps defaults below are the class defaults of that release -- get_down_block /
# get_up_block do NOT forward the resnet_eps the UNet passes (unet_spatio_temporal_condition.py:176, 229).
# ------------------------------------------------------------------------------------------------
class SpatioTemporalResBlock(nn.Module):
    def __init__(self, in_channels: int, out_channels: Optional[int] = None, temb_channels: int = 512, eps: float = 1e-6,
                 temporal_eps: Optional[float] = None, merge_factor: float = 0.5,
                 merge_strategy: str = "learned_with_images", switch_spatial_to_temporal_mix: bool = False):
        super().__init__()
        self.spatial_res_block = ResnetBlock2D(in_channels=in_channels, out_channels=out_channels,
                                               temb_channels=temb_channels, eps=eps)
        mid = out_channels if out_channels is not None else in_channels
        self.temporal_res_block = TemporalResnetBlock(in_channels=mid, out_channels=mid, temb_channels=temb_channels,
                                                      eps=temporal_eps if temporal_eps is not None else eps)
        self.time_mixer = AlphaBlender(alpha=merge_factor, merge_strategy=merge_strategy,
                                       switch_spatial_to_temporal_mix=switch_spatial_to_temporal_mix)

    def forward(self, hidden_states, temb=None, image_only_indicator=None):
        num_frames = image_only_indicator.shape[-1]
        hidden_states = self.spatial_res_block(hidden_states, temb)
        batch_frames, channels, height, width = hidden_states.shape
        batch_size = batch_frames // num_frames
        hidden_states_mix = (hidden_states[None, :].reshape(batch_size, num_frames, channels, height, width)
                             .permute(0, 2, 1, 3, 4))
        hidden_states = (hidden_states[None, :].reshape(batch_size, num_frames, channels, height, width)
                         .permute(0, 2, 1, 3, 4))
        if temb is not None:
            temb = temb.reshape(batch_size, num_frames, -1)
        hidden_states = self.temporal_res_block(hidden_states, temb)
        hidden_states = self.time_mixer(x_spatial=hidden_states_mix, x_temporal=hidden_states,
                                        image_only_indicator=image_only_indicator)
        return hidden_states.permute(0, 2, 1, 3, 4).reshape(batch_frames, channels, height, width)


class TransformerSpatioTemporalModel(nn.Module):
    def __init__(self, num_attention_heads: int = 16, attention_head_dim: int = 88, in_channels: int = 320,
                 out_channels: Optional[int] = None, num_layers: int = 1, cross_attention_dim: Optional[int] = None):
        super().__init__()
        self.num_attention_heads = num_attention_heads
        self.attention_head_dim = attention_head_dim
        inner_dim = num_attention_heads * attention_head_dim
        self.inner_dim = inner_dim
        self.in_channels = in_channels
        self.norm = nn.GroupNorm(num_groups=32, num_channels=in_channels, eps=1e-6)
        self.proj_in = nn.Linear(in_channels, inner_dim)
        self.transformer_blocks = nn.ModuleList([
            BasicTransformerBlock(inner_dim, num_attention_heads, attention_head_dim, cross_attention_dim=cross_attention_dim)
            for _ in range(num_layers)])
        self.temporal_transformer_blocks = nn.ModuleList([
            TemporalBasicTransformerBlock(inner_dim, inner_dim, num_attention_heads, attention_head_dim,
                                          cross_attention_dim=cross_attention_dim)
            for _ in range(num_layers)])
        time_embed_dim = in_channels * 4
        self.time_pos_embed = TimestepEmbedding(in_channels, time_embed_dim, out_dim=in_channels)
        self.time_proj = Timesteps(in_channels, True, 0)
        self.time_mixer = AlphaBlender(alpha=0.5, merge_strategy="learned_with_images")
        self.out_channels = in_channels if out_channels is None else out_channels
        self.proj_out = nn.Linear(inner_dim, in_channels)

    def forward(self, hidden_states, encoder_hidden_states=None, image_only_indicator=None, return_dict: bool = False):
        batch_frames, _, height, width = hidden_states.shape
        num_frames = image_only_indicator.shape[-1]
        batch_size = batch_frames // num_frames
        time_context = encoder_hidden_states
        time_context_first_timestep = time_context[None, :].reshape(batch_size, num_frames, -1, time_context.shape[-1])[:, 0]
        time_context = time_context_first_timestep[None, :].broadcast_to(height * width, batch_size, 1, time_context.shape[-1])
        time_context = time_context.reshape(height * width * batch_size, 1, time_context.shape[-1])

        residual = hidden_states
        hidden_states = self.norm(hidden_states)
        inner_dim = hidden_states.shape[1]
        hidden_states = hidden_states.permute(0, 2, 3, 1).reshape(batch_frames, height * width, inner_dim)
        hidden_states = self.proj_in(hidden_states)

        num_frames_emb = torch.arange(num_frames, device=hidden_states.device)
        num_frames_emb = num_frames_emb.repeat(batch_size, 1).reshape(-1)
        t_emb = self.time_proj(num_frames_emb).to(dtype=hidden_states.dtype)
        emb = self.time_pos_embed(t_emb)[:, None, :]

        for block, temporal_block in zip(self.transformer_blocks, self.temporal_transformer_blocks):
            hidden_states = block(hidden_states, encoder_hidden_states=encoder_hidden_states)
            hidden_states_mix = hidden_states + emb
            hidden_states_mix = temporal_block(hidden_states_mix, num_frames=num_frames, encoder_hidden_states=time_context)
            hidden_states = self.time_mixer(x_spatial=hidden_states, x_temporal=hidden_states_mix,
                                            image_only_indicator=image_only_indicator)

        hidden_states = self.proj_out(hidden_states)
        hidden_states = hidden_states.reshape(batch_frames, height, width, inner_dim).permute(0, 3, 1, 2).contiguous()
        output = hidden_states + residual
        return (output,)


class DownBlockSpatioTemporal(nn.Module):
    has_cross_attention = False

    def __init__(self, in_channels: int, out_channels: int, temb_channels: int, num_layers: int = 1,
                 add_downsample: bool = True):
        super().__init__()
        self.resnets = nn.ModuleList([
            SpatioTemporalResBlock(in_channels=in_channels if i == 0 else out_channels, out_channels=out_channels,
                                   temb_channels=temb_channels, eps=1e-5)
            for i in range(num_layers)])
        self.downsamplers = (nn.ModuleList([Downsample2D(out_channels, use_conv=True, out_channels=out_channels, name="op")])
                             if add_downsample else None)

    def forward(self, hidden_states, temb=None, image_only_indicator=None):
        output_states = ()
        for resnet in self.resnets:
            hidden_states = resnet(hidden_states, temb, image_only_indicator=image_only_indicator)
            output_states = output_states + (hidden_states,)
        if self.downsamplers is not None:
            for downsampler in self.downsamplers:
                hidden_states = downsampler(hidden_states)
            output_states = output_states + (hidden_states,)
        return hidden_states, output_states


class CrossAttnDownBlockSpatioTemporal(nn.Module):
    has_cross_attention = True

    def __init__(self, in_channels: int, out_channels: int, temb_channels: int, num_layers: int = 1,
                 transformer_layers_per_block=1, num_attention_heads: int = 1, cross_attention_dim: int = 1280,
                 add_downsample: bool = True):
        super().__init__()
        self.num_attention_heads = num_attention_heads
        tl = _as_list(transformer_layers_per_block, num_layers)
        self.resnets = nn.ModuleList([
            SpatioTemporalResBlock(in_channels=in_channels if i == 0 else out_channels, out_channels=out_channels,
                                   temb_channels=temb_channels, eps=1e-6)
            for i in range(num_layers)])
        self.attentions = nn.ModuleList([
            TransformerSpatioTemporalModel(num_attention_heads, out_channels // num_attention_heads,
                                           in_channels=out_channels, num_layers=tl[i],
                                           cross_attention_dim=cross_attention_dim)
            for i in range(num_layers)])
        self.downsamplers = (nn.ModuleList([Downsample2D(out_channels, use_conv=True, out_channels=out_channels,
                                                         padding=1, name="op")]) if add_downsample else None)

    def forward(self, hidden_states, temb=None, encoder_hidden_states=None, image_only_indicator=None):
        output_states = ()
        for resnet, attn in zip(self.resnets, self.attentions):
            hidden_states = resnet(hidden_states, temb, image_only_indicator=image_only_indicator)
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states,
                                 image_only_indicator=image_only_indicator, return_dict=False)[0]
            output_states = output_states + (hidden_states,)
        if self.downsamplers is not None:
            for downsampler in self.downsamplers:
                hidden_states = downsampler(hidden_states)
            output_states = output_states + (hidden_states,)
        return hidden_states, output_states


class UNetMidBlockSpatioTemporal(nn.Module):
    has_cross_attention = True

    def __init__(self, in_channels: int, temb_channels: int, num_layers: int = 1, transformer_layers_per_block=1,
                 num_attention_heads: int = 1, cross_attention_dim: int = 1280):
        super().__init__()
        self.num_attention_heads = num_attention_heads
        tl = _as_list(transformer_layers_per_block, num_layers)
        resnets = [SpatioTemporalResBlock(in_channels=in_channels, out_channels=in_channels, temb_channels=temb_channels,
                                          eps=1e-5)]
        attentions = []
        for i in range(num_layers):
            attentions.append(TransformerSpatioTemporalModel(num_attention_heads, in_channels // num_attention_heads,
                                                             in_channels=in_channels, num_layers=tl[i],
                                                             cross_attention_dim=cross_attention_dim))
            resnets.append(SpatioTemporalResBlock(in_channels=in_channels, out_channels=in_channels,
                                                  temb_channels=temb_channels, eps=1e-5))
        self.attentions = nn.ModuleList(attentions)
        self.resnets = nn.ModuleList(resnets)

    def forward(self, hidden_states, temb=None, encoder_hidden_states=None, image_only_indicator=None):
        hidden_states = self.resnets[0](hidden_states, temb, image_only_indicator=image_only_indicator)
        for attn, resnet in zip(self.attentions, self.resnets[1:]):
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states,
                                 image_only_indicator=image_only_indicator, return_dict=False)[0]
            hidden_states = resnet(hidden_states, temb, image_only_indicator=image_only_indicator)
        return hidden_states


class UpBlockSpatioTemporal(nn.Module):
    has_cross_attention = False

    def __init__(self, in_channels: int, prev_output_channel: int, out_channels: int, temb_channels: int,
                 resolution_idx: Optional[int] = None, num_layers: int = 1, resnet_eps: float = 1e-6,
                 add_upsample: bool = True):
        super().__init__()
        resnets = []
        for i in range(num_layers):
            res_skip_channels = in_channels if (i == num_layers - 1) else out_channels
            resnet_in_channels = prev_output_channel if i == 0 else out_channels
            resnets.append(SpatioTemporalResBlock(in_channels=resnet_in_channels + res_skip_channels,
                                                  out_channels=out_channels, temb_channels=temb_channels, eps=resnet_eps))
        self.resnets = nn.ModuleList(resnets)
        self.upsamplers = (nn.ModuleList([Upsample2D(out_channels, use_conv=True, out_channels=out_channels)])
                           if add_upsample else None)
        self.resolution_idx = resolution_idx

    def forward(self, hidden_states, res_hidden_states_tuple, temb=None, image_only_indicator=None):
        for resnet in self.resnets:
            res_hidden_states = res_hidden_states_tuple[-1]
            res_hidden_states_tuple = res_hidden_states_tuple[:-1]
            hidden_states = torch.cat([hidden_states, res_hidden_states], dim=1)
            hidden_states = resnet(hidden_states, temb, image_only_indicator=image_only_indicator)
        if self.upsamplers is not None:
            for upsampler in self.upsamplers:
                hidden_states = upsampler(hidden_states)
        return hidden_states


class CrossAttnUpBlockSpatioTemporal(nn.Module):
    has_cross_attention = True

    def __init__(self, in_channels: int, out_channels: int, prev_output_channel: int, temb_channels: int,
                 resolution_idx: Optional[int] = None, num_layers: int = 1, transformer_layers_per_block=1,
                 resnet_eps: float = 1e-6, num_attention_heads: int = 1, cross_attention_dim: int = 1280,
                 add_upsample: bool = True):
        super().__init__()
        self.num_attention_heads = num_attention_heads
        tl = _as_list(transformer_layers_per_block, num_layers)
        resnets, attentions = [], []
        for i in range(num_layers):
            res_skip_channels = in_channels if (i == num_layers - 1) else out_channels
            resnet_in_channels = prev_output_channel if i == 0 else out_channels
            resnets.append(SpatioTemporalResBlock(in_channels=resnet_in_channels + res_skip_channels,
                                                  out_channels=out_channels, temb_channels=temb_channels, eps=resnet_eps))
            attentions.append(TransformerSpatioTemporalModel(num_attention_heads, out_channels // num_attention_heads,
                                                             in_channels=out_channels, num_layers=tl[i],
                                                             cross_attention_dim=cross_attention_dim))
        self.attentions = nn.ModuleList(attentions)
        self.resnets = nn.ModuleList(resnets)
        self.upsamplers = (nn.ModuleList([Upsample2D(out_channels, use_conv=True, out_channels=out_channels)])
                           if add_upsample else None)
        self.resolution_idx = resolution_idx

    def forward(self, hidden_states, res_hidden_states_tuple, temb=None, encoder_hidden_states=None,
                image_only_indicator=None):
        for resnet, attn in zip(self.resnets, self.attentions):
            res_hidden_states = res_hidden_states_tuple[-1]
            res_hidden_states_tuple = res_hidden_states_tuple[:-1]
            hidden_states = torch.cat([hidden_states, res_hidden_states], dim=1)
            hidden_states = resnet(hidden_states, temb, image_only_indicator=image_only_indicator)
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states,
                                 image_only_indicator=image_only_indicator, return_dict=False)[0]
        if self.upsamplers is not None:
            for upsampler in self.upsamplers:
                hidden_states = upsampler(hidden_states)
        return hidden_states


_get_down_block_3d_base = get_down_block_3d
_get_up_block_3d_base = get_up_block_3d


def get_down_block_3d(down_block_type, num_layers, in_channels, out_channels, temb_channels, add_downsample,  # noqa: F811
                      resnet_eps=None, transformer_layers_per_block=1, cross_attention_dim=None,
                      num_attention_heads=None, **kw):
    """unet_3d_blocks.get_down_block including the spatio-temporal (SVD) types, which ignore resnet_eps."""
    if down_block_type == "DownBlockSpatioTemporal":
        return DownBlockSpatioTemporal(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                                       temb_channels=temb_channels, add_downsample=add_downsample)
    if down_block_type == "CrossAttnDownBlockSpatioTemporal":
        return CrossAttnDownBlockSpatioTemporal(in_channels=in_channels, out_channels=out_channels,
                                                temb_channels=temb_channels, num_layers=num_layers,
                                                transformer_layers_per_block=transformer_layers_per_block,
                                                add_downsample=add_downsample, cross_attention_dim=cross_attention_dim,
                                                num_attention_heads=num_attention_heads)
    return _get_down_block_3d_base(down_block_type, num_layers, in_channels, out_channels, temb_channels, add_downsample,
                                   resnet_eps, cross_attention_dim=cross_attention_dim,
                                   num_attention_heads=num_attention_heads, **kw)


def get_up_block_3d(up_block_type, num_layers, in_channels, out_channels, prev_output_channel, temb_channels,  # noqa: F811
                    add_upsample, resnet_eps=None, transformer_layers_per_block=1, resolution_idx=None,
                    cross_attention_dim=None, num_attention_heads=None, **kw):
    if up_block_type == "UpBlockSpatioTemporal":
        return UpBlockSpatioTemporal(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                                     prev_output_channel=prev_output_channel, temb_channels=temb_channels,
                                     resolution_idx=resolution_idx, add_upsample=add_upsample)
    if up_block_type == "CrossAttnUpBlockSpatioTemporal":
        return CrossAttnUpBlockSpatioTemporal(in_channels=in_channels, out_channels=out_channels,
                                              prev_output_channel=prev_output_channel, temb_channels=temb_channels,
                                              resolution_idx=resolution_idx, num_layers=num_layers,
                                              transformer_layers_per_block=transformer_layers_per_block,
                                              add_upsample=add_upsample, cross_attention_dim=cross_attention_dim,
                                              num_attention_heads=num_attention_heads)
    return _get_up_block_3d_base(up_block_type, num_layers, in_channels, out_channels, prev_output_channel, temb_channels,
                                 add_upsample, resnet_eps, cross_attention_dim=cross_attention_dim,
                                 num_attention_heads=num_attention_heads, **kw)
