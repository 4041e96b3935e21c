"""CPU/torch restatement of the Qwen-Image rollout path (TEST INFRASTRUCTURE - see oracle/__init__.py).

SURVEY.md section 8(f) "next" row 4 / BASELINE config 5.  Groundwork only: there is no native engine for this model yet; the oracle
is pinned against the imported reference (tests/golden/make_golden.py -> tests/golden/qwen_tiny.pt) so that the engine of a later
round starts from a checked specification.  Paths relative to /root/reference: FF = src/flow_factory ; DF = diffusers/src/diffusers.
Same convention as the other oracles: the reference's torch ops in the reference's order.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

from .sd3_oracle import _ff, _layer_norm, _linear, _rms_norm


# ----------------------------------------------------------------------------------------------
# Model config (DF/models/transformers/transformer_qwenimage.py:797-811 register_to_config arguments)
# ----------------------------------------------------------------------------------------------
@dataclass
class QwenImageConfig:
    patch_size: int = 2
    in_channels: int = 64
    out_channels: int = 16
    num_layers: int = 60
    attention_head_dim: int = 128
    num_attention_heads: int = 24
    joint_attention_dim: int = 3584
    axes_dims_rope: Tuple[int, int, int] = (16, 56, 56)

    @property
    def inner_dim(self) -> int:
        return self.num_attention_heads * self.attention_head_dim

    def ref_kwargs(self) -> dict:
        return dict(patch_size=self.patch_size, in_channels=self.in_channels, out_channels=self.out_channels,
                    num_layers=self.num_layers, attention_head_dim=self.attention_head_dim,
                    num_attention_heads=self.num_attention_heads, joint_attention_dim=self.joint_attention_dim,
                    axes_dims_rope=tuple(self.axes_dims_rope))


def qwen_image_20b() -> QwenImageConfig:
    return QwenImageConfig()


def tiny_qwen_config(num_layers: int = 2, heads: int = 2, joint_dim: int = 64) -> QwenImageConfig:
    return QwenImageConfig(num_layers=num_layers, num_attention_heads=heads, joint_attention_dim=joint_dim)


def make_qwen_weights(cfg: QwenImageConfig, seed: int = 0, dtype: torch.dtype = torch.float32) -> Dict[str, torch.Tensor]:
    """Random weights keyed like QwenImageTransformer2DModel.state_dict()."""
    g = torch.Generator().manual_seed(seed)
    D, d = cfg.inner_dim, cfg.attention_head_dim
    w: Dict[str, torch.Tensor] = {}

    def lin(name: str, out_f: int, in_f: int, scale: float = 1.0):
        w[name + ".weight"] = torch.randn(out_f, in_f, generator=g) * (scale / math.sqrt(in_f))
        w[name + ".bias"] = torch.randn(out_f, generator=g) * 0.02

    lin("img_in", D, cfg.in_channels)
    w["txt_norm.weight"] = 1.0 + 0.1 * torch.randn(cfg.joint_attention_dim, generator=g)
    lin("txt_in", D, cfg.joint_attention_dim)
    lin("time_text_embed.timestep_embedder.linear_1", D, 256)
    lin("time_text_embed.timestep_embedder.linear_2", D, D)
    for i in range(cfg.num_layers):
        pre = f"transformer_blocks.{i}."
        lin(pre + "img_mod.1", 6 * D, D, 0.5)
        lin(pre + "txt_mod.1", 6 * D, D, 0.5)
        for nm in ("to_q", "to_k", "to_v", "add_q_proj", "add_k_proj", "add_v_proj", "to_out.0", "to_add_out"):
            lin(pre + "attn." + nm, D, D)
        for nm in ("norm_q", "norm_k", "norm_added_q", "norm_added_k"):
            w[pre + f"attn.{nm}.weight"] = 1.0 + 0.1 * torch.randn(d, generator=g)
        for mlp in ("img_mlp", "txt_mlp"):
            lin(pre + mlp + ".net.0.proj", 4 * D, D)
            lin(pre + mlp + ".net.2", D, 4 * D)
    lin("norm_out.linear", 2 * D, D, 0.5)
    lin("proj_out", cfg.patch_size * cfg.patch_size * cfg.out_channels, D)
    return {k: v.to(dtype) for k, v in w.items()}


# ----------------------------------------------------------------------------------------------
# QwenEmbedRope (transformer_qwenimage.py:195-345, scale_rope=True): complex frequencies for image and text tokens
# ----------------------------------------------------------------------------------------------
def _rope_params(index: torch.Tensor, dim: int, theta: float = 10000.0) -> torch.Tensor:
    freqs = torch.outer(index, 1.0 / torch.pow(theta, torch.arange(0, dim, 2).to(torch.float32).div(dim)))
    return torch.polar(torch.ones_like(freqs), freqs)


def qwen_rope(frame: int, height: int, width: int, n_text: int, axes_dim: Sequence[int], theta: float = 10000.0):
    """-> (vid_freqs [frame*height*width, sum(axes)/2], txt_freqs [n_text, sum(axes)/2]) complex64, one image per sample."""
    pos_index = torch.arange(4096)
    neg_index = torch.arange(4096).flip(0) * -1 - 1
    pos = torch.cat([_rope_params(pos_index, a, theta) for a in axes_dim], dim=1)
    neg = torch.cat([_rope_params(neg_index, a, theta) for a in axes_dim], dim=1)
    fp = pos.split([x // 2 for x in axes_dim], dim=1)
    fn = neg.split([x // 2 for x in axes_dim], dim=1)
    f_frame = fp[0][0:frame].view(frame, 1, 1, -1).expand(frame, height, width, -1)
    f_h = torch.cat([fn[1][-(height - height // 2):], fp[1][: height // 2]], dim=0).view(1, height, 1, -1).expand(frame, height, width, -1)
    f_w = torch.cat([fn[2][-(width - width // 2):], fp[2][: width // 2]], dim=0).view(1, 1, width, -1).expand(frame, height, width, -1)
    vid = torch.cat([f_frame, f_h, f_w], dim=-1).reshape(frame * height * width, -1).clone().contiguous()
    max_vid_index = max(height // 2, width // 2)
    txt = pos[max_vid_index: max_vid_index + n_text]
    return vid, txt


def apply_rope_complex(x: torch.Tensor, freqs: torch.Tensor) -> torch.Tensor:
    """apply_rotary_emb_qwen(use_real=False) (transformer_qwenimage.py:137-142); x [B, S, H, d], freqs complex [S, d/2]."""
    xr = torch.view_as_complex(x.float().reshape(*x.shape[:-1], -1, 2))
    out = torch.view_as_real(xr * freqs.unsqueeze(1)).flatten(3)
    return out.type_as(x)


# ----------------------------------------------------------------------------------------------
# Block (QwenImageTransformerBlock.forward, 668-747) and attention (QwenDoubleStreamAttnProcessor2_0, 505-592)
# ----------------------------------------------------------------------------------------------
def _qwen_attention(w, pre: str, cfg: QwenImageConfig, hs, ehs, vid_freqs, txt_freqs, mask=None):
    H, d = cfg.num_attention_heads, cfg.attention_head_dim
    nt = ehs.shape[1]
    iq = _linear(w, pre + "to_q", hs).unflatten(-1, (H, d))
    ik = _linear(w, pre + "to_k", hs).unflatten(-1, (H, d))
    iv = _linear(w, pre + "to_v", hs).unflatten(-1, (H, d))
    tq = _linear(w, pre + "add_q_proj", ehs).unflatten(-1, (H, d))
    tk = _linear(w, pre + "add_k_proj", ehs).unflatten(-1, (H, d))
    tv = _linear(w, pre + "add_v_proj", ehs).unflatten(-1, (H, d))
    iq = _rms_norm(iq, w[pre + "norm_q.weight"])            # diffusers RMSNorm (qk_norm="rms_norm", eps 1e-6)
    ik = _rms_norm(ik, w[pre + "norm_k.weight"])
    tq = _rms_norm(tq, w[pre + "norm_added_q.weight"])
    tk = _rms_norm(tk, w[pre + "norm_added_k.weight"])
    iq, ik = apply_rope_complex(iq, vid_freqs), apply_rope_complex(ik, vid_freqs)
    tq, tk = apply_rope_complex(tq, txt_freqs), apply_rope_complex(tk, txt_freqs)
    q = torch.cat([tq, iq], dim=1)          # order [text, image] (556-560)
    k = torch.cat([tk, ik], dim=1)
    v = torch.cat([tv, iv], dim=1)
    o = F.scaled_dot_product_attention(q.permute(0, 2, 1, 3), k.permute(0, 2, 1, 3), v.permute(0, 2, 1, 3), attn_mask=mask,
                                       dropout_p=0.0, is_causal=False).permute(0, 2, 1, 3)
    o = o.flatten(2, 3).to(q.dtype)
    to, io = o[:, :nt], o[:, nt:]
    return _linear(w, pre + "to_out.0", io.contiguous()), _linear(w, pre + "to_add_out", to.contiguous())


def _modulate(x, mod):
    shift, scale, gate = mod.chunk(3, dim=-1)
    return x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1), gate.unsqueeze(1)


def _qwen_block(w, i: int, cfg: QwenImageConfig, hs, ehs, temb, vid_freqs, txt_freqs, mask=None):
    pre = f"transformer_blocks.{i}."
    img_mod = _linear(w, pre + "img_mod.1", F.silu(temb))
    txt_mod = _linear(w, pre + "txt_mod.1", F.silu(temb))
    img_mod1, img_mod2 = img_mod.chunk(2, dim=-1)
    txt_mod1, txt_mod2 = txt_mod.chunk(2, dim=-1)
    img_m, img_g1 = _modulate(_layer_norm(hs), img_mod1)
    txt_m, txt_g1 = _modulate(_layer_norm(ehs), txt_mod1)
    img_attn, txt_attn = _qwen_attention(w, pre + "attn.", cfg, img_m, txt_m, vid_freqs, txt_freqs, mask)
    hs = hs + img_g1 * img_attn
    ehs = ehs + txt_g1 * txt_attn
    img_m2, img_g2 = _modulate(_layer_norm(hs), img_mod2)
    hs = hs + img_g2 * _ff(w, pre + "img_mlp.", img_m2)
    txt_m2, txt_g2 = _modulate(_layer_norm(ehs), txt_mod2)
    ehs = ehs + txt_g2 * _ff(w, pre + "txt_mlp.", txt_m2)
    return ehs, hs


def qwen_forward(w: Dict[str, torch.Tensor], cfg: QwenImageConfig, hidden_states: torch.Tensor, encoder_hidden_states: torch.Tensor,
                 timestep: torch.Tensor, img_shape: Tuple[int, int, int], encoder_hidden_states_mask: Optional[torch.Tensor] = None):
    """QwenImageTransformer2DModel.forward (transformer_qwenimage.py:878-993), one image per sample, no zero_cond_t / guidance.
    hidden_states: packed latents [B, Ni, 64]; timestep already / 1000 (FF/models/qwen_image/qwen_image.py:556)."""
    hs = _linear(w, "img_in", hidden_states)
    timestep = timestep.to(hs.dtype)
    ehs = _rms_norm(encoder_hidden_states, w["txt_norm.weight"])       # diffusers RMSNorm over the joint dim (eps 1e-6)
    ehs = _linear(w, "txt_in", ehs)
    # QwenTimestepProjEmbeddings: Timesteps(256, flip_sin_to_cos, shift 0, scale=1000) -> TimestepEmbedding (176-193)
    tproj = _timesteps_scaled(timestep)
    temb = _linear(w, "time_text_embed.timestep_embedder.linear_2",
                   F.silu(_linear(w, "time_text_embed.timestep_embedder.linear_1", tproj.to(dtype=hs.dtype))))
    vid_freqs, txt_freqs = (f.to(hs.device) for f in qwen_rope(*img_shape, encoder_hidden_states.shape[1], cfg.axes_dims_rope))
    mask = None
    if encoder_hidden_states_mask is not None:
        m = encoder_hidden_states_mask.to(device=hs.device, dtype=torch.bool)
        mask = torch.cat([m, torch.ones((hs.shape[0], hs.shape[1]), dtype=torch.bool, device=hs.device)], dim=1)[:, None, None, :]
    for i in range(cfg.num_layers):
        ehs, hs = _qwen_block(w, i, cfg, hs, ehs, temb, vid_freqs, txt_freqs, mask)
    emb = _linear(w, "norm_out.linear", F.silu(temb).to(hs.dtype))
    scale, shift = torch.chunk(emb, 2, dim=1)
    hs = _layer_norm(hs) * (1 + scale)[:, None, :] + shift[:, None, :]
    return _linear(w, "proj_out", hs)


def _timesteps_scaled(timesteps: torch.Tensor, dim: int = 256, scale: float = 1000.0) -> torch.Tensor:
    """get_timestep_embedding(flip_sin_to_cos=True, downscale_freq_shift=0, scale=1000) (DF/models/embeddings.py:26-77)."""
    half = dim // 2
    exponent = -math.log(10000) * torch.arange(0, half, dtype=torch.float32, device=timesteps.device) / half
    emb = torch.exp(exponent)
    emb = timesteps[:, None].float() * emb[None, :]
    emb = scale * emb
    emb = torch.cat([torch.sin(emb), torch.cos(emb)], dim=-1)
    return torch.cat([emb[:, half:], emb[:, :half]], dim=-1)


def true_cfg_combine(noise_pred: torch.Tensor, neg_noise_pred: torch.Tensor, guidance_scale: float) -> torch.Tensor:
    """Per-token norm-rescaled CFG (FF/models/qwen_image/qwen_image.py:580-587)."""
    comb = neg_noise_pred + guidance_scale * (noise_pred - neg_noise_pred)
    cond_norm = torch.norm(noise_pred, dim=-1, keepdim=True)
    noise_norm = torch.norm(comb, dim=-1, keepdim=True)
    return comb * (cond_norm / noise_norm)


def make_qwen_inputs(cfg: QwenImageConfig, batch: int, h2: int, w2: int, n_text: int, seed: int = 1):
    g = torch.Generator().manual_seed(seed)
    lat = torch.randn(batch, h2 * w2, cfg.in_channels, generator=g)
    pe = torch.randn(batch, n_text, cfg.joint_attention_dim, generator=g)
    return lat, pe
