"""CPU/torch restatement of the FLUX.1 rollout path (TEST INFRASTRUCTURE - see oracle/__init__.py).

SURVEY.md section 8(f) "next" row 2 / BASELINE config 3.  Every function cites the reference file:line it follows
(paths relative to /root/reference: FF = src/flow_factory ; DF = diffusers/src/diffusers).  Same convention as
oracle/sd3_oracle.py: the same torch functional ops in the same order as the reference modules, so that running under
`torch.autocast` reproduces the reference's autocast numerics, and without autocast on fp32 weights the fp32 truth.
Pinned bit-exact against the imported reference by tests/golden/make_golden.py -> tests/golden/flux_*.pt.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

from .sd3_oracle import _ff, _layer_norm, _linear, timestep_embedding


# ----------------------------------------------------------------------------------------------
# Model config (DF/models/transformers/transformer_flux.py:583-596 register_to_config arguments)
# ----------------------------------------------------------------------------------------------
@dataclass
class FluxConfig:
    patch_size: int = 1
    in_channels: int = 64
    num_layers: int = 19
    num_single_layers: int = 38
    attention_head_dim: int = 128
    num_attention_heads: int = 24
    joint_attention_dim: int = 4096
    pooled_projection_dim: int = 768
    guidance_embeds: bool = True
    axes_dims_rope: Tuple[int, int, int] = (16, 56, 56)

    @property
    def inner_dim(self) -> int:
        return self.num_attention_heads * self.attention_head_dim

    def ref_kwargs(self) -> dict:
        return dict(patch_size=self.patch_size, in_channels=self.in_channels, num_layers=self.num_layers,
                    num_single_layers=self.num_single_layers, attention_head_dim=self.attention_head_dim,
                    num_attention_heads=self.num_attention_heads, joint_attention_dim=self.joint_attention_dim,
                    pooled_projection_dim=self.pooled_projection_dim, guidance_embeds=self.guidance_embeds,
                    axes_dims_rope=tuple(self.axes_dims_rope))


def flux1_dev() -> FluxConfig:
    """FLUX.1-dev (transformer_flux.py defaults 583-596 + guidance_embeds=True, the dev checkpoint's setting)."""
    return FluxConfig()


def tiny_flux_config(num_layers: int = 1, num_single_layers: int = 2, heads: int = 2, joint_dim: int = 64,
                     pooled_dim: int = 32) -> FluxConfig:
    return FluxConfig(num_layers=num_layers, num_single_layers=num_single_layers, num_attention_heads=heads,
                      joint_attention_dim=joint_dim, pooled_projection_dim=pooled_dim)


def make_flux_weights(cfg: FluxConfig, seed: int = 0, dtype: torch.dtype = torch.float32, device: str = "cpu") -> Dict[str, torch.Tensor]:
    """Random weights keyed like FluxTransformer2DModel.state_dict() (seeded, checkpoint-independent)."""
    g = torch.Generator(device=device).manual_seed(seed)
    D, d = cfg.inner_dim, cfg.attention_head_dim
    w: Dict[str, torch.Tensor] = {}

    def randn(*shape):
        return torch.randn(*shape, generator=g, device=device)

    def lin(name: str, out_f: int, in_f: int, scale: float = 1.0, bias_std: float = 0.02):
        w[name + ".weight"] = randn(out_f, in_f) * (scale / math.sqrt(in_f))
        w[name + ".bias"] = randn(out_f) * bias_std

    def rms(name: str):
        w[name + ".weight"] = 1.0 + 0.1 * randn(d)

    lin("x_embedder", D, cfg.in_channels)
    lin("context_embedder", D, cfg.joint_attention_dim)
    lin("time_text_embed.timestep_embedder.linear_1", D, 256)
    lin("time_text_embed.timestep_embedder.linear_2", D, D)
    if cfg.guidance_embeds:
        lin("time_text_embed.guidance_embedder.linear_1", D, 256)
        lin("time_text_embed.guidance_embedder.linear_2", D, D)
    lin("time_text_embed.text_embedder.linear_1", D, cfg.pooled_projection_dim)
    lin("time_text_embed.text_embedder.linear_2", D, D)
    for i in range(cfg.num_layers):
        pre = f"transformer_blocks.{i}."
        lin(pre + "norm1.linear", 6 * D, D, scale=0.5)
        lin(pre + "norm1_context.linear", 6 * D, D, scale=0.5)
        for nm in ("to_q", "to_k", "to_v", "add_q_proj", "add_k_proj", "add_v_proj", "to_out.0", "to_add_out"):
            lin(pre + "attn." + nm, D, D)
        for nm in ("norm_q", "norm_k", "norm_added_q", "norm_added_k"):
            rms(pre + "attn." + nm)
        for ff in ("ff", "ff_context"):
            lin(pre + ff + ".net.0.proj", 4 * D, D)
            lin(pre + ff + ".net.2", D, 4 * D)
    for i in range(cfg.num_single_layers):
        pre = f"single_transformer_blocks.{i}."
        lin(pre + "norm.linear", 3 * D, D, scale=0.5)
        lin(pre + "proj_mlp", 4 * D, D)
        lin(pre + "proj_out", D, 5 * D)
        for nm in ("to_q", "to_k", "to_v"):
            lin(pre + "attn." + nm, D, D)
        rms(pre + "attn.norm_q")
        rms(pre + "attn.norm_k")
    lin("norm_out.linear", 2 * D, D, scale=0.5)
    lin("proj_out", cfg.patch_size * cfg.patch_size * cfg.in_channels, D)
    return {k: v.to(dtype) for k, v in w.items()}


# ----------------------------------------------------------------------------------------------
# Rotary position tables (FluxPosEmbed.forward, transformer_flux.py:500-522; get_1d_rotary_pos_embed, embeddings.py:1119-1174)
# ----------------------------------------------------------------------------------------------
def rope_tables(ids: torch.Tensor, axes_dim: Sequence[int], theta: float = 10000.0) -> Tuple[torch.Tensor, torch.Tensor]:
    """ids [S, 3] -> (cos, sin) each fp32 [S, sum(axes_dim)], frequencies in float64, each value repeated twice (interleaved)."""
    pos = ids.float()
    cos_out, sin_out = [], []
    for i, dim in enumerate(axes_dim):
        freqs = 1.0 / (theta ** (torch.arange(0, dim, 2, dtype=torch.float64, device=pos.device) / dim))
        freqs = torch.outer(pos[:, i], freqs)
        cos_out.append(freqs.cos().repeat_interleave(2, dim=1, output_size=freqs.shape[1] * 2).float())
        sin_out.append(freqs.sin().repeat_interleave(2, dim=1, output_size=freqs.shape[1] * 2).float())
    return torch.cat(cos_out, dim=-1), torch.cat(sin_out, dim=-1)


def apply_rope(x: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor) -> torch.Tensor:
    """apply_rotary_emb(use_real=True, use_real_unbind_dim=-1, sequence_dim=1) (embeddings.py:1207-1233); x [B, S, H, d]."""
    cos, sin = cos[None, :, None, :], sin[None, :, None, :]
    x_real, x_imag = x.reshape(*x.shape[:-1], -1, 2).unbind(-1)
    x_rot = torch.stack([-x_imag, x_real], dim=-1).flatten(3)
    return (x.float() * cos + x_rot.float() * sin).to(x.dtype)


def latent_image_ids(lat_h: int, lat_w: int, device="cpu", dtype=torch.float32) -> torch.Tensor:
    """FluxPipeline._prepare_latent_image_ids (DF/pipelines/flux/pipeline_flux.py): (h/2 * w/2, 3) with (0, row, col)."""
    h2, w2 = lat_h // 2, lat_w // 2
    ids = torch.zeros(h2, w2, 3)
    ids[..., 1] = ids[..., 1] + torch.arange(h2)[:, None]
    ids[..., 2] = ids[..., 2] + torch.arange(w2)[None, :]
    return ids.reshape(h2 * w2, 3).to(device=device, dtype=dtype)


def pack_latents(lat: torch.Tensor) -> torch.Tensor:
    """FluxPipeline._pack_latents: [B, C, H, W] -> [B, (H/2)(W/2), 4C]."""
    B, C, H, W = lat.shape
    lat = lat.view(B, C, H // 2, 2, W // 2, 2).permute(0, 2, 4, 1, 3, 5)
    return lat.reshape(B, (H // 2) * (W // 2), C * 4)


# ----------------------------------------------------------------------------------------------
# Attention (FluxAttnProcessor.__call__, transformer_flux.py:83-139)
# ----------------------------------------------------------------------------------------------
def _rms(x: torch.Tensor, weight: torch.Tensor, eps: float) -> torch.Tensor:
    """torch.nn.RMSNorm over the head dim (transformer_flux.py:311-312, 324-325)."""
    return F.rms_norm(x, (x.shape[-1],), weight, eps)


def _flux_attention(w, pre: str, cfg: FluxConfig, hs: torch.Tensor, ehs: Optional[torch.Tensor], cos, sin, eps: float):
    B = hs.shape[0]
    H, d = cfg.num_attention_heads, cfg.attention_head_dim
    q = _linear(w, pre + "to_q", hs).unflatten(-1, (H, d))
    k = _linear(w, pre + "to_k", hs).unflatten(-1, (H, d))
    v = _linear(w, pre + "to_v", hs).unflatten(-1, (H, d))
    q = _rms(q, w[pre + "norm_q.weight"], eps)
    k = _rms(k, w[pre + "norm_k.weight"], eps)
    if ehs is not None:
        eq = _linear(w, pre + "add_q_proj", ehs).unflatten(-1, (H, d))
        ek = _linear(w, pre + "add_k_proj", ehs).unflatten(-1, (H, d))
        ev = _linear(w, pre + "add_v_proj", ehs).unflatten(-1, (H, d))
        eq = _rms(eq, w[pre + "norm_added_q.weight"], eps)
        ek = _rms(ek, w[pre + "norm_added_k.weight"], eps)
        q = torch.cat([eq, q], dim=1)   # TEXT tokens first, then image (110-112)
        k = torch.cat([ek, k], dim=1)
        v = torch.cat([ev, v], dim=1)
    q = apply_rope(q, cos, sin)
    k = apply_rope(k, cos, sin)
    # dispatch_attention_fn, native backend: SDPA on [B, H, S, d] (attention_dispatch.py _native_attention)
    o = F.scaled_dot_product_attention(q.permute(0, 2, 1, 3), k.permute(0, 2, 1, 3), v.permute(0, 2, 1, 3),
                                       dropout_p=0.0, is_causal=False).permute(0, 2, 1, 3)
    o = o.flatten(2, 3).to(q.dtype)
    if ehs is not None:
        eo, o = o[:, : ehs.shape[1]], o[:, ehs.shape[1]:]
        o = _linear(w, pre + "to_out.0", o.contiguous())
        eo = _linear(w, pre + "to_add_out", eo.contiguous())
        return o, eo
    return o, None


def _dual_block(w, i: int, cfg: FluxConfig, hs, ehs, temb, cos, sin):
    """FluxTransformerBlock.forward (transformer_flux.py:438-492); AdaLayerNormZero (normalization.py:157-170)."""
    pre = f"transformer_blocks.{i}."
    emb = _linear(w, pre + "norm1.linear", F.silu(temb))
    shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = emb.chunk(6, dim=1)
    norm_hs = _layer_norm(hs) * (1 + scale_msa[:, None]) + shift_msa[:, None]
    cemb = _linear(w, pre + "norm1_context.linear", F.silu(temb))
    c_shift_msa, c_scale_msa, c_gate_msa, c_shift_mlp, c_scale_mlp, c_gate_mlp = cemb.chunk(6, dim=1)
    norm_ehs = _layer_norm(ehs) * (1 + c_scale_msa[:, None]) + c_shift_msa[:, None]
    attn_out, ctx_out = _flux_attention(w, pre + "attn.", cfg, norm_hs, norm_ehs, cos, sin, eps=1e-6)
    hs = hs + gate_msa.unsqueeze(1) * attn_out
    norm_hs = _layer_norm(hs)
    norm_hs = norm_hs * (1 + scale_mlp[:, None]) + shift_mlp[:, None]
    hs = hs + gate_mlp.unsqueeze(1) * _ff(w, pre + "ff.", norm_hs)
    ehs = ehs + c_gate_msa.unsqueeze(1) * ctx_out
    norm_ehs = _layer_norm(ehs)
    norm_ehs = norm_ehs * (1 + c_scale_mlp[:, None]) + c_shift_mlp[:, None]
    ehs = ehs + c_gate_mlp.unsqueeze(1) * _ff(w, pre + "ff_context.", norm_ehs)
    return ehs, hs


def _single_block(w, i: int, cfg: FluxConfig, hs, ehs, temb, cos, sin):
    """FluxSingleTransformerBlock.forward (transformer_flux.py:378-407); AdaLayerNormZeroSingle (normalization.py:194-202)."""
    pre = f"single_transformer_blocks.{i}."
    nt = ehs.shape[1]
    x = torch.cat([ehs, hs], dim=1)
    residual = x
    emb = _linear(w, pre + "norm.linear", F.silu(temb))
    shift_msa, scale_msa, gate = emb.chunk(3, dim=1)
    nx = _layer_norm(x) * (1 + scale_msa[:, None]) + shift_msa[:, None]
    mlp = F.gelu(_linear(w, pre + "proj_mlp", nx), approximate="tanh")
    attn_out, _ = _flux_attention(w, pre + "attn.", cfg, nx, None, cos, sin, eps=1e-6)
    x = torch.cat([attn_out, mlp], dim=2)
    x = gate.unsqueeze(1) * _linear(w, pre + "proj_out", x)
    x = residual + x
    return x[:, :nt], x[:, nt:]


def flux_forward(w: Dict[str, torch.Tensor], cfg: FluxConfig, hidden_states: torch.Tensor, encoder_hidden_states: torch.Tensor,
                 pooled_projections: torch.Tensor, timestep: torch.Tensor, img_ids: torch.Tensor, txt_ids: torch.Tensor,
                 guidance: Optional[torch.Tensor] = None, return_intermediates: bool = False):
    """FluxTransformer2DModel.forward (transformer_flux.py:676-778).  hidden_states: packed latents [B, Ni, 64];
    timestep already divided by 1000 by the caller (FF/models/flux/flux1.py:325)."""
    inter = {}
    hs = _linear(w, "x_embedder", hidden_states)
    timestep = timestep.to(hs.dtype) * 1000
    if guidance is not None:
        guidance = guidance.to(hs.dtype) * 1000
    # CombinedTimestep(Guidance)TextProjEmbeddings (embeddings.py:1612-1624 / 1592-1600)
    def _mlp(name, x):
        return _linear(w, name + ".linear_2", F.silu(_linear(w, name + ".linear_1", x)))
    temb = _mlp("time_text_embed.timestep_embedder", timestep_embedding(timestep, 256).to(dtype=pooled_projections.dtype))
    if guidance is not None:
        temb = temb + _mlp("time_text_embed.guidance_embedder", timestep_embedding(guidance, 256).to(dtype=pooled_projections.dtype))
    temb = temb + _mlp("time_text_embed.text_embedder", pooled_projections)
    ehs = _linear(w, "context_embedder", encoder_hidden_states)
    cos, sin = (t.to(hs.device) for t in rope_tables(torch.cat((txt_ids, img_ids), dim=0), cfg.axes_dims_rope))
    if return_intermediates:
        inter["temb"], inter["hs0"], inter["ehs0"], inter["cos"], inter["sin"] = temb, hs, ehs, cos, sin
    for i in range(cfg.num_layers):
        ehs, hs = _dual_block(w, i, cfg, hs, ehs, temb, cos, sin)
        if return_intermediates:
            inter[f"hs_{i}"], inter[f"ehs_{i}"] = hs, ehs
    for i in range(cfg.num_single_layers):
        ehs, hs = _single_block(w, i, cfg, hs, ehs, temb, cos, sin)
        if return_intermediates:
            inter[f"s_hs_{i}"], inter[f"s_ehs_{i}"] = hs, ehs
    # norm_out: AdaLayerNormContinuous (normalization.py:346-351)
    emb = _linear(w, "norm_out.linear", F.silu(temb).to(hs.dtype))
    scale, shift = torch.chunk(emb, 2, dim=1)
    hs = _layer_norm(hs) * (1 + scale)[:, None, :] + shift[:, None, :]
    out = _linear(w, "proj_out", hs)
    return (out, inter) if return_intermediates else out


def calculate_shift(image_seq_len: int, base_seq_len: int = 256, max_seq_len: int = 4096, base_shift: float = 0.5,
                    max_shift: float = 1.15) -> float:
    """FF/scheduler/flow_match_euler_discrete.py:37-47."""
    m = (max_shift - base_shift) / (max_seq_len - base_seq_len)
    b = base_shift - m * base_seq_len
    return image_seq_len * m + b


def make_flux_inputs(cfg: FluxConfig, batch: int, lat_h: int, lat_w: int, n_text: int, seed: int = 1):
    """Packed latents [B, (h/2)(w/2), 64], prompt embeds, pooled, ids (fp32)."""
    g = torch.Generator().manual_seed(seed)
    lat = torch.randn(batch, cfg.in_channels // 4, lat_h, lat_w, generator=g)
    pe = torch.randn(batch, n_text, cfg.joint_attention_dim, generator=g)
    pooled = torch.randn(batch, cfg.pooled_projection_dim, generator=g)
    return pack_latents(lat), pe, pooled, latent_image_ids(lat_h, lat_w), torch.zeros(n_text, 3)


def flux_flops_per_forward(cfg: FluxConfig, ni: int, nt: int) -> Tuple[float, float]:
    """(linear, attention) FLOPs of one sample-forward (MAC = 2 FLOP)."""
    D, S = cfg.inner_dim, ni + nt
    dual = cfg.num_layers * (2 * S * D * (3 * D + D + 8 * D))
    single = cfg.num_single_layers * (2 * S * D * (3 * D + 4 * D) + 2 * S * 5 * D * D)
    attn = (cfg.num_layers + cfg.num_single_layers) * 4.0 * S * S * D
    return float(dual + single), float(attn)


# ----------------------------------------------------------------------------------------------
# Scheduler with resolution-dependent ("dynamic") shifting and the rollout loop
# ----------------------------------------------------------------------------------------------
def flux_make_schedule(num_inference_steps: int, image_seq_len: int, num_train_timesteps: int = 1000):
    """set_scheduler_timesteps (FF/scheduler/flow_match_euler_discrete.py:49-77) -> mu = calculate_shift(seq_len) ->
    diffusers set_timesteps with use_dynamic_shifting (DF/schedulers/scheduling_flow_match_euler_discrete.py:346-348, 648-649):
    sigmas = exp(mu) / (exp(mu) + (1/sigma - 1)**1.0) on the float32 linspace; timesteps = sigmas*1000; trailing 0."""
    import numpy as np
    mu = calculate_shift(image_seq_len)
    sig = np.linspace(1.0, 1 / num_inference_steps, num_inference_steps).astype(np.float32)
    sig = math.exp(mu) / (math.exp(mu) + (1 / sig - 1) ** 1.0)
    sigmas = torch.from_numpy(sig).to(dtype=torch.float32)
    timesteps = sigmas * num_train_timesteps
    return timesteps, torch.cat([sigmas, torch.zeros(1)])


def flux_rollout(w, cfg: FluxConfig, packed_x0: torch.Tensor, prompt_embeds: torch.Tensor, pooled: torch.Tensor,
                 img_ids: torch.Tensor, num_steps: int, guidance_scale: float, noise_level: float = 0.7, noises=None,
                 dynamics: str = "Flow-SDE", compute_log_prob: bool = True, storage_dtype: torch.dtype = torch.float16):
    """Flux1Adapter.inference loop + forward (FF/models/flux/flux1.py:211-250, 310-349): no CFG (embedded guidance),
    timestep / 1000 into the model, zeros txt_ids, scheduler.step on the packed [B, Ni, 64] latents."""
    from .sd3_oracle import cast_latents, current_sde_steps, sde_step
    B = packed_x0.shape[0]
    timesteps, sigmas = flux_make_schedule(num_steps, packed_x0.shape[1])
    sde = set(current_sde_steps(num_steps, None, None, 42))
    latents = cast_latents(packed_x0, storage_dtype)
    lats, lps, vps = [latents], {}, []
    txt_ids = torch.zeros(prompt_embeds.shape[1], 3)
    for i in range(num_steps):
        t = timesteps[i]
        nl = noise_level if i in sde else 0.0
        guidance = torch.as_tensor(guidance_scale, dtype=latents.dtype).expand(B)
        v = flux_forward(w, cfg, latents.to(prompt_embeds.dtype), prompt_embeds, pooled, t.expand(B) / 1000, img_ids, txt_ids,
                         guidance=guidance.to(prompt_embeds.dtype))
        r = sde_step(v, latents, float(sigmas[i]), float(sigmas[i + 1]), nl, float(sigmas[1]), dynamics,
                     noise=None if noises is None else noises[i], compute_log_prob=compute_log_prob and nl > 0)
        latents = cast_latents(r["next_latents"], storage_dtype)
        lats.append(latents); vps.append(v)
        if compute_log_prob and nl > 0:
            lps[i] = r["log_prob"]
    return dict(latents=lats, log_probs=lps, noise_preds=vps, timesteps=timesteps, sigmas=sigmas)
