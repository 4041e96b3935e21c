"""Record what the original Flow-Factory project (and its vendored diffusers) computes for the drop-in boundary checks of
tests/test_reference_hooks.py, so that those checks run without the original project on the machine.

    python tests/golden/make_reference_hooks.py <Flow-Factory checkout>

Reference commits: Flow-Factory a0b2bc5, diffusers submodule f7fd76a.  torch 2.11.0 CPU.  Writes tests/golden/reference_hooks.pt.xz
(torch.save, xz-compressed): the inputs of every randomised case and the reference's results on them; the test computes this repository's
side and compares.
"""
import dataclasses
import importlib
import inspect
import io
import logging
import lzma
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.path.abspath(sys.argv[1])
sys.path[:0] = [os.path.join(HERE, "ref_stubs"), os.path.join(REF, "diffusers", "src"), os.path.join(REF, "src"), ROOT]

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tests.test_reference_hooks import ADAPTERS, SAMPLES, _O, _f1, _f2, _f3, _behaviour, _probe  # noqa: E402


def shapes(sd):
    return {k: tuple(v.shape) for k, v in sd.items()}


def adapters():
    from flow_factory.models.registry import get_model_adapter_class
    out = {}
    for name, (ref_path, _) in ADAPTERS.items():
        ref = get_model_adapter_class(ref_path)
        out[name] = {fn: [p for p in inspect.signature(getattr(ref, fn)).parameters if p != "self"] for fn in ("inference", "forward")}
    return out


def samples():
    out = {}
    for name, (mod, ref_cls, _) in SAMPLES.items():
        R = getattr(importlib.import_module(mod), ref_cls)
        out[name] = {"fields": sorted(f.name for f in dataclasses.fields(R)), "shared_fields": sorted(R.shared_fields()),
                     "behaviour": _behaviour(R)}
    return out


def trajectory(rng):
    from flow_factory.utils.trajectory_collector import create_trajectory_collector as ref_collector, compute_trajectory_indices as ref_cti
    cases = []
    for _ in range(300):
        T = rng.choice([1, 2, 4, 7, 10, 30])
        kind = rng.choice(["all", "none", "list", "neg", "dups", "cti"])
        cti = None
        if kind == "all": idx = "all"
        elif kind == "none": idx = None
        elif kind == "list": idx = sorted(rng.sample(range(T + 1), rng.randint(1, T + 1)))
        elif kind == "neg": idx = [rng.randint(-(T + 1), T) for _ in range(rng.randint(1, 5))]
        elif kind == "dups": idx = [rng.randint(0, T) for _ in range(rng.randint(1, 8))]
        else:
            tr = sorted(rng.sample(range(T), rng.randint(1, T)))
            inc = rng.random() < 0.5
            idx = ref_cti(tr, T, include_initial=inc)
            cti = (tr, inc, idx)
        has_lp = [rng.random() < 0.5 for _ in range(T)]
        case = {"kind": kind, "T": T, "idx": idx, "has_lp": has_lp, "cti": cti, "ref": None}
        cases.append(case)
        try:
            lc, pc = ref_collector(idx, T), ref_collector(idx, T)
        except Exception:
            continue                                        # ref["ref"] stays None: the reference raised
        lc.collect(torch.zeros(1), step_idx=0)
        for i in range(T):
            lc.collect(torch.zeros(1), i + 1)
            if has_lp[i]: pc.collect(torch.zeros(1), i)
        rl, rp = lc.get_result(), pc.get_result()
        case["ref"] = {"n_lat": 0 if rl is None else len(rl), "n_lp": 0 if rp is None else len(rp),
                       "lat_map": lc.get_index_map(), "lp_map": pc.get_index_map()}
    return cases


def callback(rng):
    from flow_factory.utils.trajectory_collector import create_callback_collector as ref_cb
    cases = []
    for _ in range(120):
        T = rng.choice([1, 3, 6, 10])
        idx = rng.choice(["all", None, sorted(rng.sample(range(T + 1), rng.randint(1, T + 1))), [rng.randint(-(T + 1), T) for _ in range(3)]])
        keys = rng.choice([[], ["next_latents_mean"], ["next_latents_mean", "noise_level", "tag", "log_prob", "missing"]])
        a = ref_cb(idx, T)
        for i in range(T):
            a.collect_step(i, _O(i), keys, {"noise_level": 0.7 if i % 2 else None})
        cases.append({"T": T, "idx": idx, "keys": keys,
                      "ref": {"result": a.get_result(), "len": len(a), "collected_indices": a.collected_indices, "is_disabled": a.is_disabled,
                              "index_map": a.get_index_map()}})
    return cases


def scheduler(rng):
    from flow_factory.scheduler import FlowMatchEulerDiscreteSDEScheduler as RefFM, UniPCMultistepSDEScheduler as RefUP, set_scheduler_timesteps as ref_set
    x = torch.randn(2, 4, 4, 4, generator=torch.Generator().manual_seed(0)).half()
    v = torch.randn(2, 4, 4, 4, generator=torch.Generator().manual_seed(1)).bfloat16()
    logging.disable(logging.WARNING)
    cases = []
    for _ in range(60):
        T = rng.choice([4, 10, 28, 30])
        dyn = rng.choice(["Flow-SDE", "Dance-SDE", "CPS", "ODE"])
        nsde = rng.choice([None, 1, 2, 3])
        sde = rng.choice([None, sorted(rng.sample(range(T), rng.randint(1, T)))])
        seed = rng.randint(0, 1000)
        nl = rng.choice([0.3, 0.7, 1.0])
        c = {"T": T, "dyn": dyn, "nsde": nsde, "sde": sde, "seed": seed, "nl": nl}
        if rng.random() < 0.5:
            dynshift = rng.random() < 0.5
            kw = dict(use_dynamic_shifting=True) if dynshift else dict(shift=rng.choice([1.0, 3.0, 5.0]))
            r = RefFM(noise_level=nl, sde_steps=sde, num_sde_steps=nsde, seed=seed, dynamics_type=dyn, **kw)
            seq = rng.choice([256, 1024, 4096])
            rt = ref_set(r, T, seq_len=seq, device="cpu")
            c.update(cls="FlowMatch", kw=kw, seq=seq)
        else:
            fs = rng.choice([3.0, 5.0])
            r = RefUP(noise_level=nl, sde_steps=sde, num_sde_steps=nsde, seed=seed, dynamics_type=dyn, prediction_type="flow_prediction",
                      use_flow_sigmas=True, flow_shift=fs, num_train_timesteps=1000)
            r.set_timesteps(T, device="cpu"); rt = r.timesteps
            c.update(cls="UniPC", fs=fs)
        r.rollout()
        i = rng.randrange(T)
        t, tn = rt[i], (rt[i + 1] if i + 1 < T else torch.tensor(0, dtype=rt.dtype))
        cur = r.get_noise_level_for_timestep(t)
        o = r.step(noise_pred=v, timestep=t, latents=x, timestep_next=tn, noise_level=cur, compute_log_prob=False, return_dict=True)
        ref = {"timesteps": rt.cpu(), "sigmas": r.sigmas.cpu(), "sde_steps": r.sde_steps, "num_sde_steps": r.num_sde_steps,
               "current_sde_steps": r.current_sde_steps, "noise_levels": r.get_noise_levels().float(),
               "train_timesteps": torch.as_tensor(r.train_timesteps), "noise_level_t": cur, "index_t": r.index_for_timestep(t),
               "dt": float(o.dt.flatten()[0]), "std_dev_t": float(torch.as_tensor(o.std_dev_t).flatten()[0])}
        if isinstance(r, RefFM):       # timestep_next omitted: the reference reads sigmas[i], sigmas[i + 1] from its tables
            o2 = r.step(noise_pred=v, timestep=t, latents=x, noise_level=cur, compute_log_prob=False, return_dict=True)
            ref.update(dt_no_next=float(o2.dt.flatten()[0]), std_dev_t_no_next=float(torch.as_tensor(o2.std_dev_t).flatten()[0]))
        c.update(i=i, ref=ref)
        cases.append(c)
    logging.disable(logging.NOTSET)
    return cases


def positional():
    from diffusers.models.transformers.transformer_flux import FluxPosEmbed
    from diffusers.models.transformers.transformer_qwenimage import QwenEmbedRope
    from diffusers.models.transformers.transformer_wan import WanRotaryPosEmbed
    from diffusers.pipelines.flux.pipeline_flux import FluxPipeline
    from flow_factory.scheduler.flow_match_euler_discrete import calculate_shift
    h2, w2, nt = 6, 10, 7
    ids = torch.cat([torch.zeros(nt, 3), FluxPipeline._prepare_latent_image_ids(1, h2, w2, "cpu", torch.float32)], 0)
    fc, fs = FluxPosEmbed(theta=10000, axes_dim=[16, 56, 56])(ids)
    lat = torch.randn(2, 16, 2 * h2, 2 * w2, generator=torch.Generator().manual_seed(0))
    vid, txt = QwenEmbedRope(theta=10000, axes_dim=[16, 56, 56], scale_rope=True)([(1, h2, w2)], max_txt_seq_len=nt, device=torch.device("cpu"))
    wr = WanRotaryPosEmbed(attention_head_dim=128, patch_size=(1, 2, 2), max_seq_len=64)
    wc, ws = wr(torch.zeros(1, 16, 3, 8, 10))
    wcb, wsb = wr.to(torch.bfloat16)(torch.zeros(1, 16, 3, 8, 10))
    return {"flux_cos": fc, "flux_sin": fs, "flux_lat": lat, "flux_packed": FluxPipeline._pack_latents(lat, 2, 16, 2 * h2, 2 * w2),
            "shift": {n: calculate_shift(n) for n in (256, 1024, 4096, 4429)}, "qwen": torch.cat([txt, vid], 0),
            "wan_cos": wc, "wan_sin": ws, "wan_cos_bf16": wcb, "wan_sin_bf16": wsb}


def vae_host():
    from diffusers.models.autoencoders.autoencoder_kl import AutoencoderKL
    from diffusers.image_processor import VaeImageProcessor
    vm = AutoencoderKL(in_channels=3, out_channels=3, down_block_types=("DownEncoderBlock2D",) * 2, up_block_types=("UpDecoderBlock2D",) * 2,
                       block_out_channels=(32, 64), layers_per_block=1, latent_channels=4, norm_num_groups=8, use_quant_conv=False,
                       use_post_quant_conv=False, scaling_factor=1.5305, shift_factor=0.0609)
    img = torch.randn(2, 3, 8, 8, generator=torch.Generator().manual_seed(0)) * 2
    return {"config": dict(vm.config), "state_dict": shapes(vm.state_dict()), "img": img,
            "postprocessed": VaeImageProcessor(vae_scale_factor=8).postprocess(img, output_type="pt"),
            "default_config": dict(AutoencoderKL(block_out_channels=(32,), norm_num_groups=8).config)}


def intake():
    """Config and state-dict key / shape of a real (tiny) model per engine: what the config intakes and weight packers read."""
    from diffusers.models.transformers.transformer_sd3 import SD3Transformer2DModel
    from diffusers.models.transformers.transformer_flux import FluxTransformer2DModel
    from diffusers.models.transformers.transformer_qwenimage import QwenImageTransformer2DModel
    from diffusers.models.transformers.transformer_wan import WanTransformer3DModel
    models = {
        "sd3": SD3Transformer2DModel(sample_size=16, patch_size=2, in_channels=16, num_layers=2, attention_head_dim=64, num_attention_heads=2,
                                     joint_attention_dim=64, caption_projection_dim=128, pooled_projection_dim=32, out_channels=16,
                                     pos_embed_max_size=16, dual_attention_layers=(0,), qk_norm="rms_norm"),
        "flux": FluxTransformer2DModel(patch_size=1, in_channels=64, num_layers=1, num_single_layers=1, attention_head_dim=128,
                                       num_attention_heads=2, joint_attention_dim=64, pooled_projection_dim=32, guidance_embeds=True,
                                       axes_dims_rope=(16, 56, 56)),
        "qwen": QwenImageTransformer2DModel(patch_size=2, in_channels=64, out_channels=16, num_layers=1, attention_head_dim=128,
                                            num_attention_heads=2, joint_attention_dim=64, axes_dims_rope=(16, 56, 56)),
        "wan": WanTransformer3DModel(patch_size=(1, 2, 2), num_attention_heads=2, attention_head_dim=128, in_channels=16, out_channels=16,
                                     text_dim=64, freq_dim=256, ffn_dim=320, num_layers=1, cross_attn_norm=True, qk_norm="rms_norm_across_heads",
                                     eps=1e-6, rope_max_seq_len=64)}
    return {k: {"config": dict(m.config), "state_dict": shapes(m.state_dict())} for k, m in models.items()}


def from_reference():
    """The reference scheduler instance B200SD3_5Adapter.from_reference_adapter reads (attributes) and its schedule for T = 10."""
    from flow_factory.scheduler import FlowMatchEulerDiscreteSDEScheduler as RefFM, set_scheduler_timesteps as ref_set
    s = RefFM(noise_level=0.6, sde_steps=[1, 2, 5], num_sde_steps=2, seed=7, dynamics_type="Dance-SDE", shift=3.0)
    attrs = {"noise_level": s.noise_level, "_sde_steps": s._sde_steps, "_num_sde_steps": s._num_sde_steps, "seed": s.seed,
             "dynamics_type": s.dynamics_type, "config": dict(s.config)}
    ref_set(s, 10, seq_len=64, device="cpu")
    return {"scheduler": attrs, "timesteps": s.timesteps.clone(), "current_sde_steps": s.current_sde_steps.clone()}


def advantage():
    from flow_factory.advantage.advantage_processor import AdvantageProcessor
    nrng = np.random.default_rng(1)
    cases = []
    for _ in range(40):
        n_groups, k = int(nrng.integers(1, 7)), int(nrng.integers(1, 6))
        gid = nrng.permutation(np.repeat(np.arange(n_groups), k))
        keys = ["pick", "ocr", "aes"][: int(nrng.integers(1, 4))]
        rewards = {kk: (nrng.normal(size=len(gid)) if nrng.random() < 0.8 else np.full(len(gid), 0.5)) for kk in keys}
        if nrng.random() < 0.3:
            rewards[keys[0]][gid == 0] = 1.25                       # one group with identical rewards: std clamps
        weights = {kk: float(nrng.choice([1.0, 0.5, 2.0])) for kk in keys}
        c = {"gid": gid, "rewards": rewards, "weights": weights, "sum": {}}
        for global_std in (True, False):
            ap = AdvantageProcessor.__new__(AdvantageProcessor)
            ap.reward_weights, ap.global_std, ap.group_size, ap.group_on_same_rank = weights, global_std, k, False
            ap.collect_group_rewards = lambda samples, rw, gid=gid: ({kk: np.asarray(v, dtype=np.float64) for kk, v in rw.items()}, gid)
            ap._to_local = lambda a: a
            ap._build_weighted_sum_log_data = lambda *a, **kw: {}
            ap._build_gdpo_log_data = lambda *a, **kw: {}
            c["sum"][global_std] = np.asarray(ap.compute_weighted_sum([], rewards, False))
        ap.global_std = True
        c["gdpo"] = np.asarray(ap.compute_gdpo([], rewards, False))
        cases.append(c)
    return cases


def randn():
    from diffusers.utils.torch_utils import randn_tensor
    from flow_factory.utils.base import create_generator_by_prompt
    prompts = ["a cat", "a dog", "a cat"]                        # what GRPOTrainer.evaluate passes (grpo.py:110)
    cpu = torch.device("cpu")
    return {"prompt_seeds": [g.initial_seed() for g in create_generator_by_prompt(prompts, 42)],
            "by_prompt": randn_tensor((3, 4, 2, 2), generator=create_generator_by_prompt(prompts, 42), device=cpu, dtype=torch.bfloat16),
            "one": randn_tensor((2, 5), generator=torch.Generator().manual_seed(3), device=cpu, dtype=torch.float32),
            "list_of_one": randn_tensor((1, 5), generator=[torch.Generator().manual_seed(4)], device=cpu, dtype=torch.float32)}


def main():
    from flow_factory.scheduler.abc import SDESchedulerOutput
    from flow_factory.utils.base import filter_kwargs
    rng = random.Random(0)
    golden = {"adapters": adapters(), "samples": samples(), "trajectory": trajectory(rng), "callback": callback(rng), "scheduler": scheduler(rng),
              "positional": positional(), "vae_host": vae_host(), "intake": intake(), "from_reference": from_reference(), "advantage": advantage(),
              "scheduler_output": _probe(SDESchedulerOutput), "randn_tensor": randn(),
              "filter_kwargs": [sorted(filter_kwargs(f, a=1, b=2, c=3, z=4)) for f in (_f1, _f2, _f3)]}
    buf = io.BytesIO()
    torch.save(golden, buf)
    with lzma.open(os.path.join(HERE, "reference_hooks.pt.xz"), "wb", preset=9) as f:
        f.write(buf.getvalue())


if __name__ == "__main__":
    main()
