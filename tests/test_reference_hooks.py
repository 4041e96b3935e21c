"""The drop-in boundary (SURVEY.md section 8b) checked against the original Flow-Factory project and its vendored diffusers:
* the reference's own plug points resolve this repo's classes - `get_model_adapter_class(<python path>)` (FF/models/registry.py:73-79, what
  `model.model_type: "<path>"` in the YAML goes through) and `register_scheduler` / `get_sde_scheduler_class` (FF/scheduler/registry.py);
* "parameter names are the ABI" (`filter_kwargs`, FF/utils/base.py:38-63): every keyword the reference adapters' `inference()` /
  `forward()` accept is accepted by the B200 adapters, so whatever a trainer passes through `filter_kwargs` arrives.
The reference's side of every comparison is recorded in tests/golden/reference_hooks.pt.xz (tests/golden/make_reference_hooks.py, run
against the original project); this repository's side is computed here.  The checks that run the reference's own classes on this repository's
objects (the glue subclass of SD3_5Adapter, diffusers' attention registry, BaseSample.stack) need the original project's code and run
where oracle/_ref has been laid out (tools/make_oracle_ref.py)."""
import dataclasses
import importlib
import inspect
import io
import json
import lzma
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

from oracle import ref_runner as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_hooks.pt.xz")
needs_reference = pytest.mark.skipif(not R.available(), reason="runs the original project's own classes: oracle/_ref has not been laid out")

ADAPTERS = {"sd3_5": ("flow_factory.models.stable_diffusion.sd3_5.SD3_5Adapter", "flow_factory_b200.adapter.B200SD3_5Adapter"),
            "flux1": ("flow_factory.models.flux.flux1.Flux1Adapter", "flow_factory_b200.flux_adapter.B200Flux1Adapter"),
            "qwen": ("flow_factory.models.qwen_image.qwen_image.QwenImageAdapter", "flow_factory_b200.qwen_adapter.B200QwenImageAdapter"),
            "wan": ("flow_factory.models.wan.wan2_t2v.Wan2_T2V_Adapter", "flow_factory_b200.wan_adapter.B200Wan21Adapter")}
SAMPLES = {"sd3_5": ("flow_factory.models.stable_diffusion.sd3_5", "SD3_5Sample", "SD3_5Sample"),
           "flux1": ("flow_factory.models.flux.flux1", "Flux1Sample", "Flux1Sample"),
           "qwen": ("flow_factory.models.qwen_image.qwen_image", "QwenImageSample", "QwenImageSample"),
           "wan": ("flow_factory.models.wan.wan2_t2v", "WanT2VSample", "WanT2VSample")}


# ------------------------------------------------------------------------------------------------ shared by the golden generator
def _mk_sample(cls, i, prompt):
    kw = dict(timesteps=torch.arange(4.0), all_latents=torch.full((2, 3, 4), float(i)), log_probs=torch.tensor([0.5 * i]),
              latent_index_map=torch.tensor([0, -1, 1, -1, -1]), log_prob_index_map=torch.tensor([-1, 0, -1, -1]), height=64, width=32,
              prompt=prompt, prompt_ids=torch.tensor([1, 2, i]), prompt_embeds=torch.ones(5, 2) * i,
              extra_kwargs={"final_latents": torch.full((3, 4), float(i)), "callback_index_map": None, "tag": {"a": torch.tensor([float(i)])}})
    if "img_ids" in {f.name for f in dataclasses.fields(cls)}:
        kw["img_ids"] = torch.arange(6.0).reshape(2, 3)
    if "img_shapes" in {f.name for f in dataclasses.fields(cls)}:
        kw["img_shapes"] = [(1, 4, 2)]
    return cls(**kw)


def _norm(v):
    if isinstance(v, torch.Tensor): return ["T", list(v.shape), v.flatten().tolist()]
    if isinstance(v, dict): return {k: _norm(x) for k, x in v.items()}
    if isinstance(v, (list, tuple)): return [_norm(x) for x in v]
    return v


def _behaviour(cls):
    """Unique ids, dict views, attribute fall-through and collate of a sample record class on fixed data."""
    rs = [_mk_sample(cls, 1, "a cat"), _mk_sample(cls, 2, "a dog")]
    beh = {"unique_id": [int(x.unique_id) for x in rs],
           "unique_id_ids": int(cls(prompt_ids=torch.tensor([7, 8]), negative_prompt="n").unique_id),
           "to_dict_keys": list(rs[0].to_dict().keys()), "getattr_extra": [_norm(rs[0].final_latents), _norm(rs[0]["tag"])],
           "stack": _norm(cls.stack(rs)), "from_dict": _norm(cls.from_dict(rs[0].to_dict()).to_dict())}
    rs[0].prompt = "changed"
    beh["reset_on_set"] = int(rs[0].unique_id)
    return beh


class _O:
    def __init__(self, i): self.next_latents_mean = torch.full((2, 3), float(i)); self.log_prob = None; self.tag = "s%d" % i


def _probe(cls):
    o = cls.from_dict(dict(next_latents=torch.ones(2), log_prob=torch.zeros(2), noise_pred=torch.full((2,), 3.0), junk=1))
    res = {"keys": list(o.keys()), "len": len(o), "by_key": o["noise_pred"].tolist(), "by_index": o[0].tolist(), "tuple_len": len(o.to_tuple()),
           "iter": list(iter(o)), "contains": ["log_prob" in o, "dt" in o], "attr_none": o.dt is None}
    try:
        o["dt"]; res["missing_key"] = "no error"
    except KeyError:
        res["missing_key"] = "KeyError"
    return res


def _f1(a, b=1): pass
def _f2(a, **kw): pass
def _f3(*args, c=3): pass


# ------------------------------------------------------------------------------------------------ this repository's side
def _resolve(path):
    """The fall-through of both reference registries for a python path (FF/models/registry.py:73-79, FF/scheduler/registry.py:61-64)."""
    module_path, name = path.rsplit(".", 1)
    return getattr(importlib.import_module(module_path), name)


class _Config(dict):
    """A model's `config` as diffusers hands it over (FrozenDict): a mapping with attribute access."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k) from None


def _model(rec):
    """Stand-in for a real (tiny) diffusers model: its recorded config and a state dict of its recorded keys and shapes."""
    sd = {k: torch.zeros(s) for k, s in rec["state_dict"].items()}
    return types.SimpleNamespace(config=_Config(rec["config"]), state_dict=lambda: dict(sd))


def _against_golden(G):
    from flow_factory_b200 import advantage as MyAdv, flux as MF, qwen as MQ, vae as MV, wan as MW
    import flow_factory_b200.adapter as MA
    from flow_factory_b200.adapter import filter_kwargs as my_filter
    from flow_factory_b200.rng import randn_tensor as my_randn
    from flow_factory_b200.scheduler import (FlowMatchEulerDiscreteSDEScheduler as MyFM, SDESchedulerOutput as MyOut,
                                             UniPCMultistepSDEScheduler as MyUP, calculate_shift as my_shift)
    from flow_factory_b200.trajectory import compute_trajectory_indices as my_cti, create_callback_collector as my_cb, plan_slots
    from flow_factory_b200.weights import EngineConfig, PackedWeights
    out = {}
    for name, (_, my_path) in ADAPTERS.items():
        mine = _resolve(my_path)
        rec = {"resolved": mine.__module__ + "." + mine.__name__}
        for fn in ("inference", "forward"):
            rp = G["adapters"][name][fn]
            mp = [p for p in inspect.signature(getattr(mine, fn)).parameters if p != "self"]
            rec[fn + "_missing"] = [p for p in rp if p not in mp]
            rec[fn + "_filtered"] = sorted(my_filter(getattr(mine, fn), **{p: 0 for p in rp})) == sorted(p for p in rp if p in mp)
        out[name] = rec
    mine_mod = importlib.import_module("flow_factory_b200.samples")
    for name, (_, _, my_cls) in SAMPLES.items():
        ref, M = G["samples"][name], getattr(mine_mod, my_cls)
        out[name]["sample_fields_missing"] = sorted(set(ref["fields"]) ^ {f.name for f in dataclasses.fields(M)})
        out[name]["shared_fields"] = [ref["shared_fields"], sorted(M.shared_fields())]
        rb, mb = ref["behaviour"], _behaviour(M)
        beh = {k: [rb[k], mb[k]] for k in mb}
        beh["getattr_extra"] = [rb["getattr_extra"][0], mb["getattr_extra"][0], rb["getattr_extra"][1], mb["getattr_extra"][1]]
        out[name]["behaviour"] = beh
    # ---- trajectory bookkeeping: plan_slots vs the reference's two collectors driven as in sd3_5.py:266-304, on randomised index specs
    mism = []
    for c in G["trajectory"]:
        T, idx, has_lp, ref = c["T"], c["idx"], c["has_lp"], c["ref"]
        if c["cti"] is not None:
            tr, inc, ref_idx = c["cti"]
            if ref_idx != my_cti(tr, T, include_initial=inc): mism.append(("cti", T, tr, inc))
        if ref is None:                                     # the reference raised on this spec
            try:
                plan_slots(idx, T, has_lp); mism.append(("ref raised, mine did not", T, idx))
            except Exception:
                pass
            continue
        lat_slot, lp_slot, lat_map, lp_map = plan_slots(idx, T, has_lp)
        n_lat, n_lp = sum(1 for x in lat_slot if x >= 0), sum(1 for x in lp_slot if x >= 0)
        ok = ref["n_lat"] == n_lat and ref["n_lp"] == n_lp
        for mine, r in ((lat_map, ref["lat_map"]), (lp_map, ref["lp_map"])):
            ok = ok and ((mine is None) == (r is None)) and (mine is None or torch.equal(mine, r))
        if not ok: mism.append((c["kind"], T, idx, has_lp))
    for c in G["callback"]:
        T, ref = c["T"], c["ref"]
        b_ = my_cb(c["idx"], T)
        for i in range(T):
            b_.collect_step(i, _O(i), c["keys"], {"noise_level": 0.7 if i % 2 else None})
        ra, rb = ref["result"], b_.get_result()
        ok = list(ra.keys()) == list(rb.keys()) and ref["len"] == len(b_) and ref["collected_indices"] == b_.collected_indices and ref["is_disabled"] == b_.is_disabled
        for k in ra:
            ok = ok and (torch.equal(ra[k], rb[k]) if isinstance(ra[k], torch.Tensor) else ra[k] == rb[k])
        ma, mb = ref["index_map"], b_.get_index_map()
        ok = ok and ((ma is None) == (mb is None)) and (ma is None or torch.equal(ma, mb))
        if not ok: mism.append(("callback", T, c["idx"], c["keys"]))
    out["trajectory_mismatches"] = [repr(m) for m in mism[:5]]
    # ---- scheduler mirrors: schedule, SDE-step selection and per-step scalars vs the reference on randomised settings
    smis = []
    for case, c in enumerate(G["scheduler"]):
        T, ref = c["T"], c["ref"]
        if c["cls"] == "FlowMatch":
            m = MyFM(noise_level=c["nl"], sde_steps=c["sde"], num_sde_steps=c["nsde"], seed=c["seed"], dynamics_type=c["dyn"], **c["kw"])
            mt = m.set_timesteps(T, seq_len=c["seq"])
        else:
            m = MyUP(noise_level=c["nl"], sde_steps=c["sde"], num_sde_steps=c["nsde"], seed=c["seed"], dynamics_type=c["dyn"], flow_shift=c["fs"])
            mt = m.set_timesteps(T)
        m.rollout()
        rt = ref["timesteps"]
        ok = torch.equal(rt, mt) and torch.equal(ref["sigmas"], m.sigmas)
        ok = ok and torch.equal(ref["sde_steps"], m.sde_steps) and ref["num_sde_steps"] == m.num_sde_steps and torch.equal(ref["current_sde_steps"], m.current_sde_steps)
        ok = ok and torch.equal(ref["noise_levels"], m.get_noise_levels().float()) and torch.equal(ref["train_timesteps"], torch.as_tensor(m.train_timesteps))
        i = c["i"]
        t, tn = rt[i], (rt[i + 1] if i + 1 < T else torch.tensor(0, dtype=rt.dtype))
        cur = ref["noise_level_t"]
        ok = ok and cur == m.get_noise_level_for_timestep(t) and ref["index_t"] == m.index_for_timestep(t)
        co = m.step_coef(t, tn, cur, compute_log_prob=False)
        ok = ok and ref["dt"] == co.dt and ref["std_dev_t"] == co.std_dev_t
        # timestep_next omitted: the reference reads sigmas[i], sigmas[i + 1] from its tables (FlowMatch only: UniPC reads an integer timestep as an index)
        if c["cls"] == "FlowMatch":
            c2 = m.step_coef(t, None, cur, compute_log_prob=False)
            ok = ok and ref["dt_no_next"] == c2.dt and ref["std_dev_t_no_next"] == c2.std_dev_t
        if not ok: smis.append((case, T, c["dyn"], c["nsde"], c["sde"], c["seed"], c["cls"]))
    out["scheduler_mismatches"] = [repr(m) for m in smis[:5]]
    # ---- positional tables and latent packing vs the real diffusers modules
    P, pos = G["positional"], {}
    h2, w2, nt = 6, 10, 7
    mc, ms_ = MF.rope_tables(torch.cat([torch.zeros(nt, 3), MF.latent_image_ids(h2, w2)], 0), (16, 56, 56))
    pos["flux_rope"] = bool(torch.equal(P["flux_cos"], mc) and torch.equal(P["flux_sin"], ms_))
    pos["flux_pack"] = bool(torch.equal(P["flux_packed"], MF.pack_latents(P["flux_lat"])))
    pos["shift"] = [P["shift"][n] == my_shift(n) for n in (256, 1024, 4096, 4429)]
    qc, qs = MQ.qwen_rope_tables(h2, w2, nt, (16, 56, 56))
    pos["qwen_rope"] = bool(torch.equal(P["qwen"].real.float().repeat_interleave(2, 1), qc) and torch.equal(P["qwen"].imag.float().repeat_interleave(2, 1), qs))
    mwc, mws = MW.wan_rope_tables(MW.WanEngineConfig(rope_max_seq_len=64), 3, 4, 5, table_dtype=torch.float32)
    pos["wan_rope"] = bool(torch.equal(P["wan_cos"].reshape(60, 128), mwc) and torch.equal(P["wan_sin"].reshape(60, 128), mws))
    mwcb, mwsb = MW.wan_rope_tables(MW.WanEngineConfig(rope_max_seq_len=64), 3, 4, 5)
    pos["wan_rope_bf16"] = bool(P["wan_cos_bf16"].dtype == torch.bfloat16 and torch.equal(P["wan_cos_bf16"].float().reshape(60, 128), mwcb)
                                and torch.equal(P["wan_sin_bf16"].float().reshape(60, 128), mwsb))
    out["positional"] = pos
    # ---- VAE host side against the real AutoencoderKL / VaeImageProcessor
    V = G["vae_host"]
    vm = _model(V)
    vcfg = MV.VaeDecoderConfig.from_config(vm.config)
    packed = MV.pack_vae_decoder_weights(vm.state_dict(), vcfg)
    vae_rec = {"cfg": [vcfg.latent_channels, list(vcfg.block_out_channels), vcfg.layers_per_block, vcfg.norm_num_groups, vcfg.scaling_factor, vcfg.shift_factor],
               "n_packed": [len(packed), MV.expected_weight_count(vcfg)],
               "postprocess": bool(torch.equal(V["postprocessed"], MV.postprocess_pt(V["img"])))}
    try:
        MV.VaeDecoderConfig.from_config(_Config(V["default_config"])); vae_rec["post_quant_guard"] = "no error"
    except NotImplementedError:
        vae_rec["post_quant_guard"] = "NotImplementedError"
    out["vae_host"] = vae_rec
    # ---- config intake + weight packing from REAL (tiny) diffusers transformers: every key the packers read exists in the real state dicts
    cpu = torch.device("cpu")
    I, intake = G["intake"], {}
    m = _model(I["sd3"])
    c = EngineConfig.from_model_config(m.config)
    pw = PackedWeights(c, m.state_dict(), cpu)
    intake["sd3"] = [c.num_layers, c.num_heads, c.num_dual_layers, len(pw.tensors) > 0]
    m = _model(I["flux"])
    c = MF.FluxEngineConfig.from_model_config(m.config)
    pw = MF.FluxPackedWeights(c, m.state_dict(), cpu)
    intake["flux"] = [c.num_layers, c.num_single_layers, c.num_heads, bool(c.guidance_embeds), pw.mod_rows == (12 + 3 + 2) * 256]
    m = _model(I["qwen"])
    c = MQ.qwen_engine_config(m.config)
    pw = MF.FluxPackedWeights(c, m.state_dict(), cpu)
    intake["qwen"] = [c.num_layers, c.variant, c.num_heads, len(pw.tensors) > 0]
    m = _model(I["wan"])
    c = MW.WanEngineConfig.from_model_config(m.config)
    g_, layers_ = MW.pack_wan_state_dict(c, m.state_dict())
    intake["wan"] = [c.num_layers, c.num_attention_heads, c.ffn_dim, list(g_["pe_w"].shape), len(layers_)]
    out["intake"] = intake
    # ---- B200SD3_5Adapter.from_reference_adapter fed with the reference objects' recorded state (engine stubbed: no GPU here)
    F = G["from_reference"]

    class _Eng:
        def __init__(self, model_config, state_dict, device):
            self.device, self.cfg, self.n_keys = torch.device("cpu"), EngineConfig.from_model_config(model_config), len(state_dict)
    ra = types.SimpleNamespace(transformer=_model(I["sd3"]), scheduler=types.SimpleNamespace(**F["scheduler"]), device="cpu",
                               decode_latents=lambda lat, output_type="pt": lat * 0 + 0.5)
    engine_cls, MA.RolloutEngine = MA.RolloutEngine, _Eng
    try:
        b = MA.B200SD3_5Adapter.from_reference_adapter(ra, rng="torch")
    finally:
        MA.RolloutEngine = engine_cls
    b.scheduler.set_timesteps(10, seq_len=64)
    out["from_reference"] = {"cfg": [b.model_config.num_layers, b.model_config.num_heads], "n_keys": b.engine.n_keys == len(I["sd3"]["state_dict"]),
                             "sched": [b.scheduler.noise_level, b.scheduler.dynamics_type, b.scheduler.seed, b.scheduler.num_sde_steps, b.scheduler.sde_steps.tolist()],
                             "timesteps_equal": bool(torch.equal(F["timesteps"], b.scheduler.timesteps)),
                             "sde_equal": bool(torch.equal(F["current_sde_steps"], b.scheduler.current_sde_steps)),
                             "decode": float(b.decode_latents(torch.zeros(1, 2)).mean())}
    # ---- GRPO / GDPO advantage arithmetic (FF/advantage/advantage_processor.py:314-481) on randomised groups, incl. constant-reward groups
    amis = []
    for case, c in enumerate(G["advantage"]):
        for global_std in (True, False):
            m_sum = MyAdv.advantages_sum(c["rewards"], c["weights"], c["gid"], global_std=global_std)
            if not np.allclose(c["sum"][global_std], np.asarray(m_sum), rtol=1e-12, atol=1e-12): amis.append(("sum", case, global_std))
        if not np.allclose(c["gdpo"], np.asarray(MyAdv.advantages_gdpo(c["rewards"], c["weights"], c["gid"])), rtol=1e-12, atol=1e-12):
            amis.append(("gdpo", case))
    out["advantage_mismatches"] = [repr(m) for m in amis[:5]]
    out["scheduler_output"] = [G["scheduler_output"], _probe(MyOut)]
    # ---- initial latents from per-prompt CPU generator lists (the seeds the reference's create_generator_by_prompt derives)
    Rn = G["randn_tensor"]
    gens = lambda: [torch.Generator().manual_seed(s) for s in Rn["prompt_seeds"]]
    rr = [bool(torch.equal(Rn["by_prompt"], my_randn((3, 4, 2, 2), generator=gens(), device="cpu", dtype=torch.bfloat16))),
          bool(torch.equal(Rn["one"], my_randn((2, 5), generator=torch.Generator().manual_seed(3), device="cpu", dtype=torch.float32))),
          bool(torch.equal(Rn["list_of_one"], my_randn((1, 5), generator=[torch.Generator().manual_seed(4)], device="cpu", dtype=torch.float32)))]
    g3 = gens()
    rr.append(bool(torch.equal(my_randn((3, 2), generator=g3, dtype=torch.float32)[0], my_randn((3, 2), generator=gens(), dtype=torch.float32)[2])))  # same prompt, same noise
    out["randn_tensor"] = rr
    out["filter_kwargs"] = [G["filter_kwargs"], [sorted(my_filter(f, a=1, b=2, c=3, z=4)) for f in (_f1, _f2, _f3)]]
    out["sched"] = [_resolve("flow_factory_b200.scheduler.FlowMatchEulerDiscreteSDEScheduler").__module__,
                    _resolve("flow_factory_b200.scheduler.UniPCMultistepSDEScheduler").__module__]
    return json.loads(json.dumps(out))


@pytest.fixture(scope="module")
def hooks():
    with lzma.open(GOLDEN) as f:
        return _against_golden(torch.load(io.BytesIO(f.read()), weights_only=False))


# ------------------------------------------------------------------------------------------------ the reference's own classes on this repo's objects
_SCRIPT = r'''
import importlib, json, sys
sys.path[:0] = [sys.argv[2], sys.argv[1]]
import torch
from diffusers.models.transformers.transformer_sd3 import SD3Transformer2DModel
from diffusers.models.transformers.transformer_flux import FluxTransformer2DModel
from flow_factory.samples import BaseSample as RefBase
from flow_factory.scheduler import FlowMatchEulerDiscreteSDEScheduler as RefFM, set_scheduler_timesteps as ref_set
from flow_factory_b200.weights import EngineConfig
from tests.test_reference_hooks import SAMPLES, _mk_sample, _norm
out = {"ref_stack_on_mine": {}}
mine_mod = importlib.import_module("flow_factory_b200.samples")
for name, (mod, ref_cls, my_cls) in SAMPLES.items():
    R, M = getattr(importlib.import_module(mod), ref_cls), getattr(mine_mod, my_cls)
    rs, ms = [_mk_sample(R, 1, "a cat"), _mk_sample(R, 2, "a dog")], [_mk_sample(M, 1, "a cat"), _mk_sample(M, 2, "a dog")]
    out["ref_stack_on_mine"][name] = _norm(RefBase.stack(ms)) == _norm(R.stack(rs))
# ---- B200SD3_5Adapter.from_reference_adapter fed with real reference objects (engine stubbed: no GPU here)
import flow_factory_b200.adapter as MA
class _Eng:
    def __init__(self, model_config, state_dict, device):
        self.device, self.cfg, self.n_keys = torch.device("cpu"), EngineConfig.from_model_config(model_config), len(state_dict)
MA.RolloutEngine = _Eng
class _RefAdapter:                                   # the attributes from_reference_adapter reads off a flow_factory SD3_5Adapter
    pass
ra = _RefAdapter()
ra.transformer = SD3Transformer2DModel(sample_size=16, patch_size=2, in_channels=16, num_layers=2, attention_head_dim=64, num_attention_heads=2,
                                       joint_attention_dim=64, caption_projection_dim=128, pooled_projection_dim=32, out_channels=16,
                                       pos_embed_max_size=16, dual_attention_layers=(0,), qk_norm="rms_norm")
ra.scheduler = RefFM(noise_level=0.6, sde_steps=[1, 2, 5], num_sde_steps=2, seed=7, dynamics_type="Dance-SDE", shift=3.0)
ra.device = "cpu"
ra.decode_latents = lambda lat, output_type="pt": lat * 0 + 0.5
b = MA.B200SD3_5Adapter.from_reference_adapter(ra, rng="torch")
ref_set(ra.scheduler, 10, seq_len=64, device="cpu"); b.scheduler.set_timesteps(10, seq_len=64)
# ---- the reference-side glue file (integration/ff_b200_glue.py, quoted by INTEGRATION.md) driven with the heavy base-class parts stubbed
sys.path.insert(0, sys.argv[1] + "/integration")
import ff_b200_glue as GL
import flow_factory.models.abc as ABC
glue = GL.B200GlueSD3_5Adapter.__new__(GL.B200GlueSD3_5Adapter)
GL.B200GlueSD3_5Adapter.transformer = property(lambda self: ra.transformer)
GL.B200GlueSD3_5Adapter.device = property(lambda self: "cpu")
import types
glue.pipeline = types.SimpleNamespace(scheduler=ra.scheduler)        # BaseAdapter.scheduler is a property over pipeline.scheduler
glue.decode_latents = ra.decode_latents
glue._mode = "train"
GL.B200GlueSD3_5Adapter.trainable_component_names = property(lambda self: [])   # BaseAdapter.eval / rollout / train loop over these
glue._b200 = MA.B200SD3_5Adapter.from_reference_adapter(glue, rng="torch")
ra.scheduler.set_seed(123)
def _refresh(self, sd):
    self.refreshed = getattr(self, "refreshed", 0) + 1
    self.last_sd = {k: v.detach().clone() for k, v in sd.items()}
_Eng.refresh_weights = _refresh
glue.rollout()
stale_after_rollout = glue._engine_stale
glue._sync_engine_if_stale()                          # what inference() / the no-grad forward() do first
g1 = [glue.mode, glue._b200.scheduler.seed, glue._b200.scheduler.is_eval, ra.scheduler.is_eval, glue._b200.engine.refreshed]
# ---- weight-swapping contexts (ADVICE r1: the KL-reference / EMA forward must run on the swapped weights, grpo.py:282, nft.py:360)
from flow_factory.ema import EMAModuleWrapper
params = list(ra.transformer.parameters())
GL.B200GlueSD3_5Adapter.get_trainable_parameters = lambda self: params
GL.B200GlueSD3_5Adapter.target_module_map = property(lambda self: {})
glue.model_args = types.SimpleNamespace(lora_alpha=8.0, finetune_type="full")
glue.ema_wrapper = EMAModuleWrapper(parameters=params, decay=0.5, update_step_interval=1, device="cpu")
glue._ref_ema = EMAModuleWrapper(parameters=params, decay=0.0, update_step_interval=0, device="cpu")
key = "proj_out.bias"
with torch.no_grad():
    for e in glue.ema_wrapper.ema_parameters: e.fill_(0.25)          # the EMA policy
    for e in glue._ref_ema.ema_parameters: e.fill_(-0.5)             # theta_ref
    for q in params: q.fill_(1.0)                                     # the current policy (an optimizer step happened)
glue._b200.forward = lambda *a, **k: float(glue._b200.engine.last_sd[key].mean())   # stand-in: reports which weights the engine holds
glue.rollout()
ctx = {}
with torch.no_grad():
    ctx["policy"] = glue.forward()
    with glue.use_ref_parameters():
        ctx["ref"] = glue.forward()
        ctx["ref_again_refreshes"] = glue._b200.engine.refreshed
        glue.forward()
        ctx["ref_again_refreshes"] = glue._b200.engine.refreshed - ctx["ref_again_refreshes"]
    ctx["after_ref"] = glue.forward()
    with glue.use_ema_parameters():
        ctx["ema"] = glue.forward()
        with glue.use_ref_parameters():
            ctx["ema_then_ref"] = glue.forward()
        ctx["back_in_ema"] = glue.forward()
    ctx["after_ema"] = glue.forward()
    ctx["module_restored"] = float(dict(ra.transformer.named_parameters())[key].mean())
# train mode: the optimizer steps between no-grad calls without any context edge
glue.train(True)
with torch.no_grad():
    for q in params: q.fill_(2.0)
    ctx["train_mode_tracks_optimizer"] = glue.forward()
    for q in params: q.fill_(1.0)
# ---- LoRA (finetune_type='lora'): PEFT key names at post_init time, adapter folded for the policy, NOT folded inside use_ref_parameters
import torch.nn as nn
class _LoraLinear(nn.Module):                           # PEFT's lora.Linear layout: base_layer + lora_A / lora_B ModuleDicts keyed by adapter name
    def __init__(self, base, r):
        super().__init__()
        self.base_layer = base
        self.lora_A = nn.ModuleDict({"default": nn.Linear(base.in_features, r, bias=False)})
        self.lora_B = nn.ModuleDict({"default": nn.Linear(r, base.out_features, bias=False)})
class _PeftLike(nn.Module):                             # PeftModel(base_model=LoraModel(model=transformer)) -> keys 'base_model.model.<...>'
    def __init__(self, model):
        super().__init__()
        self.base_model = nn.Module(); self.base_model.model = model
        self.config = model.config
tr2 = SD3Transformer2DModel(sample_size=16, patch_size=2, in_channels=16, num_layers=2, attention_head_dim=64, num_attention_heads=2,
                            joint_attention_dim=64, caption_projection_dim=128, pooled_projection_dim=32, out_channels=16,
                            pos_embed_max_size=16, dual_attention_layers=(0,), qk_norm="rms_norm")
base_q = tr2.transformer_blocks[0].attn.to_q.weight.detach().clone()
tr2.transformer_blocks[0].attn.to_q = _LoraLinear(tr2.transformer_blocks[0].attn.to_q, r=4)
with torch.no_grad():
    tr2.transformer_blocks[0].attn.to_q.lora_A["default"].weight.fill_(0.5)
    tr2.transformer_blocks[0].attn.to_q.lora_B["default"].weight.fill_(0.25)
peft_like = _PeftLike(tr2)
GL.B200GlueSD3_5Adapter.transformer = property(lambda self: peft_like)
glue.model_args = types.SimpleNamespace(lora_alpha=8.0, finetune_type="lora")
lora = {"peft_keys": sorted(k for k in peft_like.state_dict() if "to_q" in k and "transformer_blocks.0.attn." in k)}
built = MA.B200SD3_5Adapter.from_reference_adapter(glue, rng="torch")          # what post_init does; raised KeyError before the fix
lora["post_init_plain_keys"] = built.engine.n_keys == len(ra.transformer.state_dict())
qk = "transformer_blocks.0.attn.to_q.weight"
glue._b200.forward = lambda *a, **k: float((glue._b200.engine.last_sd[qk] - base_q).abs().max())
glue.rollout()
with torch.no_grad():
    lora["policy_delta"] = glue.forward()              # (alpha / r) * B A = 2 * (0.25 * 0.5 * 4) = 1.0 on every entry
    with glue.use_ref_parameters():
        lora["ref_delta"] = glue.forward()             # adapter disabled: base weights
    lora["after_delta"] = glue.forward()
lora["plain_keys_only"] = not any(("lora_" in k) or ("base_layer" in k) or k.startswith("base_model.") for k in glue._b200.engine.last_sd)
GL.B200GlueSD3_5Adapter.transformer = property(lambda self: ra.transformer)
glue.model_args = types.SimpleNamespace(lora_alpha=8.0, finetune_type="full")
glue.rollout(); glue._sync_engine_if_stale()
# ---- option (b) of SURVEY 7.2 #1: old_log_prob of the stored SDE transitions re-evaluated through the REFERENCE forward
from flow_factory_b200.samples import SD3_5Sample as MySample
from flow_factory_b200.scheduler import SDESchedulerOutput as MyOut
def _mk(b):
    # T = 4: latents kept at positions 0, 1, 2, 4 (slots 0..3); log-probs kept for steps 0, 1 (slots 0, 1) and step 3 (slot 2), whose start
    # latent (position 3) is NOT stored
    return MySample(timesteps=torch.tensor([1000.0, 900.0, 750.0, 500.0]), all_latents=torch.arange(4.0).view(4, 1, 1, 1) + 10 * b,
                    log_probs=torch.full((3,), -1.0), latent_index_map=torch.tensor([0, 1, 2, -1, 3]), log_prob_index_map=torch.tensor([0, 1, -1, 2]))
fake = [_mk(0), _mk(1)]
glue._b200.inference = lambda *a, **k: fake
calls_b = []
def _ref_forward(self, **kw):
    calls_b.append({"t": float(kw["t"]), "t_next": float(kw["t_next"]), "x_t": kw["latents"].flatten().tolist(), "x_n": kw["next_latents"].flatten().tolist(),
                    "g": kw["guidance_scale"], "rk": kw["return_kwargs"], "nl": kw["noise_level"], "pe": kw["prompt_embeds"].shape[0]})
    return MyOut(log_prob=torch.tensor([100.0 + kw["latents"].flatten()[0].item(), 200.0 + kw["latents"].flatten()[1].item()]))
GL.SD3_5Adapter.forward = _ref_forward
ra.scheduler.get_noise_level_for_timestep = lambda t: 0.7
glue._mode = "rollout"
res = glue.inference(prompt_embeds=torch.zeros(2, 3, 4), pooled_prompt_embeds=torch.zeros(2, 4), guidance_scale=4.5, compute_log_prob=True)
rec = {"calls": calls_b, "log_probs": [s_.log_probs.tolist() for s_ in res]}
glue.recompute_old_log_probs = False
fake[0].log_probs.fill_(-1.0); n_before = len(calls_b)
glue.inference(prompt_embeds=torch.zeros(2, 3, 4), pooled_prompt_embeds=torch.zeros(2, 4), guidance_scale=4.5, compute_log_prob=True)
rec["disabled_keeps_engine_values"] = [len(calls_b) == n_before, fake[0].log_probs.tolist()]
out["glue_contexts"] = {"stale_after_rollout": stale_after_rollout, "ctx": ctx, "lora": lora, "recompute": rec}
glue.eval()
g2 = [glue.mode, glue._b200.scheduler.is_eval, ra.scheduler.is_eval]
glue.train(True)
g3 = [glue.mode, glue._b200.scheduler.is_eval]
out["glue"] = [g1, g2, g3, [c.__name__ for c in GL.B200GlueSD3_5Adapter.__mro__[:3]]]
# ---- diffusers' own attention plug points (SURVEY 8b ii / iii) with the real vendored classes; the kernels need a GPU, so the native forward
# is replaced by an SDPA stand-in HERE and everything around it (registry slot, dispatch, (B,S,H,D) layout, scale, the SD3 processor's joint
# [image ; text] order, output split, to_out / to_add_out, autograd) is the shipped code
import flow_factory_b200.diffusers_hooks as DH
from diffusers.models.attention_dispatch import AttentionBackendName, _AttentionBackendRegistry as REG, dispatch_attention_fn
import torch.nn.functional as F
hk = {}
try:
    dispatch_attention_fn(torch.zeros(1, 4, 2, 64), torch.zeros(1, 4, 2, 64), torch.zeros(1, 4, 2, 64), backend=DH.install_attention_backend("_native_flash"))
    hk["cpu_call_raises"] = False
except RuntimeError as e:
    hk["cpu_call_raises"] = "CUDA tensors only" in str(e)                  # dispatch reached OUR function, which has no CPU path
hk["slot"] = [REG._backends[AttentionBackendName._NATIVE_FLASH] is DH.b200_attention_backend,
              sorted(REG._supported_arg_names[AttentionBackendName._NATIVE_FLASH]) == sorted(REG._supported_arg_names[AttentionBackendName.NATIVE]),
              REG._constraints[AttentionBackendName._NATIVE_FLASH] == []]
calls = []
def _stand_in(q, k, v, scale):
    calls.append((tuple(q.shape), tuple(k.shape), scale))
    return F.scaled_dot_product_attention(q.permute(0, 2, 1, 3), k.permute(0, 2, 1, 3), v.permute(0, 2, 1, 3), scale=scale).permute(0, 2, 1, 3)
DH._forward_native = _stand_in
DH._check_device_dtype = lambda q, k, v: None
torch.manual_seed(0)
fl = FluxTransformer2DModel(patch_size=1, in_channels=16, num_layers=1, num_single_layers=1, attention_head_dim=64, num_attention_heads=2,
                            joint_attention_dim=32, pooled_projection_dim=16, guidance_embeds=True, axes_dims_rope=(8, 28, 28)).eval()
fin = dict(hidden_states=torch.randn(2, 12, 16), encoder_hidden_states=torch.randn(2, 5, 32), pooled_projections=torch.randn(2, 16),
           timestep=torch.tensor([0.5, 0.5]), img_ids=torch.zeros(12, 3), txt_ids=torch.zeros(5, 3), guidance=torch.tensor([3.5, 3.5]))
with torch.no_grad():
    base = fl(**fin).sample
    fl.set_attention_backend("_native_flash")            # what model.attn_backend: "_native_flash" does (FF/models/abc.py:782-798)
    n0 = len(calls)
    hooked = fl(**fin).sample
hk["flux_calls"] = len(calls) - n0
hk["flux_shapes"] = [list(calls[-1][0]), calls[-1][2]]
hk["flux_max_diff"] = float((base - hooked).abs().max())
# autograd through the backend function: native forward, gradients from the SDPA recomputation
q = torch.randn(1, 6, 2, 64, requires_grad=True); k = torch.randn(1, 6, 2, 64, requires_grad=True); v = torch.randn(1, 6, 2, 64, requires_grad=True)
o = DH.b200_attention_backend(q, k, v, scale=0.2); o.square().sum().backward()
q2, k2, v2 = (t.detach().clone().requires_grad_(True) for t in (q, k, v))
o2 = F.scaled_dot_product_attention(q2.permute(0, 2, 1, 3), k2.permute(0, 2, 1, 3), v2.permute(0, 2, 1, 3), scale=0.2).permute(0, 2, 1, 3); o2.square().sum().backward()
hk["grad_max_diff"] = max(float((a.grad - b.grad).abs().max()) for a, b in ((q, q2), (k, k2), (v, v2)))
rej = []
for kw in (dict(attn_mask=torch.ones(1, 6, dtype=torch.bool)), dict(is_causal=True), dict(dropout_p=0.1), dict(return_lse=True), dict(enable_gqa=True)):
    try:
        DH.b200_attention_backend(q.detach(), k.detach(), v.detach(), **kw); rej.append(False)
    except (NotImplementedError, ValueError):
        rej.append(True)
hk["unsupported_arguments_raise"] = rej
DH.uninstall_attention_backend("_native_flash")
hk["uninstalled"] = REG._backends[AttentionBackendName._NATIVE_FLASH] is not DH.b200_attention_backend
fl.reset_attention_backend()
# the SD3 processor on a real SD3Transformer2DModel (dual-attention block 0 + a context_pre_only last block)
sd = SD3Transformer2DModel(sample_size=16, patch_size=2, in_channels=16, num_layers=2, attention_head_dim=64, num_attention_heads=2,
                           joint_attention_dim=64, caption_projection_dim=128, pooled_projection_dim=32, out_channels=16,
                           pos_embed_max_size=16, dual_attention_layers=(0,), qk_norm="rms_norm").eval()
sin = dict(hidden_states=torch.randn(2, 16, 8, 8), encoder_hidden_states=torch.randn(2, 7, 64), pooled_projections=torch.randn(2, 32),
           timestep=torch.tensor([500.0, 500.0]))
with torch.no_grad():
    base = sd(**sin).sample
    proc = DH.install_sd3_attn_processor(sd)
    n0 = len(calls)
    hooked = sd(**sin).sample
hk["sd3_processors"] = sorted({type(p_).__name__ for p_ in sd.attn_processors.values()})
hk["sd3_calls"] = len(calls) - n0                       # block 0: joint + attn2, block 1: joint
hk["sd3_joint_len"] = sorted({c[0][1] for c in calls[n0:]})
hk["sd3_max_diff"] = float((base - hooked).abs().max())
import inspect as _insp
from diffusers.models.attention_processor import JointAttnProcessor2_0
hk["sd3_signature"] = list(_insp.signature(DH.B200JointAttnProcessor.__call__).parameters)[:5] == list(_insp.signature(JointAttnProcessor2_0.__call__).parameters)[:5]
out["diffusers_hooks"] = hk
print("RESULT " + json.dumps(out))
'''


@pytest.fixture(scope="module")
def live():
    r = subprocess.run([sys.executable, "-c", _SCRIPT, ROOT, R.REF_DIR], capture_output=True, text=True, timeout=600)
    lines = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
    assert lines, r.stdout[-2000:] + r.stderr[-4000:]
    return json.loads(lines[-1][7:])


def test_registry_resolves_b200_adapters_by_python_path(hooks):
    assert hooks["sd3_5"]["resolved"] == "flow_factory_b200.adapter.B200SD3_5Adapter"
    assert hooks["flux1"]["resolved"] == "flow_factory_b200.flux_adapter.B200Flux1Adapter"
    assert hooks["qwen"]["resolved"] == "flow_factory_b200.qwen_adapter.B200QwenImageAdapter"
    assert hooks["wan"]["resolved"] == "flow_factory_b200.wan_adapter.B200Wan21Adapter"
    assert hooks["sched"] == ["flow_factory_b200.scheduler", "flow_factory_b200.scheduler"]


@pytest.mark.parametrize("model", ["sd3_5", "flux1", "qwen", "wan"])
def test_keyword_abi_is_a_superset_of_the_reference(hooks, model):
    rec = hooks[model]
    assert rec["inference_missing"] == [], rec
    assert rec["forward_missing"] == [], rec
    assert rec["inference_filtered"] and rec["forward_filtered"]


@pytest.mark.parametrize("model", ["sd3_5", "flux1", "qwen", "wan"])
def test_sample_records_carry_the_reference_fields(hooks, model):
    rec = hooks[model]
    assert rec["shared_fields"][0] == rec["shared_fields"][1], rec["shared_fields"]      # what stack() collates as one value per batch
    assert rec["sample_fields_missing"] == [], rec["sample_fields_missing"]            # every field of the reference record exists


@pytest.mark.parametrize("model", ["sd3_5", "flux1", "qwen", "wan"])
def test_sample_records_behave_like_the_reference(hooks, model):
    """Same data into the reference record and the B200 record: identical ids, dict views, extra_kwargs fall-through and collate."""
    beh = hooks[model]["behaviour"]
    assert beh["unique_id"][0] == beh["unique_id"][1] and beh["unique_id"][0][0] != beh["unique_id"][0][1]
    assert beh["unique_id_ids"][0] == beh["unique_id_ids"][1]
    assert beh["to_dict_keys"][0] == beh["to_dict_keys"][1]
    assert beh["getattr_extra"][0] == beh["getattr_extra"][1] and beh["getattr_extra"][2] == beh["getattr_extra"][3]
    assert beh["stack"][0] == beh["stack"][1]
    assert beh["from_dict"][0] == beh["from_dict"][1]
    assert beh["reset_on_set"][0] == beh["reset_on_set"][1]


@needs_reference
def test_reference_stack_accepts_b200_records(live):
    """The reference's own `BaseSample.stack` (what the trainers call) accepts B200 records and returns the batch it builds from its own."""
    assert live["ref_stack_on_mine"] == {"sd3_5": True, "flux1": True, "qwen": True, "wan": True}


def test_trajectory_bookkeeping_matches_the_reference_collectors(hooks):
    """300 randomised (T, trajectory_indices, SDE-step) cases: stored-latent / log-prob counts and both index maps equal what the
    reference's TrajectoryCollector pair produces when driven like SD3_5Adapter.inference."""
    assert hooks["trajectory_mismatches"] == []


def test_scheduler_mirrors_match_the_reference_on_random_settings(hooks):
    """60 randomised settings of both scheduler mirrors: timesteps, sigmas, SDE-step selection under the seed, noise levels, index lookup
    and the per-step scalars (dt, std_dev_t of the reference's step) - all bit-exact."""
    assert hooks["scheduler_mismatches"] == []


def test_filter_kwargs_mirror(hooks):
    assert hooks["filter_kwargs"][0] == hooks["filter_kwargs"][1]


def test_scheduler_output_mapping_protocol(hooks):
    """`output['noise_pred']` (NFT / AWM / CRD trainers), `output[0]`, keys / iteration over the non-None fields - as diffusers' BaseOutput."""
    assert hooks["scheduler_output"][0] == hooks["scheduler_output"][1]


def test_advantage_arithmetic_matches_the_reference_on_random_groups(hooks):
    assert hooks["advantage_mismatches"] == []


def test_positional_tables_and_packing_match_diffusers(hooks):
    """FluxPosEmbed / QwenEmbedRope (scale_rope) / WanRotaryPosEmbed (fp32 and bf16-cast buffers), FLUX latent packing + image ids and
    calculate_shift: the host tables the kernels read are bit-identical to what the real modules produce."""
    pos = hooks["positional"]
    assert all(pos["shift"])
    assert {k: v for k, v in pos.items() if k != "shift"} == {"flux_rope": True, "flux_pack": True, "qwen_rope": True, "wan_rope": True, "wan_rope_bf16": True}


def test_vae_host_side_against_the_real_autoencoder(hooks):
    """Config intake from a real AutoencoderKL.config, packing of its real state_dict, the 'pt' postprocess, and the post_quant_conv guard
    (diffusers' default AutoencoderKL has one)."""
    v = hooks["vae_host"]
    assert v["cfg"] == [4, [32, 64], 1, 8, 1.5305, 0.0609]
    assert v["n_packed"][0] == v["n_packed"][1]
    assert v["postprocess"] is True and v["post_quant_guard"] == "NotImplementedError"


def test_config_intake_and_packing_from_real_models(hooks):
    """`transformer.config` (FrozenDict) and `transformer.state_dict()` of real (tiny) diffusers models go through every engine's config
    intake and weight packer - the key names the packers read are the real ones."""
    it = hooks["intake"]
    assert it["sd3"] == [2, 2, 1, True]
    assert it["flux"] == [1, 1, 2, True, True]
    assert it["qwen"] == [1, 1, 2, True]
    assert it["wan"] == [1, 2, 320, [256, 64], 1]


def test_from_reference_adapter_reads_real_reference_objects(hooks):
    """The constructor INTEGRATION.md's glue uses: a real SD3Transformer2DModel and a real reference scheduler instance in, the engine config,
    every weight, the scheduler settings (incl. SDE-step list / seed / dynamics) and the decode callback out."""
    r = hooks["from_reference"]
    assert r["cfg"] == [2, 2] and r["n_keys"] is True
    assert r["sched"] == [0.6, "Dance-SDE", 7, 2, [1, 2, 5]]
    assert r["timesteps_equal"] and r["sde_equal"] and r["decode"] == 0.5


def test_randn_tensor_mirror(hooks):
    """Initial latents from per-prompt CPU generator lists (GRPOTrainer.evaluate) are the same numbers diffusers' randn_tensor draws."""
    assert hooks["randn_tensor"] == [True, True, True, True]


@needs_reference
def test_reference_side_glue_file(live):
    """integration/ff_b200_glue.py (subclass of the REAL SD3_5Adapter): rollout() re-packs the weights and syncs the seed, eval() / train()
    reach both schedulers."""
    g1, g2, g3, mro = live["glue"]
    assert g1 == ["rollout", 123, False, False, 1]
    assert g2 == ["eval", True, True] and g3 == ["train", False]
    assert mro[:2] == ["B200GlueSD3_5Adapter", "SD3_5Adapter"]


@needs_reference
def test_glue_engine_follows_weight_swapping_contexts(live):
    """The engine's packed copy follows use_ref_parameters / use_ema_parameters (nested too) and the optimizer in train mode: the no-grad
    KL-reference forward (grpo.py:282-292) and NFT's sampling_context forward (nft.py:360) see theta_ref / the EMA policy, not the weights
    of the last rollout.  The stand-in forward reports the mean of the packed proj_out.bias: policy 1.0, EMA 0.25, theta_ref -0.5."""
    g = live["glue_contexts"]
    assert g["stale_after_rollout"] is True
    c = g["ctx"]
    assert c["policy"] == 1.0 and c["ref"] == -0.5 and c["after_ref"] == 1.0
    assert c["ref_again_refreshes"] == 0                      # same context, nothing changed: no second re-pack
    assert c["ema"] == 0.25 and c["ema_then_ref"] == -0.5 and c["back_in_ema"] == 0.25 and c["after_ema"] == 1.0
    assert c["module_restored"] == 1.0
    assert c["train_mode_tracks_optimizer"] == 2.0


@needs_reference
def test_glue_handles_a_peft_wrapped_transformer(live):
    """finetune_type='lora' (examples/grpo/lora/sd3_5/default.yaml): post_init sees PEFT key names; the policy engine holds W + (alpha/r) B A,
    inside use_ref_parameters() (PEFT disable_adapter: no tensor changes) it holds the base W."""
    l = live["glue_contexts"]["lora"]
    assert any(k.endswith("to_q.base_layer.weight") for k in l["peft_keys"]) and any("lora_A.default" in k for k in l["peft_keys"])
    assert all(k.startswith("base_model.model.") for k in l["peft_keys"])
    assert l["post_init_plain_keys"] and l["plain_keys_only"]
    assert abs(l["policy_delta"] - 1.0) < 1e-6 and l["ref_delta"] == 0.0 and abs(l["after_delta"] - 1.0) < 1e-6


@needs_reference
def test_attention_backend_slot_routes_to_the_b200_function(live):
    """`install_attention_backend` + the reference's own `set_attention_backend` / `dispatch_attention_fn`: the registry slot holds our
    function with the registry's argument names; a FLUX forward through it (kernel replaced by an SDPA stand-in on this GPU-less box) is
    the default backend's output - layout (B,S,H,D), scale and call count (1 dual + 1 single block) are right; gradients come from the
    SDPA recomputation; unsupported arguments raise instead of being ignored; uninstall restores the slot."""
    h = live["diffusers_hooks"]
    assert h["cpu_call_raises"] is True and h["slot"] == [True, True, True]
    assert h["flux_calls"] == 2 and h["flux_shapes"][0] == [2, 17, 2, 64] and h["flux_max_diff"] <= 1e-5
    assert h["grad_max_diff"] <= 1e-5
    assert all(h["unsupported_arguments_raise"]) and h["uninstalled"] is True


@needs_reference
def test_sd3_attn_processor_is_a_drop_in_for_joint_attn_processor(live):
    """`B200JointAttnProcessor` installed through `set_attn_processor` on a real SD3Transformer2DModel: same call signature as
    JointAttnProcessor2_0, three attention calls (joint + attn2 in the dual block, joint in the context_pre_only block) over
    [image ; text] (16 + 7 tokens) and image-only (16) sequences, and the model output of the stock processor."""
    h = live["diffusers_hooks"]
    assert h["sd3_processors"] == ["B200JointAttnProcessor"] and h["sd3_signature"] is True
    assert h["sd3_calls"] == 3 and h["sd3_joint_len"] == [16, 23]
    assert h["sd3_max_diff"] <= 2e-3          # q / k / v pass through bf16 (the kernel's input type); a wrong token order would be O(1)


@needs_reference
def test_glue_recomputes_old_log_probs_through_the_reference_forward(live):
    """SURVEY 7.2 #1 option (b): the stored SDE transitions (both end points kept) are replayed teacher-forced through SD3_5Adapter.forward
    (the reference path, not the engine) and their log-probs replace the engine's; a log-prob whose start latent is not stored keeps the
    engine's value; the switch turns it off."""
    r = live["glue_contexts"]["recompute"]
    assert [(c["t"], c["t_next"]) for c in r["calls"]] == [(1000.0, 900.0), (900.0, 750.0)]
    assert r["calls"][0]["x_t"] == [0.0, 10.0] and r["calls"][0]["x_n"] == [1.0, 11.0] and r["calls"][1]["x_t"] == [1.0, 11.0]
    assert all(c["g"] == 4.5 and c["rk"] == ["log_prob"] and c["nl"] == 0.7 and c["pe"] == 2 for c in r["calls"])
    assert r["log_probs"] == [[100.0, 101.0, -1.0], [210.0, 211.0, -1.0]]
    assert r["disabled_keeps_engine_values"] == [True, [-1.0, -1.0, -1.0]]
