"""-m gpu parity at the geometries the benchmarks time (bench.py --config flux1 / qwen_image / wan21, tools/vae_bench.py): full width,
token counts and forward batch, random-init weights; only the depth is cut (2 blocks of each kind - every block launches the same shapes).

Truth: the pinned oracle on the engine's bf16-rounded weights and inputs in IEEE fp32 (tests.gpu_util.ieee_fp32: TF32 off for matmul
and cuDNN, SDPA replaced by a query-chunked fp32 attention, because torch's math backend would hold 40 GB of scores at Wan2.1's 20 280
tokens).  Yardstick: the same oracle under CUDA bf16 autocast.  Every forward case bounds, against the same statistic of the bf16
reference, both the global relative error and the worst per-token relative error - the global norm hardly moves when one 128-token tile
is wrong - and checks that the worst-token bound fails once the last (ragged) tile of the engine output carries an extra error of the
reference's own size there.  Each case records its numbers (parity_measured.jsonl, bench_geom_*.json); the B200 run the tolerances
come from is profiles/r03_parity_bench_geometry.jsonl."""
import dataclasses
import gc
import time

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from tests.gpu_util import chunked_sdpa, dump, err_report, ieee_fp32, record   # noqa: E402
from flow_factory_b200 import ops                                                # noqa: E402
from flow_factory_b200 import vae as V                                           # noqa: E402
from flow_factory_b200 import wan as W                                           # noqa: E402
from flow_factory_b200.flux import FluxRolloutEngine, model_scalar               # noqa: E402
from flow_factory_b200.qwen import QwenRolloutEngine                             # noqa: E402
from flow_factory_b200.scheduler import UniPCMultistepSDEScheduler               # noqa: E402
from oracle import flux_oracle as FO                                             # noqa: E402
from oracle import qwen_oracle as QO                                             # noqa: E402
from oracle import sd3_oracle as O                                               # noqa: E402
from oracle import vae_oracle as VO                                              # noqa: E402
from oracle import wan_oracle as WO                                              # noqa: E402

DEV = "cuda"
LOG2E = 1.4426950408889634
JSONL = "parity_measured.jsonl"
TILE = 128                                   # query / key tile of the attention kernels and row tile of the GEMMs


# ------------------------------------------------------------------------------------------------ metrics
def _rel(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-30))


def _token_err(got, truth):
    """[B, tokens, features] -> per-token relative error [B, tokens]."""
    return (got - truth).norm(dim=-1) / truth.norm(dim=-1).clamp_min(1e-30)


def _forward_report(tag, got, truth, ref, tail):
    """got / truth / ref fp32 [B, tokens, features], tokens in the order of the engine's sequence; `tail` = tokens in its last tile.
    The perturbed copy adds to each tail token, along the engine's own error there, an error as large as the bf16 reference's."""
    te, tr = _token_err(got, truth), _token_err(ref, truth)
    d = got[:, -tail:] - truth[:, -tail:]
    bad = got.clone()
    bad[:, -tail:] += d / d.norm(dim=-1, keepdim=True).clamp_min(1e-30) * (ref[:, -tail:] - truth[:, -tail:]).norm(dim=-1, keepdim=True)
    i = int(te.argmax())
    rep = dict(tag=tag, shape=list(got.shape), tail_tokens=tail, n_nan=int(torch.isnan(got).sum()),
               e_engine=_rel(got, truth), e_ref_bf16=_rel(ref, truth),
               worst_engine=float(te.max()), worst_ref=float(tr.max()), worst_engine_at=[i // te.shape[1], i % te.shape[1]],
               tail_engine=float(te[:, -tail:].max()), tail_ref=float(tr[:, -tail:].max()),
               e_perturbed=_rel(bad, truth), worst_perturbed=float(_token_err(bad, truth).max()))
    rep["ratio"] = rep["e_engine"] / rep["e_ref_bf16"]
    rep["worst_ratio"] = rep["worst_engine"] / rep["worst_ref"]
    rep["rows"] = err_report(got.reshape(-1, got.shape[-1]), truth.reshape(-1, truth.shape[-1]), tag)
    return rep


def _check_forward(rep, k_global, k_worst):
    """Engine within k x the bf16 reference's global and worst-token error (+ the 5e-4 floor of the existing forward tests), and the
    worst-token bound trips on the perturbed copy."""
    rep["bound_global"] = k_global * rep["e_ref_bf16"] + 5e-4
    rep["bound_worst"] = k_worst * rep["worst_ref"] + 5e-4
    _finish(rep)
    assert rep["n_nan"] == 0, rep
    assert rep["e_engine"] <= rep["bound_global"], rep
    assert rep["worst_engine"] <= rep["bound_worst"], rep
    assert rep["worst_perturbed"] > rep["bound_worst"], rep       # the metric sees a reference-sized error confined to the last tile


def _start():
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    return time.perf_counter()


def _finish(rep):
    torch.cuda.synchronize()
    rep["peak_torch_alloc_gb"] = torch.cuda.max_memory_allocated() / 2 ** 30
    rep["wall_s"] = time.perf_counter() - rep.pop("t0", time.perf_counter())
    dump(f"bench_geom_{rep['tag']}.json", rep)
    record(JSONL, {k: v for k, v in rep.items() if k != "rows"})


def _free(d):
    d.clear()
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _tail(n_joint):
    return n_joint % TILE or TILE


# ------------------------------------------------------------------------------------------------ FLUX.1-dev: B 2, 1024^2, 512 text tokens
FLUX_B, FLUX_LAT, FLUX_NT, FLUX_GS, FLUX_T = 2, 128, 512, 3.5, 612.0


@pytest.fixture(scope="class")
def flux():
    cfg = dataclasses.replace(FO.flux1_dev(), num_layers=2, num_single_layers=2)
    wb = {k: v.bfloat16() for k, v in FO.make_flux_weights(cfg, seed=0, device=DEV).items()}
    lat, pe, pooled, img_ids, _ = FO.make_flux_inputs(cfg, FLUX_B, FLUX_LAT, FLUX_LAT, FLUX_NT, seed=1)
    eng = FluxRolloutEngine(cfg, wb)
    plan = eng.plan(FLUX_B, FLUX_LAT // 2, FLUX_LAT // 2, FLUX_NT)
    pe, pooled = pe.bfloat16().to(DEV), pooled.bfloat16().to(DEV)
    eng.set_prompts(plan, pe, pooled, FLUX_GS)
    d = dict(cfg=cfg, wb=wb, lat=lat.half().to(DEV), pe=pe, pooled=pooled, img_ids=img_ids, eng=eng, plan=plan)
    yield d
    _free(d)


class TestFlux:
    def test_forward_vs_oracle(self, flux):
        t0 = _start()
        cfg, wb, lat, pe, pooled, img_ids = (flux[k] for k in ("cfg", "wb", "lat", "pe", "pooled", "img_ids"))
        got = flux["eng"].transformer_forward(flux["plan"], lat, FLUX_T).float()
        B, txt_ids = FLUX_B, torch.zeros(FLUX_NT, 3)
        t_eff = torch.full((B,), model_scalar(FLUX_T / 1000) / 1000, device=DEV)       # the scalars the engine's bf16 semantics see
        g_eff = torch.full((B,), model_scalar(FLUX_GS, torch.float16) / 1000, device=DEV)
        wt = {k: v.float() for k, v in wb.items()}
        with ieee_fp32():
            truth = FO.flux_forward(wt, cfg, lat.float(), pe.float(), pooled.float(), t_eff, img_ids, txt_ids, guidance=g_eff)
        del wt
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            ref = FO.flux_forward(wb, cfg, lat.bfloat16(), pe, pooled, torch.full((B,), FLUX_T / 1000, device=DEV), img_ids.bfloat16(),
                                  txt_ids.bfloat16(), guidance=torch.full((B,), FLUX_GS, device=DEV).half()).float()
        rep = _forward_report("flux_fwd_1024_b2", got, truth, ref, _tail(FLUX_NT + got.shape[1]))
        rep.update(t0=t0, workspace_gb=flux["plan"].workspace_bytes / 2 ** 30)
        _check_forward(rep, k_global=1.3, k_worst=1.3)      # measured on B200: 1.002 x (global), 1.003 x (worst token) the bf16 reference

    def test_step_and_rollout(self, flux):
        """FluxRolloutEngine.step on explicit noise vs O.sde_step on the engine's own noise prediction (the log-prob mean runs over
        4096 x 64 = 262 144 elements per sample); a 2-step rollout with and without the CUDA graph, bit for bit."""
        t0 = _start()
        eng, plan, lat = flux["eng"], flux["plan"], flux["lat"]
        T, i, nl = 28, 3, 0.7
        ts, sig, coefs = eng.make_coefs(plan, T, nl, [i])
        g = torch.Generator(device=DEV).manual_seed(5)
        noise = torch.randn(lat.shape, generator=g, device=DEV)
        out = eng.step(plan, lat, coefs[i], noise=noise)
        v = eng.transformer_forward(plan, lat, float(ts[i]))
        o = O.sde_step(out["noise_pred"], lat, float(sig[i]), float(sig[i + 1]), nl, float(sig[1]), "Flow-SDE", noise=noise,
                       compute_log_prob=True)
        rep = dict(tag="flux_step_1024_b2", t0=t0,
                   noise_pred_equals_forward=bool(torch.equal(out["noise_pred"], v)),
                   mean_max_abs=float((out["next_latents_mean"] - o["next_latents_mean"]).abs().max()),
                   next_latents_mismatches=int((out["next_latents"].float() != o["next_latents"]).sum()),
                   log_prob=out["log_prob"].tolist(), log_prob_oracle=o["log_prob"].tolist(),
                   log_prob_rel=float(((out["log_prob"] - o["log_prob"]).abs() / o["log_prob"].abs().clamp_min(1e-6)).max()),
                   overflow=int(out["overflow"]))
        _, _, c2 = eng.make_coefs(plan, 2, nl, [0], store_slots=[1, 2], logp_slots=[0, -1])
        noises = torch.randn((2, *lat.shape), generator=g, device=DEV)
        runs = {}
        for graph in (False, True):
            r = eng.rollout(plan, lat, c2, n_latent_slots=3, store_initial_slot=0, n_logp_slots=1, noise=noises, use_graph=graph)
            torch.cuda.synchronize()
            runs[graph] = r
        rep["rollout_graph_equals_eager"] = all(torch.equal(runs[False][k], runs[True][k]) for k in ("all_latents", "log_probs", "final_latents"))
        rep["rollout_log_probs"] = runs[True]["log_probs"].flatten().tolist()
        _finish(rep)
        assert rep["overflow"] == 0 and int(runs[True]["overflow"]) == 0, rep
        assert rep["noise_pred_equals_forward"], rep
        torch.testing.assert_close(out["next_latents_mean"], o["next_latents_mean"], rtol=1e-6, atol=1e-6)
        assert rep["next_latents_mismatches"] == 0, rep           # measured on B200: 0 of 2 x 262 144
        assert rep["log_prob_rel"] <= 1e-5, rep                   # measured on B200: 0 (same reduction order)
        assert rep["rollout_graph_equals_eager"], rep


# ------------------------------------------------------------------------------------------------ Qwen-Image: 1024^2, 256 text tokens, true CFG 4.0
QWEN_H2, QWEN_NT, QWEN_GS, QWEN_T = 64, 256, 4.0, 612.0


@pytest.fixture(scope="class")
def qwen():
    cfg = dataclasses.replace(QO.qwen_image_20b(), num_layers=2)
    wb = {k: v.bfloat16().to(DEV) for k, v in QO.make_qwen_weights(cfg, seed=0).items()}
    lat, pe = QO.make_qwen_inputs(cfg, 1, QWEN_H2, QWEN_H2, QWEN_NT, seed=1)
    _, npe = QO.make_qwen_inputs(cfg, 1, QWEN_H2, QWEN_H2, QWEN_NT, seed=7)
    eng = QwenRolloutEngine(cfg, wb)
    plan = eng.plan(1, QWEN_H2, QWEN_H2, QWEN_NT, cfg=True)
    d = dict(cfg=cfg, wb=wb, lat=lat.half().to(DEV), pe=pe.bfloat16().to(DEV), npe=npe.bfloat16().to(DEV), eng=eng, plan=plan)
    yield d
    _free(d)


class TestQwen:
    @pytest.mark.parametrize("pos_len,k_global,k_worst", [
        (QWEN_NT, 1.33, 1.31),          # measured on B200: 1.024 x (global), 1.012 x (worst token) the bf16 reference
        (77, 1.33, 1.28),               # measured on B200: 1.024 x, 0.992 x
    ])
    def test_true_cfg_forward_vs_oracle(self, qwen, pos_len, k_global, k_worst):
        """Forward batch 2 = [negative ; positive]; pos_len < 256: the positive prompt right-padded, its padded keys masked."""
        t0 = _start()
        cfg, wb, lat, pe, npe, eng, plan = (qwen[k] for k in ("cfg", "wb", "lat", "pe", "npe", "eng", "plan"))
        eng.set_prompts(plan, pe, npe, QWEN_GS, prompt_lengths=[pos_len])
        got = eng.transformer_forward(plan, lat, QWEN_T).float()
        mask = None if pos_len == QWEN_NT else (torch.arange(QWEN_NT) < pos_len).float()[None].to(DEV)
        shape = (1, QWEN_H2, QWEN_H2)
        wt = {k: v.float() for k, v in wb.items()}
        te = torch.full((1,), eng.t_model(QWEN_T), device=DEV)
        with ieee_fp32():
            tp = QO.qwen_forward(wt, cfg, lat.float(), pe.float(), te, shape, encoder_hidden_states_mask=mask)
            tn = QO.qwen_forward(wt, cfg, lat.float(), npe.float(), te, shape)
            truth = QO.true_cfg_combine(tp, tn, QWEN_GS)
        del wt, tp, tn
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            tr = torch.full((1,), QWEN_T / 1000, device=DEV)
            rp = QO.qwen_forward(wb, cfg, lat.bfloat16(), pe, tr, shape, encoder_hidden_states_mask=mask)
            rn = QO.qwen_forward(wb, cfg, lat.bfloat16(), npe, tr, shape)
            ref = QO.true_cfg_combine(rp.bfloat16(), rn, QWEN_GS).float()
        rep = _forward_report(f"qwen_cfg_fwd_1024_pos{pos_len}", got, truth, ref, _tail(QWEN_NT + got.shape[1]))
        rep.update(t0=t0, workspace_gb=plan.workspace_bytes / 2 ** 30)
        _check_forward(rep, k_global, k_worst)


# ------------------------------------------------------------------------------------------------ Wan2.1-T2V-1.3B: 480x832, 49 frames, 512 text tokens, CFG 5.0
WAN_F, WAN_H, WAN_W, WAN_NT, WAN_GS, WAN_T = 13, 60, 104, 512, 5.0, 875.0      # latent 13 x 60 x 104 -> 20 280 tokens


def _wan_tokens(x):
    """[B, C, F, H, W] -> [B, F (H/2) (W/2), 4C]: the engine's token order (f, h', w')."""
    B, Cc, Fr, H, Wd = x.shape
    return x.float().reshape(B, Cc, Fr, H // 2, 2, Wd // 2, 2).permute(0, 2, 3, 5, 1, 4, 6).reshape(B, Fr * (H // 2) * (Wd // 2), Cc * 4)


@pytest.fixture(scope="class")
def wan():
    ocfg = dataclasses.replace(WO.wan21_t2v_1_3b(), num_layers=2)
    cfg = W.WanEngineConfig(num_layers=2, num_attention_heads=ocfg.num_attention_heads, text_dim=ocfg.text_dim, ffn_dim=ocfg.ffn_dim,
                            rope_max_seq_len=ocfg.rope_max_seq_len)
    w = {k: v.bfloat16().float() for k, v in WO.make_wan_weights(ocfg, seed=3).items()}
    lat, pe = WO.make_wan_inputs(ocfg, 1, WAN_F, WAN_H, WAN_W, WAN_NT, seed=4)
    neg = torch.randn(pe.shape, generator=torch.Generator().manual_seed(5))
    eng = W.WanRolloutEngine(cfg, w, device=DEV)
    plan = eng.plan(1, WAN_F, WAN_H, WAN_W, WAN_NT, cfg=True)
    pe, neg = pe.bfloat16().to(DEV), neg.bfloat16().to(DEV)
    eng.set_prompts(plan, pe, neg)
    d = dict(ocfg=ocfg, w=w, lat=lat.half().to(DEV), pe=pe, neg=neg, eng=eng, plan=plan)
    yield d
    _free(d)


class TestWan:
    def test_cfg_forward_vs_oracle(self, wan):
        t0 = _start()
        ocfg, lat, pe, neg, eng, plan = (wan[k] for k in ("ocfg", "lat", "pe", "neg", "eng", "plan"))
        got = eng.transformer_forward(plan, lat, WAN_T, guidance_scale=WAN_GS)
        tt = torch.full((1,), WAN_T, device=DEV)
        wt = {k: v.to(DEV) for k, v in wan["w"].items()}
        with ieee_fp32():
            tc = WO.wan_forward(wt, ocfg, lat.float(), tt, pe.float())
            tu = WO.wan_forward(wt, ocfg, lat.float(), tt, neg.float())
            truth = tu + WAN_GS * (tc - tu)
        wb = {k: v.bfloat16() for k, v in wt.items()}
        del wt, tc, tu
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            rc = WO.wan_forward(wb, ocfg, lat.bfloat16(), tt, pe)
            ru = WO.wan_forward(wb, ocfg, lat.bfloat16(), tt, neg)
            ref = ru + WAN_GS * (rc - ru)                                              # bf16 tensor ops (wan2_t2v.py:526)
        n_tok = WAN_F * (WAN_H // 2) * (WAN_W // 2)
        rep = _forward_report("wan_cfg_fwd_480p_49f", _wan_tokens(got), _wan_tokens(truth), _wan_tokens(ref), _tail(n_tok))
        rep.update(t0=t0, workspace_gb=plan.workspace_bytes / 2 ** 30)
        _check_forward(rep, k_global=1.29, k_worst=1.28)    # measured on B200: 0.998 x (global), 0.988 x (worst token) the bf16 reference

    def test_step_and_rollout(self, wan):
        """WanRolloutEngine.step on explicit noise vs O.sde_step on the engine's own CFG noise prediction (log-prob mean over
        16 x 13 x 60 x 104 = 1.3 M elements); a 2-step rollout with and without the CUDA graph, bit for bit."""
        t0 = _start()
        lat, eng, plan = wan["lat"], wan["eng"], wan["plan"]
        sch = UniPCMultistepSDEScheduler(noise_level=0.7, flow_shift=3.0, num_sde_steps=1, seed=1)
        ts = sch.set_timesteps(40)
        i, nl = 2, 0.7
        c = sch.step_coef(ts[i], ts[i + 1], nl, compute_log_prob=True, t_model=float(ts[i]))
        g = torch.Generator(device=DEV).manual_seed(6)
        noise = torch.randn(lat.shape, generator=g, device=DEV)
        out = eng.step(plan, lat, c, WAN_GS, noise=noise)
        v = eng.transformer_forward(plan, lat, float(ts[i]), guidance_scale=WAN_GS)
        o = O.sde_step(out["noise_pred"], lat, c.sigma, c.sigma_prev, nl, float(sch.sigmas[1]), "Flow-SDE", noise=noise, compute_log_prob=True)
        rep = dict(tag="wan_step_480p_49f", t0=t0,
                   noise_pred_equals_forward=bool(torch.equal(out["noise_pred"], v)),
                   mean_max_abs=float((out["next_latents_mean"] - o["next_latents_mean"]).abs().max()),
                   next_latents_mismatches=int((out["next_latents"].float() != o["next_latents"]).sum()),
                   log_prob=out["log_prob"].tolist(), log_prob_oracle=o["log_prob"].tolist(),
                   log_prob_rel=float(((out["log_prob"] - o["log_prob"]).abs() / o["log_prob"].abs().clamp_min(1e-6)).max()),
                   overflow=int(out["overflow"]))
        s2 = UniPCMultistepSDEScheduler(noise_level=0.7, flow_shift=3.0, seed=1)
        t2 = s2.set_timesteps(2)
        c2 = [s2.step_coef(t2[0], t2[1], nl, compute_log_prob=True, t_model=float(t2[0]), store_slot=1, logp_slot=0),
              s2.step_coef(t2[1], torch.tensor(0), 0.0, compute_log_prob=False, t_model=float(t2[1]), store_slot=2, logp_slot=-1)]
        noises = torch.randn((2, *lat.shape), generator=g, device=DEV)
        runs = {}
        for graph in (False, True):
            r = eng.rollout(plan, lat, c2, WAN_GS, n_latent_slots=3, store_initial_slot=0, n_logp_slots=1, noise=noises, use_graph=graph)
            torch.cuda.synchronize()
            runs[graph] = r
        rep["rollout_graph_equals_eager"] = all(torch.equal(runs[False][k], runs[True][k]) for k in ("all_latents", "log_probs", "final_latents"))
        rep["rollout_log_probs"] = runs[True]["log_probs"].flatten().tolist()
        _finish(rep)
        assert rep["overflow"] == 0 and int(runs[True]["overflow"]) == 0, rep
        assert rep["noise_pred_equals_forward"], rep
        torch.testing.assert_close(out["next_latents_mean"], o["next_latents_mean"], rtol=1e-6, atol=1e-6)
        assert rep["next_latents_mismatches"] == 0, rep           # measured on B200: 0 of 1 297 920
        assert rep["log_prob_rel"] <= 1e-5, rep                   # measured on B200: 0
        assert rep["rollout_graph_equals_eager"], rep


# ------------------------------------------------------------------------------------------------ SD3.5 VAE decode: 1024^2, batch 8
VAE_B, VAE_LAT = 8, 128


def _vae_tokens(img):
    """[B, 3, 8h, 8w] -> [B, h w, 192]: one token per latent position (its 8 x 8 pixel patch), row-major like the mid-block attention."""
    B, Cc, H, Wd = img.shape
    return img.float().reshape(B, Cc, H // 8, 8, Wd // 8, 8).permute(0, 2, 4, 1, 3, 5).reshape(B, (H // 8) * (Wd // 8), Cc * 64)


def test_vae_decode_1024_b8_vs_oracle():
    """The full SD3.5 decoder at 1024^2, batch 8: 16 384-token mid-block attention (the row softmax at its maximum n), GroupNorm over
    1 M-pixel planes, activations of 4 GB (8 x 1024^2 x 256 bf16 after the last upsample).  Oracle one image at a time."""
    t0 = _start()
    ocfg = VO.sd35_vae()
    w32 = {k: v.bfloat16().float() for k, v in VO.make_vae_decoder_weights(ocfg, seed=11).items()}
    cfg = V.VaeDecoderConfig(ocfg.latent_channels, ocfg.out_channels, tuple(ocfg.block_out_channels), ocfg.layers_per_block,
                             ocfg.norm_num_groups, ocfg.scaling_factor, ocfg.shift_factor)
    lat = torch.randn(VAE_B, 16, VAE_LAT, VAE_LAT, generator=torch.Generator().manual_seed(12)).half().to(DEV)
    dec = V.B200VaeDecoder(cfg, w32, VAE_LAT, VAE_LAT, batch=VAE_B, device=DEV)
    img = dec.decode(lat).float()
    ws = dec.workspace_bytes()
    dec.close()
    del dec
    wd = {k: v.to(DEV) for k, v in w32.items()}
    wb = {k: v.bfloat16() for k, v in wd.items()}
    truth, ref = torch.empty_like(img), torch.empty_like(img)
    for b in range(VAE_B):
        with ieee_fp32():
            truth[b] = VO.vae_decode(wd, ocfg, lat[b:b + 1].float())[0]
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            ref[b] = VO.vae_decode(wb, ocfg, lat[b:b + 1].bfloat16())[0].float()
    rep = _forward_report("vae_decode_1024_b8", _vae_tokens(img), _vae_tokens(truth), _vae_tokens(ref), _tail(VAE_LAT * VAE_LAT))
    rep.update(t0=t0, workspace_gb=ws / 2 ** 30)
    _check_forward(rep, k_global=1.13, k_worst=1.15)        # measured on B200: 0.871 x (global), 0.89 - 0.93 x (worst token, two runs)


# ------------------------------------------------------------------------------------------------ op level, at the same shapes
def _op_check(tag, got, ref, tol):
    """max |got - ref| <= tol * max(1, max |ref|) - the convention of test_gpu_attention.py / test_gpu_gemm.py."""
    rep = err_report(got.reshape(-1, got.shape[-1]), ref.reshape(-1, ref.shape[-1]), tag)
    rep["rel_fro"] = _rel(got, ref)
    rep["max_abs_over_scale"] = rep["max_abs"] / max(1.0, rep["ref_absmax"])
    dump(f"bench_geom_op_{tag}.json", rep)
    record(JSONL, dict(tag=tag, max_abs_over_scale=rep["max_abs_over_scale"], rel_fro=rep["rel_fro"],
                       peak_torch_alloc_gb=torch.cuda.max_memory_allocated() / 2 ** 30))
    assert rep["n_nan"] == 0 and rep["max_abs_over_scale"] <= tol, rep


def _sdpa_ref(q, k, v, H, d, scale=None):
    B, S = q.shape[:2]
    sp = lambda t: t.float().reshape(B, t.shape[1], H, d).transpose(1, 2)
    with ieee_fp32():
        return chunked_sdpa(sp(q), sp(k), sp(v), scale=scale).transpose(1, 2).reshape(B, S, H * d)


# FLUX joint 4096 + 512 tokens ; Wan self-attention 13 x 30 x 52 tokens.  Last element: the tolerance of test_op_attention_d128_dense
# and then of test_op_attention_d128_prescaled, 1.3 x the max |err| / max(1, max |ref|) measured on B200 (9.1e-4, 3.3e-4 ; 8.2e-4, 2.7e-4)
ATTN_GEOMS = [(2, 4608, 24, 1.15e-3, 1.05e-3), (2, 20280, 12, 4.3e-4, 3.4e-4)]


@pytest.mark.parametrize("B,S,H,tol,_", ATTN_GEOMS)
def test_op_attention_d128_dense(B, S, H, tol, _):
    g = torch.Generator(device=DEV).manual_seed(S + H)
    qkv = torch.randn(B, S, 3 * 128 * H, generator=g, device=DEV).bfloat16()
    out = ops.attention(qkv, H, head_dim=128)
    q, k, v = qkv.split(128 * H, dim=-1)
    _op_check(f"attn128_dense_{B}_{S}_{H}", out.float(), _sdpa_ref(q, k, v, H, 128), tol)


@pytest.mark.parametrize("B,S,H,_,tol", ATTN_GEOMS)
def test_op_attention_d128_prescaled(B, S, H, _, tol):
    """The engines' layout: keys carry softmax_scale * log2(e) (one bf16 rounding); reference = fp32 softmax in base 2."""
    g = torch.Generator(device=DEV).manual_seed(7 * S + H)
    q, k, v = (torch.randn(B, S, 128 * H, generator=g, device=DEV) for _ in range(3))
    kp = (k * (128 ** -0.5 * LOG2E)).bfloat16()
    qkv = torch.cat([q.bfloat16(), kp, v.bfloat16()], dim=-1).contiguous()
    out = ops.attention(qkv, H, head_dim=128, k_prescaled=True)
    _op_check(f"attn128_prescaled_{B}_{S}_{H}", out.float(), _sdpa_ref(q.bfloat16(), kp, v.bfloat16(), H, 128, scale=1.0 / LOG2E), tol)


def test_op_attention_d128_into_single_block_row():
    """FLUX single block: the attention output is the first 3072 columns of the 15 360-wide [attn | mlp] row (pre-scaled keys)."""
    B, S, H, row = 2, 4608, 24, 15360
    g = torch.Generator(device=DEV).manual_seed(17)
    q, k, v = (torch.randn(B, S, 128 * H, generator=g, device=DEV) for _ in range(3))
    kp = (k * (128 ** -0.5 * LOG2E)).bfloat16()
    qkv = torch.cat([q.bfloat16(), kp, v.bfloat16()], dim=-1).contiguous()
    wide = torch.full((B, S, row), 7.0, device=DEV, dtype=torch.bfloat16)
    ops.attention(qkv, H, wide, head_dim=128, out_row_stride=row, k_prescaled=True)
    assert bool((wide[..., 128 * H:] == 7.0).all())                                   # the mlp columns untouched
    _op_check("attn128_row15360_2_4608_24", wide[..., :128 * H].float(), _sdpa_ref(q.bfloat16(), kp, v.bfloat16(), H, 128, scale=1.0 / LOG2E),
              9.2e-4)                                                               # measured on B200: 7.1e-4


def test_op_attention_cross_wan():
    B, Sq, Skv, H = 2, 20280, 512, 12
    D = 128 * H
    g = torch.Generator(device=DEV).manual_seed(Sq + Skv)
    q = torch.randn(B, Sq, D, generator=g, device=DEV).bfloat16()
    kv = torch.randn(B, Skv, 2 * D, generator=g, device=DEV).bfloat16()
    out = W.attention_cross(q, kv, H)
    _op_check("attn_cross_2_20280_512_12", out.float(), _sdpa_ref(q, kv[..., :D], kv[..., D:], H, 128), 4.8e-3)   # measured on B200: 3.7e-3


def test_op_ln_modulate_d3072_full_rows():
    """LayerNorm-modulate at D = 3072 (the kernel's LN_MAXC limit) over FLUX's 2 x 4096 image rows."""
    g = torch.Generator(device=DEV).manual_seed(3)
    B, R, D = 2, 4096, 3072
    x = (2 * torch.randn(B, R, D, device=DEV, generator=g) + 0.3).bfloat16()
    mod = (0.2 * torch.randn(B, 2 * D, device=DEV, generator=g)).bfloat16()
    out = torch.empty_like(x)
    ops.ln_modulate(x, mod[:, :D], mod[:, D:], out, mod_batch_stride=2 * D)
    y = F.layer_norm(x.float(), (D,), None, None, 1e-6)
    ref = y * (1 + mod[:, D:].float())[:, None].bfloat16().float() + mod[:, :D].float()[:, None]
    _op_check("ln_modulate_2_4096_3072", out.float(), ref, 2.7e-3)          # measured on B200: 2.1e-3


def test_op_wan_rms_rope_and_layer_norm_d1536():
    g = torch.Generator(device=DEV).manual_seed(1536)
    B, D = 2, 1536
    S = WAN_F * (WAN_H // 2) * (WAN_W // 2)
    cos, sin = (t.to(DEV) for t in W.wan_rope_tables(W.WanEngineConfig(), WAN_F, WAN_H // 2, WAN_W // 2))
    qkv = torch.randn(B, S, 3 * D, generator=g, device=DEV).bfloat16()
    w = (1 + 0.1 * torch.randn(D, generator=g, device=DEV)).bfloat16()
    x = qkv.clone()
    W.rms_rope_(x, D, w, 1e-6, cos, sin, col=D)                                     # the k block of the fused q|k|v row
    assert torch.equal(x[..., :D], qkv[..., :D]) and torch.equal(x[..., 2 * D:], qkv[..., 2 * D:])
    ref = F.rms_norm(qkv[..., D:2 * D].float(), (D,), w.float(), 1e-6).bfloat16()
    rh = ref.reshape(B, S, D // 128, 128)
    c, s_ = cos.bfloat16()[None, :, None, 0::2], sin.bfloat16()[None, :, None, 1::2]
    o = torch.empty_like(rh)
    o[..., 0::2] = rh[..., 0::2] * c - rh[..., 1::2] * s_                            # bf16 tensor arithmetic, as the reference
    o[..., 1::2] = rh[..., 0::2] * s_ + rh[..., 1::2] * c
    _op_check("wan_rms_rope_2_20280_1536", x[..., D:2 * D].float(), o.reshape(B, S, D).float(), 6.6e-3)   # measured on B200: 5.1e-3
    h = (torch.randn(B, S, D, generator=g, device=DEV) * 2 + 0.3).bfloat16()
    scale, shift = torch.randn(B, D, generator=g, device=DEV) * 0.2, torch.randn(B, D, generator=g, device=DEV) * 0.2
    ln = F.layer_norm(h.float(), (D,), None, None, 1e-6)
    _op_check("wan_layer_norm_mod_2_20280_1536", W.layer_norm(h, 1e-6, scale=scale, shift=shift).float(),
              ln * (1 + scale[:, None]) + shift[:, None], 2.6e-3)                  # measured on B200: 2.0e-3
    wt, bs = (1 + 0.1 * torch.randn(D, generator=g, device=DEV)).bfloat16(), (0.1 * torch.randn(D, generator=g, device=DEV)).bfloat16()
    _op_check("wan_layer_norm_affine_2_20280_1536", W.layer_norm(h, 1e-6, weight=wt, bias=bs).float(), ln * wt.float() + bs.float(),
              2.8e-3)                                                               # measured on B200: 2.2e-3


# (tag, M, N, K, epilogue, tol): the GEMMs whose shapes only these geometries launch, derived from the model dimensions.  tol: 1.3 x the
# max |err| / max(1, max |ref|) measured on B200 (3.99e-3, 4.33e-3, 4.51e-3, 2.78e-3, 2.96e-3, 5.40e-3, 2.80e-3) - one bf16 rounding of
# the output plus, for the gelu / gate epilogues, the reference's own rounding of A W^T + b to bf16 before the epilogue
GEMMS = [
    ("flux_ff1_gelu", 2 * 4096, 12288, 3072, ops.EPI_BIAS_GELU, 5.1e-3),          # dual-block ff.net.0 on 2 x 4096 image rows
    ("flux_ff2_gate", 2 * 4096, 3072, 12288, ops.EPI_GATE_RESIDUAL, 5.6e-3),     # dual-block ff.net.2, K = 4 D
    ("flux_single_out_gate", 2 * 4608, 3072, 15360, ops.EPI_GATE_RESIDUAL, 5.8e-3),   # single-block proj_out over [attn | mlp], K = 5 D
    ("flux_context_embedder", 2 * 512, 3072, 4096, ops.EPI_BIAS, 3.6e-3),
    ("qwen_txt_in", 2 * 256, 3072, 3584, ops.EPI_BIAS, 3.8e-3),                  # K = joint_dim 3584, both CFG halves
    ("wan_ffn1_gelu", 2 * 20280, 8960, 1536, ops.EPI_BIAS_GELU, 7.0e-3),         # N = 8960, ragged last row tile (40 560 = 316 x 128 + 112)
    ("wan_ffn2", 2 * 20280, 1536, 8960, ops.EPI_BIAS, 3.6e-3),
]


@pytest.mark.parametrize("tag,M,N,K,epi,tol", GEMMS, ids=[gm[0] for gm in GEMMS])
def test_op_linear_bench_shapes(tag, M, N, K, epi, tol):
    g = torch.Generator(device=DEV).manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g, device=DEV).bfloat16()
    Wt = (torch.randn(N, K, generator=g, device=DEV) / K ** 0.5).bfloat16()
    b = (torch.randn(N, generator=g, device=DEV) * 0.1).bfloat16()
    with ieee_fp32():
        y = F.linear(A.float(), Wt.float(), b.float())
    if epi == ops.EPI_GATE_RESIDUAL:                                  # h += gate[b] * (A W^T + b), B = 2 halves of the rows
        B = 2
        gate = torch.randn(B, 3 * N, generator=g, device=DEV).bfloat16()
        out = torch.randn(M, N, generator=g, device=DEV).bfloat16()
        ref = (out.float().reshape(B, M // B, N) + gate[:, None, N:2 * N].float() * y.bfloat16().float().reshape(B, M // B, N)).reshape(M, N)
        ops.linear(A, Wt, b, out, num_batch=B, rows_per_batch=M // B, a_batch_stride=(M // B) * K, out_batch_stride=(M // B) * N,
                   epi=epi, gate=gate[:, N:], gate_batch_stride=3 * N)
    else:
        out = torch.full((M, N), float("nan"), device=DEV, dtype=torch.bfloat16)
        ops.linear(A, Wt, b, out, epi=epi)
        ref = F.gelu(y.bfloat16().float(), approximate="tanh") if epi == ops.EPI_BIAS_GELU else y
    _op_check(f"gemm_{tag}_{M}_{N}_{K}", out.float(), ref, tol)


def test_op_linear_qkv_rope_flux_single_block():
    """Single-block fused q|k|v + RMSNorm + RoPE over the joint 512 + 4096 rows, B = 2, K = N / 3 = 3072."""
    B, nt, ni, H, K = 2, 512, 4096, 24, 3072
    S, D = nt + ni, 128 * H
    g = torch.Generator(device=DEV).manual_seed(21)
    x = torch.randn(B, S, K, generator=g, device=DEV).bfloat16()
    Wt = (torch.randn(3 * D, K, generator=g, device=DEV) / K ** 0.5).bfloat16()
    b = (0.1 * torch.randn(3 * D, generator=g, device=DEV)).bfloat16()
    nq, nk = ((1 + 0.1 * torch.randn(128, generator=g, device=DEV)).bfloat16() for _ in range(2))
    ids = torch.cat([torch.zeros(nt, 3), FO.latent_image_ids(128, 128)])
    cos, sin = (t.to(DEV).contiguous() for t in FO.rope_tables(ids, (16, 56, 56)))
    out = torch.empty(B, S, 3 * D, device=DEV, dtype=torch.bfloat16)
    ops.linear_qkv_rope(x, Wt, b, out, nq, nk, cos, sin, num_batch=B, rows_per_batch=S, out_batch_stride=S * 3 * D)
    with ieee_fp32():
        y = F.linear(x.float(), Wt.float(), b.float()).bfloat16()
    q, k, v = y.split(D, dim=-1)
    parts = [FO.apply_rope(F.rms_norm(t.unflatten(-1, (H, 128)).float(), (128,), w.float(), 1e-6).bfloat16(), cos, sin).flatten(-2)
             for t, w in ((q, nq), (k, nk))]
    _op_check("qkv_rope_2_4608_24", out.float(), torch.cat(parts + [v], dim=-1).float(), 6.6e-3)   # measured on B200: 5.1e-3


@pytest.mark.parametrize("B,cin,cout,residual,tol", [
    (8, 256, 128, False, 6.3e-3),       # measured on B200: 4.9e-3 (one bf16 ulp at |ref| = 6.4)
    (1, 128, 128, True, 5.0e-3),        # measured on B200: 3.9e-3
])
def test_op_conv3x3_decoder_1024(B, cin, cout, residual, tol):
    """The last decoder level at 1024^2: 256 -> 128 (batch 8: a 4 GB input) and 128 -> 128 with the residual add."""
    Hh = Wd = 1024
    g = torch.Generator(device=DEV).manual_seed(B * cin + cout)
    x = torch.randn(B, Hh, Wd, cin, generator=g, device=DEV).bfloat16()
    w = (torch.randn(cout, cin, 3, 3, generator=g, device=DEV) / (3 * cin ** 0.5)).bfloat16()
    b = (torch.randn(cout, generator=g, device=DEV) * 0.1).bfloat16()
    res = torch.randn(B, Hh, Wd, cout, generator=g, device=DEV).bfloat16() if residual else None
    out = V.conv2d_nhwc(x, w, b, res)
    ref = torch.empty(B, Hh, Wd, cout, device=DEV)
    with ieee_fp32():
        for i in range(B):
            ref[i] = F.conv2d(x[i:i + 1].permute(0, 3, 1, 2).float(), w.float(), b.float(), padding=1).permute(0, 2, 3, 1)[0]
    ref = ref.bfloat16().float() + (res.float() if residual else 0)
    del x
    _op_check(f"conv3x3_{B}_1024_{cin}_{cout}_{int(residual)}", out.float(), ref, tol)


@pytest.mark.parametrize("C,offset,silu,tol", [
    (128, 0.5, True, 3.0e-3),           # measured on B200: 2.35e-3
    (256, 0.5, False, 3.0e-3),          # measured on B200: 2.34e-3
    (128, 64.0, True, 2.8e-3),          # measured on B200: 2.18e-3 - no loss to cancellation
])
def test_op_group_norm_decoder_1024(C, offset, silu, tol):
    """GroupNorm (32 groups) over a 1 M-pixel plane.  offset 64: every group's mean is ~64 x its standard deviation, which guards the
    E[x^2] - mean^2 variance of the stats kernel (csrc/vae_elementwise.cu) against cancellation."""
    B, P, groups = 2, 1024 * 1024, 32
    g = torch.Generator(device=DEV).manual_seed(C + int(offset))
    x = (torch.randn(B, P, C, generator=g, device=DEV) + offset).bfloat16()
    gamma = (1 + 0.1 * torch.randn(C, generator=g, device=DEV)).bfloat16()
    beta = (0.1 * torch.randn(C, generator=g, device=DEV)).bfloat16()
    out = V.group_norm_nhwc(x, gamma, beta, groups, 1e-6, silu)
    with ieee_fp32():
        ref = F.group_norm(x.float().permute(0, 2, 1), groups, gamma.float(), beta.float(), 1e-6).permute(0, 2, 1)
    ref = F.silu(ref) if silu else ref
    _op_check(f"group_norm_{B}_{P}_{C}_off{offset:g}", out.float(), ref, tol)
