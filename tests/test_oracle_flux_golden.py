"""The FLUX.1 oracle (oracle/flux_oracle.py, SURVEY 8f row 2) pinned against fixtures minted from the REAL reference
(tests/golden/make_golden.py: vendored diffusers FluxTransformer2DModel + Flow-Factory scheduler, CPU)."""
import os
import torch, pytest
from oracle import flux_oracle as FO
from oracle import sd3_oracle as O


def _load(golden_dir):
    return torch.load(os.path.join(golden_dir, "flux_tiny.pt"), weights_only=False)


@pytest.mark.parametrize("name", ["tiny", "tiny3"])
def test_flux_forward_fp32_and_autocast(golden_dir, name):
    g = _load(golden_dir)[name]
    cfg = FO.tiny_flux_config() if name == "tiny" else FO.tiny_flux_config(num_layers=2, num_single_layers=1, heads=3, joint_dim=96, pooled_dim=48)
    w = FO.make_flux_weights(cfg, seed=g["seed"])
    assert sorted(w.keys()) == g["keys"]            # key parity with FluxTransformer2DModel.state_dict()
    B, lh, lw, nt = g["shape"]
    lat, pe, pooled, img_ids, txt_ids = FO.make_flux_inputs(cfg, B, lh, lw, nt, seed=g["seed"] + 1)
    with torch.no_grad():
        y = FO.flux_forward(w, cfg, lat, pe, pooled, g["t"], img_ids, txt_ids, guidance=g["guidance"])
    torch.testing.assert_close(y, g["y32"], rtol=1e-5, atol=1e-5)
    wb = {k: v.bfloat16() for k, v in w.items()}
    threads = torch.get_num_threads()
    torch.set_num_threads(8)       # as the fixtures were minted (make_golden.py): above 8 threads the bf16 GEMMs split their sums differently
    try:
        with torch.no_grad(), torch.autocast("cpu", dtype=torch.bfloat16):
            yb = FO.flux_forward(wb, cfg, lat.bfloat16(), pe.bfloat16(), pooled.bfloat16(), g["t"].bfloat16(), img_ids.bfloat16(),
                                 txt_ids.bfloat16(), guidance=g["guidance"].bfloat16())
    finally:
        torch.set_num_threads(threads)
    assert torch.equal(yb, g["y_bf16_cpu_autocast"])   # same ops, same order -> bit exact on CPU


def test_flux_rollout_loop_matches_reference(golden_dir):
    g = _load(golden_dir)["rollout_fp32"]
    cfg = FO.tiny_flux_config()
    w = FO.make_flux_weights(cfg, seed=0)
    lat, pe, pooled, img_ids, _ = FO.make_flux_inputs(cfg, 2, 8, 8, 7, seed=1)
    ts, sig = FO.flux_make_schedule(4, lat.shape[1])
    assert torch.equal(ts, g["timesteps"]) and torch.equal(sig, g["sigmas"])
    noises = O.make_noises(4, tuple(lat.shape), seed=123)
    with torch.no_grad():
        r = FO.flux_rollout(w, cfg, lat, pe, pooled, img_ids, 4, 3.5, noises=noises)
    for a, b in zip(r["latents"], g["latents"]):
        torch.testing.assert_close(a.float(), b.float(), rtol=2e-3, atol=2e-3)
    assert sorted(r["log_probs"]) == sorted(g["log_probs"])
    for i in r["log_probs"]:
        torch.testing.assert_close(r["log_probs"][i], g["log_probs"][i], rtol=1e-5, atol=1e-6)
