"""Parity of the native VAE decode (csrc/vae_*.cu, SURVEY 8f row 3) against torch ops and the pinned oracle, through the C ABI.

First green run on a B200: round 2 (gpurun call 1, 23 passed)."""
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from flow_factory_b200 import vae as V          # noqa: E402
from oracle import vae_oracle as VO              # noqa: E402  (the checker)
from tests.gpu_util import ieee_fp32, record     # noqa: E402

DEV = "cuda"


def _rel(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-12))


@pytest.mark.parametrize("B,H,W,cin,cout", [(1, 16, 128, 64, 64), (2, 12, 20, 32, 64), (1, 33, 47, 128, 256), (2, 8, 8, 16, 32),
                                              (1, 64, 256, 256, 128), (3, 5, 6, 64, 8)])
@pytest.mark.parametrize("residual", [False, True])
def test_conv3x3_matches_torch(B, H, W, cin, cout, residual):
    g = torch.Generator(device=DEV).manual_seed(B * 1000 + H + W + cin + cout)
    x = torch.randn(B, H, W, cin, generator=g, device=DEV).bfloat16()
    w = (torch.randn(cout, cin, 3, 3, generator=g, device=DEV) / (3 * cin ** 0.5)).bfloat16()
    b = (torch.randn(cout, generator=g, device=DEV) * 0.1).bfloat16()
    res = torch.randn(B, H, W, cout, generator=g, device=DEV).bfloat16() if residual else None
    out = V.conv2d_nhwc(x, w, b, res)
    with ieee_fp32():
        ref = F.conv2d(x.permute(0, 3, 1, 2).float(), w.float(), b.float(), padding=1).permute(0, 2, 3, 1)
    ref = ref.bfloat16().float()
    if residual:
        ref = (ref + res.float())
    assert out.shape == (B, H, W, cout)
    assert torch.isfinite(out.float()).all()
    torch.testing.assert_close(out.float(), ref.bfloat16().float(), rtol=2e-2, atol=2e-2)
    assert _rel(out, ref) < 6e-3


@pytest.mark.parametrize("rows,cin,cout", [(256, 64, 128), (240, 512, 1024), (1000, 96, 64)])
def test_conv1x1_matches_linear(rows, cin, cout):
    g = torch.Generator(device=DEV).manual_seed(rows + cin)
    x = torch.randn(1, 1, rows, cin, generator=g, device=DEV).bfloat16()
    w = (torch.randn(cout, cin, generator=g, device=DEV) / cin ** 0.5).bfloat16()
    b = (torch.randn(cout, generator=g, device=DEV) * 0.1).bfloat16()
    out = V.conv2d_nhwc(x, w, b)
    with ieee_fp32():
        ref = F.linear(x.float(), w.float(), b.float())
    assert _rel(out, ref) < 6e-3


@pytest.mark.parametrize("B,P,C,groups,silu", [(2, 240, 64, 8, True), (1, 4096, 128, 32, True), (3, 1000, 512, 32, False), (2, 77, 32, 8, True)])
def test_group_norm_matches_torch(B, P, C, groups, silu):
    g = torch.Generator(device=DEV).manual_seed(P + C)
    x = (torch.randn(B, P, C, generator=g, device=DEV) * 2 + 0.5).bfloat16()
    gamma = (1 + 0.1 * torch.randn(C, generator=g, device=DEV)).bfloat16()
    beta = (0.1 * torch.randn(C, generator=g, device=DEV)).bfloat16()
    out = V.group_norm_nhwc(x, gamma, beta, groups, 1e-6, silu)
    with ieee_fp32():
        ref = F.group_norm(x.float().permute(0, 2, 1), groups, gamma.float(), beta.float(), 1e-6).permute(0, 2, 1)
    if silu:
        ref = F.silu(ref)
    torch.testing.assert_close(out.float(), ref.bfloat16().float(), rtol=1.6e-2, atol=1e-2)
    assert _rel(out, ref) < 4e-3


def _decode_case(ocfg, lat, batch, seed):
    w32 = {k: v.to(torch.bfloat16).float() for k, v in VO.make_vae_decoder_weights(ocfg, seed=seed).items()}
    cfg = V.VaeDecoderConfig(ocfg.latent_channels, ocfg.out_channels, tuple(ocfg.block_out_channels), ocfg.layers_per_block,
                             ocfg.norm_num_groups, ocfg.scaling_factor, ocfg.shift_factor)
    dec = V.B200VaeDecoder(cfg, w32, lat.shape[2], lat.shape[3], batch=batch, device=DEV)
    img = dec.decode(lat.half())
    torch.cuda.synchronize()
    wd = {k: v.to(DEV) for k, v in w32.items()}
    lat16 = lat.half().float().to(DEV)
    with ieee_fp32():
        truth = VO.vae_decode(wd, ocfg, lat16)                                   # IEEE fp32
    with torch.no_grad():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            ref16 = VO.vae_decode({k: v.bfloat16() for k, v in wd.items()}, ocfg, lat16.bfloat16())   # the reference's bf16 autocast numerics
    return img, truth, ref16, dec


def test_decode_tiny_golden(golden_dir):
    """The reference-minted fixture (real AutoencoderKL.decode, fp32, CPU): engine error against it bounded by the bf16 reference's."""
    e = torch.load(os.path.join(golden_dir, "vae_tiny.pt"), weights_only=False)["tiny"]
    ocfg = VO.tiny_vae_config()
    w = VO.make_vae_decoder_weights(ocfg, seed=0)
    cfg = V.VaeDecoderConfig(ocfg.latent_channels, ocfg.out_channels, tuple(ocfg.block_out_channels), ocfg.layers_per_block,
                             ocfg.norm_num_groups, ocfg.scaling_factor, ocfg.shift_factor)
    dec = V.B200VaeDecoder(cfg, w, 6, 10, batch=2, device=DEV)
    img = dec.decode(e["lat"].half().to(DEV))
    assert tuple(img.shape) == (2, 3, 12, 20) and img.dtype == torch.bfloat16
    assert _rel(img.cpu(), e["img"]) < 3e-2          # bf16 weights + bf16 activations against the fp32 reference
    assert V.B200VaeDecoder.last_launch_count() > 20


@pytest.mark.parametrize("name,ocfg,shape,batch", [
    ("two_levels", VO.VaeConfig(latent_channels=16, block_out_channels=(64, 128), layers_per_block=1, norm_num_groups=32), (3, 16, 24, 40), 2),
    ("shortcuts", VO.VaeConfig(latent_channels=16, block_out_channels=(32, 64, 128), layers_per_block=2, norm_num_groups=16), (2, 16, 16, 16), 2),
])
def test_decode_matches_oracle(name, ocfg, shape, batch):
    lat = torch.randn(*shape, generator=torch.Generator().manual_seed(5))
    img, truth, ref16, dec = _decode_case(ocfg, lat, batch, seed=7)
    assert torch.isfinite(img.float()).all()
    e_eng, e_ref = _rel(img, truth), _rel(ref16, truth)
    record("parity_measured.jsonl", dict(tag=f"vae_decode_{name}", e_engine=e_eng, e_ref_bf16=e_ref, ratio=e_eng / e_ref))
    assert e_eng <= 1.3 * e_ref + 5e-4, (e_eng, e_ref)       # as close to fp32 as the reference's own bf16 path; measured on B200: 0.89, 0.90 x
    assert _rel(img, ref16) < 4 * e_ref + 2e-3
    assert torch.allclose(V.postprocess_pt(img).float(), (img.float() / 2 + 0.5).clamp(0, 1), atol=1e-2)


def test_decode_sd35_geometry_smoke():
    """SD3.5 VAE architecture (128/256/512/512 channels, 32 groups, 4096-token mid-block attention) at 512^2 (latent 64 x 64)."""
    ocfg = VO.sd35_vae()
    lat = torch.randn(1, 16, 64, 64, generator=torch.Generator().manual_seed(9))
    img, truth, ref16, dec = _decode_case(ocfg, lat, 1, seed=11)
    e_eng, e_ref = _rel(img, truth), _rel(ref16, truth)
    record("parity_measured.jsonl", dict(tag="vae_decode_sd35_512", e_engine=e_eng, e_ref_bf16=e_ref, ratio=e_eng / e_ref))
    assert e_eng <= 1.3 * e_ref + 5e-4, (e_eng, e_ref)          # measured on B200 against the IEEE fp32 truth: 0.87 x
    assert dec.workspace_bytes() < 8 << 30
