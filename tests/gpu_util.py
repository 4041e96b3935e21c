"""Helpers for the -m gpu parity tests: call the C ABI through ctypes on torch-owned device memory."""
import contextlib
import ctypes as C
import json
import os

import torch

from flow_factory_b200 import _lib

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")


def stream():
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    return None if t is None else t.data_ptr()


def dump(name, obj):
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, name), "w") as f:
        json.dump(obj, f, indent=1, default=lambda o: o.tolist() if hasattr(o, "tolist") else str(o))


def record(file: str, obj):
    """Append one JSON line to gpurun_out/<file>: the MEASURED error of every parity case, so tolerances can be set from numbers."""
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, file), "a") as f:
        f.write(json.dumps(obj, default=lambda o: o.tolist() if hasattr(o, "tolist") else str(o)) + "\n")


def err_report(got: torch.Tensor, ref: torch.Tensor, tag: str):
    g, r = got.float(), ref.float()
    d = (g - r).abs()
    rep = dict(tag=tag, shape=list(g.shape), max_abs=float(d.max()), mean_abs=float(d.mean()), ref_absmax=float(r.abs().max()),
               got_absmax=float(g.abs().max()), n_nan=int(torch.isnan(g).sum()),
               frac_bad=float((d > 0.05 * r.abs().max()).float().mean()))
    record("parity_measured.jsonl", {k: rep[k] for k in ("tag", "max_abs", "mean_abs", "ref_absmax", "n_nan")})
    if g.dim() == 2:
        bad = d > 0.05 * r.abs().max()
        rep["bad_rows_first"] = bad.any(1).nonzero().flatten()[:16].tolist()
        rep["bad_cols_first"] = bad.any(0).nonzero().flatten()[:16].tolist()
        rep["got_00"] = g[:2, :8].tolist()
        rep["ref_00"] = r[:2, :8].tolist()
    return rep


def chunked_sdpa(q, k, v, attn_mask=None, dropout_p=0.0, is_causal=False, scale=None):
    """fp32 softmax(q k^T * scale) v over [B, H, S, d], a block of query rows at a time so that no score matrix exceeds ~2 GB
    (torch's math backend would hold all B x H x Sq x Skv scores; Wan2.1 at 20 280 tokens needs 40 GB of them).
    `attn_mask`: bool, True = attend (the Qwen-Image key-padding mask)."""
    assert dropout_p == 0.0 and not is_causal and q.dtype == torch.float32, (dropout_p, is_causal, q.dtype)
    scale = q.shape[-1] ** -0.5 if scale is None else scale
    B, H, Sq, _ = q.shape
    step = max(1, (1 << 29) // (B * H * k.shape[-2]))
    kt = k.transpose(-1, -2)
    out = torch.empty(*q.shape[:-1], v.shape[-1], dtype=q.dtype, device=q.device)
    for s in range(0, Sq, step):
        sc = torch.matmul(q[..., s:s + step, :], kt) * scale
        if attn_mask is not None:
            sc = sc.masked_fill(~attn_mask, float("-inf"))
        out[..., s:s + step, :] = torch.matmul(sc.softmax(-1), v)
    return out


@contextlib.contextmanager
def ieee_fp32():
    """The fp32 truth of a parity test in IEEE fp32: TF32 off for matmul and cuDNN (torch enables it for cuDNN convolutions by
    default), and scaled_dot_product_attention - which the oracles call through torch.nn.functional - replaced by chunked_sdpa.
    Everything is restored on exit; bf16-autocast references must run outside this context."""
    import torch.nn.functional as F
    saved = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, F.scaled_dot_product_attention
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    F.scaled_dot_product_attention = chunked_sdpa
    try:
        with torch.no_grad():
            yield
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, F.scaled_dot_product_attention = saved


from flow_factory_b200.ops import linear  # noqa: E402,F401


def device_error():
    buf = (C.c_uint * 4)()
    _lib.lib().ffb200_device_error(C.byref(buf))
    return [hex(x) for x in buf]
