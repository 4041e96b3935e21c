"""oracle/ref_runner.py (the reference's OWN classes from oracle/_ref, the CPU arm of bench.py) against the pinned oracle restatement: the
4-step CFG rollout of the tiny configuration is bit-identical under bf16 CPU autocast - i.e. the bench's reference arm calls the reference
the way the golden fixtures were minted (tests/golden/make_golden.py, whose record of that loop stands in for it where oracle/_ref has not
been laid out)."""
import os

import pytest
import torch

from oracle import ref_runner as R
from oracle import sd3_oracle as O

needs_reference = pytest.mark.skipif(not R.available(), reason="oracle/_ref absent (run tools/make_oracle_ref.py where the original project is)")


def reference_loop(T: int = 4):
    """The 4-step CFG loop of the tiny configuration through ref_runner: (latents after each step incl. the initial ones, log-probs)."""
    torch.set_num_threads(4)
    cfg = O.tiny_config()
    model = R.build_model(cfg, O.make_weights(cfg, seed=0))
    sched, ts = R.make_scheduler(T, 64, num_sde_steps=None)
    inp = {k: v.bfloat16() for k, v in O.make_inputs(cfg, 2, 16, 16, 13, seed=1).items()}
    x = inp["x0"].half()
    torch.manual_seed(123)                       # the reference draws its step noise from the global CPU RNG
    lat, lps = [x], []
    for i in range(T):
        out = R.reference_step(model, sched, ts, i, x, inp["prompt_embeds"], inp["pooled"], inp["neg_prompt_embeds"], inp["neg_pooled"], 4.5)
        x = out.next_latents.half()
        lat.append(x); lps.append(out.log_prob)
    return lat, lps


@needs_reference
def test_reference_classes_come_from_oracle_ref():
    SD3, Sched, _ = R.load()
    import inspect
    assert inspect.getsourcefile(SD3).startswith(R.REF_DIR) and inspect.getsourcefile(Sched).startswith(R.REF_DIR)


def test_reference_step_loop_equals_the_pinned_oracle(golden_dir):
    g = torch.load(os.path.join(golden_dir, "rollout_tiny.pt"), weights_only=False)["bf16"]     # the reference's loop, bf16 CPU autocast
    lat, lps = reference_loop() if R.available() else (g["latents"], g["log_probs"])
    for a, b in zip(lat, g["latents"]):
        assert torch.equal(a.float(), b.float())
    for i, lp in g["log_probs"].items():
        assert torch.equal(lps[i], lp)
    T = 4
    cfg = O.tiny_config()
    w = O.make_weights(cfg, seed=0)
    inp = {k: v.bfloat16() for k, v in O.make_inputs(cfg, 2, 16, 16, 13, seed=1).items()}
    noises = O.make_noises(T, (2, 16, 16, 16), seed=123)
    rb = O.rollout({k: v.bfloat16() for k, v in w.items()}, cfg, inp["x0"], inp["prompt_embeds"], inp["pooled"], inp["neg_prompt_embeds"],
                   inp["neg_pooled"], T, 4.5, noises=noises, autocast="cpu")
    assert len(rb["latents"]) == len(lat)
    for a, b in zip(lat, rb["latents"]):
        assert torch.equal(a.float(), b.float())
    for i, lp in rb["log_probs"].items():
        assert torch.equal(lps[i], lp)


def test_truncated_model_shares_modules_and_block_flops_add_up():
    cfg = O.tiny_config()
    if R.available():
        model = R.build_model(cfg, O.make_weights(cfg, seed=0))
    else:                                        # truncated() only touches the module dict and the block list
        model = torch.nn.Module()
        model.transformer_blocks = torch.nn.ModuleList(torch.nn.Linear(2, 2) for _ in range(cfg.num_layers))
        model.proj_out = torch.nn.Linear(2, 2)
    t1 = R.truncated(model, 1)
    assert len(t1.transformer_blocks) == 1 and len(model.transformer_blocks) == 2 and t1.transformer_blocks[0] is model.transformer_blocks[0]
    full = O.sd35_medium()
    lin, att = O.flops_per_forward(full, 4096, 333)
    assert abs(R.block_flops(full, 4096, 333, full.num_layers) - (lin + att)) / (lin + att) < 1e-12
    assert R.pick_cores()["n"] >= 1
