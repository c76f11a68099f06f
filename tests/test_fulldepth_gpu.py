"""Full-depth parity of the BENCHMARKED model on the B200: LLaMA-7B x 32 layers, CLIP ViT-L/14 x 24, Whisper-base x 6,
V = 32000 — BASELINE configs 2 (image+text, B=1, L=256) and 3 (audio+text, one sample of the batch, L=512) — against the
fp32 CPU oracle on the SAME bf16-rounded random weights and inputs.  (bench.py repeats the check on a cfg4 sample against
the unmodified reference and prints it as `parity` in its JSON line.)

Bars (norm-wise relative error).  north_star's "1e-3 relative bf16" is ONE bf16 rounding of an output (measured
1.3-1.5e-3 norm-wise in tests/test_model_gpu.py::test_real_width_alignment_block, where the alignment block alone is held
to 1.35x that).  Here the aligned prefix rows also carry the error of the 24 (6) bf16-stored encoder layers in front of
the block, and the logits that of 32 bf16-stored decoder layers, so both are held to (a) an absolute bar and (b) the
REFERENCE ALGORITHM'S OWN bf16 arithmetic measured in the same test (the oracle run in bf16 vs fp32 on the same sample).
Measured on the B200 (round 2): cfg2 prefix 4.5e-3 (reference-bf16 5.6e-3), logits 4.1e-2 at 32 layers (reference-bf16
2.8e-2 after 4 layers); cfg3 prefix 2.6e-3 (4.3e-3), logits 4.2e-2 (3.1e-2 after 4 layers)."""
import copy

import pytest
import torch

from tests import helpers as H

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def full():
    import bench
    from macaw_llm_b200.modeling import MM_LLMs, MM_LLMs_Config
    from oracle import macaw_oracle as O

    (clip, whisper, llama), hyper = bench.real_configs()
    cfg = MM_LLMs_Config(clip_config=clip, whisper_config=whisper, llm_config=llama, **hyper)
    model = MM_LLMs.build_random(cfg, device="cuda", dtype=torch.bfloat16, seed=0)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items() if not k.startswith("video_encoder")}
    return model, cfg, O.hp_from_config(cfg), sd, bench


def _run(full, modality, L, seed):
    from oracle import macaw_oracle as O

    model, cfg, hp, sd, bench = full
    V = cfg.llm_config.vocab_size
    inp = bench.synth_inputs(1, L, V, 224, 3000, seed, pin=False)
    if modality == "image":
        inp["audios"] = None
    else:
        inp["images"] = None
    dev_inp = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in inp.items()}
    out = model(dev_inp)
    emb, mask, _ = model.prepare_inputs_for_generation(dev_inp)
    torch.cuda.synchronize()
    torch.set_num_threads(bench.cpu_threads())
    ref = O.forward({k: (v.float() if isinstance(v, torch.Tensor) and v.is_floating_point() else v) for k, v in inp.items()},
                    sd, hp, dtype=torch.float32)
    n_prefix = emb.shape[1] - L
    assert n_prefix == 8 and torch.equal(mask.cpu(), ref["attention_mask"])
    # integer / layout side: text rows are pure gathers of bf16 table rows
    table = sd["llm.model.embed_tokens.weight"]
    assert torch.equal(emb[:, 1 + n_prefix:].cpu(), table[inp["input_ids"][:, 1:]])
    e_pre = H.rel_err(emb[:, 2:1 + n_prefix - 1], ref["embeds"][:, 2:1 + n_prefix - 1])  # the 6 aligned rows
    e_log = H.rel_err(out.logits.cpu(), ref["logits"])
    agree = float((out.logits.cpu().float().argmax(-1) == ref["logits"].argmax(-1)).float().mean())
    return e_pre, e_log, agree, inp, ref


def _reference_bf16_drift(full, inp, layers=4):
    """The reference algorithm's own bf16-vs-fp32 drift: aligned prefix rows at FULL encoder depth, logits on a
    depth-reduced LLaMA (CPU bf16 matmuls are slow)."""
    from oracle import macaw_oracle as O

    model, cfg, hp, sd, bench = full
    hp2 = copy.deepcopy(hp)
    hp2["llama"]["layers"] = layers
    f = {k: (v.float() if isinstance(v, torch.Tensor) and v.is_floating_point() else v) for k, v in inp.items()}
    a = O.forward(f, sd, hp2, dtype=torch.float32)
    b = O.forward(f, sd, hp2, dtype=torch.bfloat16)
    return H.rel_err(b["logits"], a["logits"]), H.rel_err(b["embeds"][:, 2:8], a["embeds"][:, 2:8]), layers


def test_cfg2_image_text_full_depth(full):
    e_pre, e_log, agree, inp, ref = _run(full, "image", 256, 1234)
    d_log, d_pre, n = _reference_bf16_drift(full, inp)
    print(f"\n[full depth cfg2: CLIP-L x24 + align + LLaMA-7B x32, B=1, T=264] prefix {e_pre:.3e}  logits {e_log:.3e}  "
          f"argmax agreement {agree:.4f}  | reference algorithm in bf16: prefix {d_pre:.3e}, logits at {n} layers {d_log:.3e}")
    assert e_pre < 6e-3 and e_pre < 1.5 * d_pre   # 24 bf16-stored CLIP layers in front of the block
    # A random-init 32-layer decoder amplifies any perturbation: the REFERENCE ALGORITHM's own bf16 arithmetic drifts
    # 2.8e-2 after only 4 layers (measured above; ~sqrt(depth) growth), so 1e-2 at full depth is not reachable in bf16 by
    # any implementation.  Bars: absolute 6e-2, and no worse than the reference's bf16 drift extrapolated to 32 layers.
    # Random-init logits are nearly flat, so top-1 flips where two logits tie within the error: agreement > 0.85.
    assert e_log < 6e-2
    assert agree > 0.85
    assert e_log < d_log * (32 / n) ** 0.5


def test_cfg3_audio_text_full_depth(full):
    e_pre, e_log, agree, inp, ref = _run(full, "audio", 512, 4321)
    d_log, d_pre, n = _reference_bf16_drift(full, inp)
    print(f"\n[full depth cfg3 sample: Whisper-base x6 + align + LLaMA-7B x32, B=1, T=520] prefix {e_pre:.3e}  "
          f"logits {e_log:.3e}  argmax agreement {agree:.4f}  | reference algorithm in bf16: prefix {d_pre:.3e}, "
          f"logits at {n} layers {d_log:.3e}")
    assert e_pre < 4e-3 and e_pre < 1.5 * d_pre   # 6 bf16-stored Whisper layers in front of the block
    assert e_log < 6e-2 and e_log < d_log * (32 / n) ** 0.5   # see test_cfg2_image_text_full_depth
    assert agree > 0.85
