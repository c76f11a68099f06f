"""Generate golden fixtures by running the UNMODIFIED reference (/root/reference/modeling.py) in-process on CPU.

Runs only where /root/reference exists (the build container); the fixtures it writes (tests/golden/*.npz, *.json)
are committed and replayed by tests/test_oracle.py and the GPU parity tests on any box.

Shims (SURVEY.md §8c; both are host-side, the reference source is untouched):
  1. modeling.py:25 imports PretrainedConfig from transformers.modeling_utils, which no longer re-exports it.
  2. modeling.py:939 calls init_weights() without post_init(); transformers 5.x then lacks all_tied_weights_keys.

Usage:  PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tests.golden import gen  # noqa: E402
from oracle import macaw_oracle as O  # noqa: E402


def import_reference():
    import transformers.modeling_utils as mu
    from transformers import PretrainedConfig, PreTrainedModel

    mu.PretrainedConfig = PretrainedConfig  # shim 1
    # load under a private module name so the repo's own drop-in `modeling` module is not shadowed
    import importlib.util

    spec = importlib.util.spec_from_file_location("_macaw_reference_modeling", "/root/reference/modeling.py")
    modeling = importlib.util.module_from_spec(spec)
    sys.modules["_macaw_reference_modeling"] = modeling
    spec.loader.exec_module(modeling)

    _orig = PreTrainedModel.init_weights

    def _iw(self):  # shim 2
        return self.post_init() if not hasattr(self, "all_tied_weights_keys") else _orig(self)

    modeling.MM_LLMs.init_weights = _iw
    return modeling


def build_reference(modeling, spec):
    clip, whisper, llama = gen.build_configs(spec)
    extra = {}
    for name in ("image", "video", "audio"):
        if f"{name}_conv" in spec:
            extra[f"{name}_conv_kernel"], extra[f"{name}_conv_stride"] = spec[f"{name}_conv"]
    cfg = modeling.MM_LLMs_Config(n_frames=spec["n_frames"], attention_heads=spec["attention_heads"],
                                  clip_config=clip, whisper_config=whisper, llm_config=llama, **extra)
    model = modeling.MM_LLMs(cfg).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    weights = gen.make_weights(shapes, seed=0)
    missing, unexpected = model.load_state_dict(weights, strict=False)
    assert not unexpected, unexpected
    assert all(any(s in m for s in gen.SKIP_SUBSTR) for m in missing), missing
    return cfg, model, shapes, weights


CASES = [
    # name, B, L, modalities, pad_tail, labels
    ("all3", 2, 16, ("image", "audio", "video"), 3, True),
    ("image", 1, 12, ("image",), 0, False),
    ("audio", 2, 10, ("audio",), 0, True),
    # text-only WITH labels crashes in the reference itself (modeling.py:1043: empty float tensor cat -> float labels)
    ("text", 2, 9, (), 2, False),
]


def main():
    torch.manual_seed(0)
    modeling = import_reference()
    spec = gen.TINY
    cfg, model, shapes, weights = build_reference(modeling, spec)
    hp = O.hp_from_config(cfg)
    with open(os.path.join(HERE, "tiny_shapes.json"), "w") as f:
        json.dump({"spec": spec, "hp": hp, "shapes": {k: list(v) for k, v in shapes.items()}}, f, indent=0,
                  sort_keys=True)

    # fp64 pin of the oracle against the reference itself
    model64 = model.double()
    sd64 = {k: v.double() for k, v in model64.state_dict().items()}
    for name, B, L, mods, pad, with_labels in CASES:
        inp = gen.make_inputs(spec, B, L, seed=100 + len(name), modalities=mods, pad_tail=pad, with_labels=with_labels)
        inp64 = {k: (v.double() if isinstance(v, torch.Tensor) and v.is_floating_point() else v) for k, v in inp.items()}
        with torch.no_grad():
            emb_r, mask_r, lab_r = model64.prepare_inputs_for_generation(inp64)
            out_r = model64(inp64)
        o = O.forward(inp64, sd64, hp, dtype=torch.float64)
        e_emb = float((o["embeds"] - emb_r).abs().max())
        e_log = float((o["logits"] - out_r.logits).abs().max())
        # the reference softmaxes in fp32 even when run in fp64 (HF eager attention; modeling.py:214), hence 1e-6 not 1e-12
        assert e_emb < 1e-6 and e_log < 1e-5, (name, e_emb, e_log)
        assert (mask_r is None) == (o["attention_mask"] is None) and (lab_r is None) == (o["labels"] is None)
        if mask_r is not None:
            assert torch.equal(mask_r.long(), o["attention_mask"])
        if lab_r is not None:
            assert torch.equal(lab_r.long(), o["labels"])
            assert abs(float(out_r.loss) - float(o["loss"])) < 1e-6
        print(f"[golden] {name}: oracle vs reference fp64 max|d| embeds {e_emb:.2e} logits {e_log:.2e}  T={emb_r.shape[1]}")
        np.savez_compressed(
            os.path.join(HERE, f"tiny_{name}.npz"),
            B=B, L=L, seed=100 + len(name), pad_tail=pad, with_labels=int(with_labels),
            modalities=np.array(list(mods), dtype="U8"),
            embeds=emb_r.float().numpy(), logits=out_r.logits.float().numpy(),
            attention_mask=(mask_r.long().numpy() if mask_r is not None else np.zeros(0, dtype=np.int64)),
            labels=(lab_r.long().numpy() if lab_r is not None else np.zeros(0, dtype=np.int64)),
            loss=(float(out_r.loss) if out_r.loss is not None else np.nan),
        )

    # second shape family (gen.ALT): oracle pinned on the reference in fp64, fixture replayed by tests/test_oracle.py
    cfg2, model2, shapes2, _ = build_reference(modeling, gen.ALT)
    hp2 = O.hp_from_config(cfg2)
    with open(os.path.join(HERE, "alt_shapes.json"), "w") as f:
        json.dump({"spec": gen.ALT, "hp": hp2, "shapes": {k: list(v) for k, v in shapes2.items()}}, f, indent=0,
                  sort_keys=True)
    model2 = model2.double()
    sd2 = {k: v.double() for k, v in model2.state_dict().items()}
    inp = gen.make_inputs(gen.ALT, 2, 13, seed=321, pad_tail=4)
    inp64 = {k: (v.double() if isinstance(v, torch.Tensor) and v.is_floating_point() else v) for k, v in inp.items()}
    with torch.no_grad():
        emb_r, mask_r, lab_r = model2.prepare_inputs_for_generation(inp64)
        out_r = model2(inp64)
    o = O.forward(inp64, sd2, hp2, dtype=torch.float64)
    e_emb, e_log = float((o["embeds"] - emb_r).abs().max()), float((o["logits"] - out_r.logits).abs().max())
    assert e_emb < 1e-6 and e_log < 1e-5, (e_emb, e_log)
    assert torch.equal(mask_r.long(), o["attention_mask"]) and torch.equal(lab_r.long(), o["labels"])
    print(f"[golden] alt family: oracle vs reference fp64 max|d| embeds {e_emb:.2e} logits {e_log:.2e}  T={emb_r.shape[1]}")
    np.savez_compressed(os.path.join(HERE, "alt_all3.npz"), B=2, L=13, seed=321, pad_tail=4,
                        embeds=emb_r.float().numpy(), logits=out_r.logits.float().numpy(),
                        attention_mask=mask_r.long().numpy(), labels=lab_r.long().numpy(), loss=float(out_r.loss))

    # stand-alone pieces with their own fixtures: video PE table (python double loop in the reference) and one MHA
    pe_ref = modeling.create_positional_encoding(40, 24)
    pe_orc = O.video_positional_encoding(40, 24)
    assert torch.equal(pe_ref, pe_orc), float((pe_ref - pe_orc).abs().max())
    np.savez_compressed(os.path.join(HERE, "video_pe_40x24.npz"), pe=pe_ref.numpy())
    print("[golden] video positional encoding: bit-exact vs reference loop")
    reference_outputs(modeling)


def reference_outputs(modeling):
    """What the reference itself returns, recorded for the tests that compare with it:
    ref_image_audio.npz   fp32 `MM_LLMs.forward` of the tiny model on an image+audio batch (tests/test_oracle.py);
    ref_state_dict_resized.json   names / shapes / dtypes of the state_dict the reference writes after
                                  `model.llm.resize_token_embeddings(V + 7)` (run_clm_llms.py:495; tests/test_wire.py)."""
    _, model, _, _ = build_reference(modeling, gen.TINY)
    B, L, seed, pad = 2, 11, 7, 2
    mods = ("image", "audio")
    inp = gen.make_inputs(gen.TINY, B, L, seed=seed, modalities=mods, pad_tail=pad)
    with torch.no_grad():
        out = model(inp)
    np.savez_compressed(os.path.join(HERE, "ref_image_audio.npz"), B=B, L=L, seed=seed, pad_tail=pad,
                        modalities=np.array(list(mods), dtype="U8"), logits=out.logits.float().numpy(),
                        loss=float(out.loss))
    print(f"[golden] reference image+audio forward: logits {tuple(out.logits.shape)}, loss {float(out.loss):.6f}")
    model.llm.resize_token_embeddings(gen.TINY["llama"]["vocab_size"] + 7)
    layout = {k: [list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in model.state_dict().items()}
    with open(os.path.join(HERE, "ref_state_dict_resized.json"), "w") as f:
        json.dump(layout, f, indent=0, sort_keys=True)
    print(f"[golden] reference state_dict after resize_token_embeddings: {len(layout)} entries")


if __name__ == "__main__":
    main()
