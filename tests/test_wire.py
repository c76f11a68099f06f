"""CPU tier: checkpoint / wire compatibility (SURVEY.md §8f rank 4) — save_pretrained -> from_pretrained round trips,
deep copies, a state_dict produced by the LIVE reference with the resized 32007-style table, the tokenizer's special ids
and the pickle dataset schema."""
import copy
import os
import pickle

import pytest
import torch

from tests import helpers as H
from tests.golden import gen


def _tiny_cfg():
    from macaw_llm_b200.modeling import MM_LLMs_Config

    clip, whisper, llama = gen.build_configs(gen.TINY)
    return MM_LLMs_Config(n_frames=2, attention_heads=2, clip_config=clip, whisper_config=whisper, llm_config=llama)


def _same_state(a, b):
    sa, sb = a.state_dict(), b.state_dict()
    assert set(sa) == set(sb)
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k


def test_save_pretrained_from_pretrained_roundtrip(tmp_path):
    """reference run_clm_llms.py:563 (trainer.save_model) -> run_clm_llms_inference.py:455-457 (from_pretrained)."""
    from macaw_llm_b200.modeling import MM_LLMs, MM_LLMs_Config

    torch.manual_seed(0)
    m = MM_LLMs(_tiny_cfg())
    m.save_pretrained(tmp_path)
    assert os.path.exists(os.path.join(tmp_path, "config.json"))
    # (a) the reference's call: config passed explicitly
    cfg = MM_LLMs_Config.from_pretrained(tmp_path)
    m2 = MM_LLMs.from_pretrained(tmp_path, config=cfg)
    _same_state(m, m2)
    # (b) without config=: PreTrainedModel.from_pretrained asks the config class for (config, unused_kwargs)
    m3 = MM_LLMs.from_pretrained(tmp_path)
    _same_state(m, m3)
    c, unused = MM_LLMs_Config.from_pretrained(tmp_path, return_unused_kwargs=True, n_frames=4, foo=1)
    assert c.n_frames == 4 and unused == {"foo": 1}
    assert m3.engine is not m.engine and m3.llm._engine_ref() is m3.engine


def test_deepcopy_and_pickle_get_their_own_engine(tmp_path):
    from macaw_llm_b200.modeling import MM_LLMs

    m = MM_LLMs(_tiny_cfg())
    c = copy.deepcopy(m)
    _same_state(m, c)
    assert c.engine is not m.engine and c.engine.m is c and c.llm._engine_ref() is c.engine
    assert c.llm.model.embed_tokens.weight.data_ptr() != m.llm.model.embed_tokens.weight.data_ptr()
    p = os.path.join(tmp_path, "m.pt")
    torch.save(m, p)
    r = torch.load(p, weights_only=False)
    _same_state(m, r)
    assert r.engine.m is r and r.llm._engine_ref() is r.engine


def test_train_mode_is_loud_without_labels_or_cuda():
    """train()-mode forward goes to the kernel-library training step: it refuses to run without labels (the loss is what
    is differentiated) and — like every other path — without CUDA parameters; it never hands back a graph-less loss."""
    from macaw_llm_b200.modeling import MM_LLMs

    m = MM_LLMs(_tiny_cfg()).train()
    spec, _, _ = H.load_shapes()
    with pytest.raises(ValueError, match="needs `labels`"):
        m(H.case_inputs(spec, H.load_case("text")))
    from tests.golden import gen as G

    inp = G.make_inputs(spec, 2, 8, seed=1, modalities=(), with_labels=True)
    with pytest.raises(RuntimeError, match="no CPU"):
        m(inp)


def test_loads_live_reference_state_dict_with_resized_table():
    """A checkpoint written by the reference after `model.llm.resize_token_embeddings(len(tokenizer))`
    (run_clm_llms.py:495; +7 rows: six modal tokens + [PAD]) loads key-for-key, shape-for-shape.  The checkpoint's layout
    (names, shapes, dtypes) was recorded from the unmodified reference (tests/golden/ref_state_dict_resized.json, written
    by make_golden.reference_outputs); its values are name-seeded."""
    import json

    from macaw_llm_b200.modeling import MM_LLMs

    with open(os.path.join(H.GOLDEN, "ref_state_dict_resized.json")) as f:
        layout = json.load(f)
    sd = {k: gen.make_tensor(k, tuple(shape), seed=0).to(getattr(torch, dtype)) for k, (shape, dtype) in layout.items()}
    V = gen.TINY["llama"]["vocab_size"]
    assert sd["llm.model.embed_tokens.weight"].shape[0] == V + 7 and sd["llm.lm_head.weight"].shape[0] == V + 7
    m = MM_LLMs(_tiny_cfg())
    m.llm.resize_token_embeddings(V + 7)
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.endswith(("inv_freq", "position_ids")) for k in missing), (missing, unexpected)
    assert torch.equal(m.llm.model.embed_tokens.weight, sd["llm.model.embed_tokens.weight"])
    assert set(m.state_dict()) == set(sd)


def test_special_ids_cache_schema_and_inputs_dict(tmp_path):
    from macaw_llm_b200 import wire

    assert [wire.SPECIAL_TOKENS[t] for t in ("<image>", "</image>", "<audio>", "</audio>", "<video>", "</video>")] == \
        list(range(32000, 32006))
    assert wire.PAD_TOKEN_ID == 32006 and wire.VOCAB_WITH_SPECIALS == 32007 and wire.IGNORE_INDEX == -100
    n, L = 5, 8
    cache = {
        "input_ids": [[1] + [100 + i] * 4 + [wire.PAD_TOKEN_ID] * 3 for i in range(n)],
        "attention_mask": [[1] * 5 + [0] * 3 for _ in range(n)],
        "labels": [[1] + [100 + i] * 4 + [wire.PAD_TOKEN_ID] * 3 for i in range(n)],
        "images": [0, -1, 2, -1, 4], "audios": [-1, 1, -1, 3, -1], "videos": [-1, 1, -1, 3, -1],
    }
    p = os.path.join(tmp_path, "train.cache")
    pickle.dump(cache, open(p, "wb"), protocol=4)  # preprocess_data_supervised.py:451
    d = wire.load_cache(p)
    b = wire.collate(d, [0, 3])
    assert b["input_ids"].shape == (2, L) and b["input_ids"].dtype == torch.int64
    assert b["labels"][0].tolist() == [1, 100, 100, 100, 100, -100, -100, -100]  # pad -> IGNORE_INDEX
    assert b["images"].tolist() == [[0], [-1]] and b["videos"].tolist() == [[-1], [3]]
    inp = wire.make_inputs(b, None, torch.ones(2, 80, 3000), None)
    assert inp["images"].shape == (2, 3, 224, 224) and float(inp["images"].abs().sum()) == 0.0
    assert inp["videos"].shape == (2, 6, 3, 224, 224) and inp["audios"].dtype == torch.bfloat16
    assert inp["image_starts"].dtype == torch.int32 and inp["image_starts"].tolist() == [32000, 32000]
    assert inp["video_ends"].tolist() == [32005, 32005] and inp["labels"] is b["labels"]
    bad = dict(cache)
    bad.pop("videos")
    with pytest.raises(KeyError):
        wire.validate_cache(bad)
