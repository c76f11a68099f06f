"""CPU tier: the oracle (oracle/macaw_oracle.py) against the golden vectors minted from the unmodified reference."""
import os

import numpy as np
import pytest
import torch

from oracle import macaw_oracle as O
from tests import helpers as H
from tests.golden import gen


@pytest.fixture(scope="module")
def tiny_weights():
    spec, hp, shapes = H.load_shapes()
    return spec, hp, gen.make_weights(shapes, seed=0)


@pytest.mark.parametrize("name", ["all3", "image", "audio", "text"])
def test_oracle_matches_golden(tiny_weights, name):
    spec, hp, weights = tiny_weights
    case = H.load_case(name)
    o = O.forward(H.case_inputs(spec, case), weights, hp, dtype=torch.float32)
    g_emb, g_log = torch.from_numpy(case["embeds"]), torch.from_numpy(case["logits"])
    assert tuple(o["embeds"].shape) == tuple(g_emb.shape)
    assert H.rel_err(o["embeds"], g_emb) < 1e-5
    assert H.rel_err(o["logits"], g_log) < 1e-4
    # integer side is bit-exact
    assert torch.equal(o["attention_mask"], torch.from_numpy(case["attention_mask"]))
    if int(case["with_labels"]):
        assert torch.equal(o["labels"], torch.from_numpy(case["labels"]))
        assert abs(float(o["loss"]) - float(case["loss"])) < 1e-4 * abs(float(case["loss"]))
    else:
        assert o["labels"] is None and o["loss"] is None


def test_oracle_matches_golden_alt_family():
    """Second shape family (different widths, head counts, 3 frames, non-default Conv1d kernels / strides)."""
    import json

    with open(os.path.join(H.GOLDEN, "alt_shapes.json")) as f:
        d = json.load(f)
    spec, hp, shapes = d["spec"], d["hp"], {k: tuple(v) for k, v in d["shapes"].items()}
    weights = gen.make_weights(shapes, seed=0)
    z = np.load(os.path.join(H.GOLDEN, "alt_all3.npz"))
    inp = gen.make_inputs(spec, int(z["B"]), int(z["L"]), seed=int(z["seed"]), pad_tail=int(z["pad_tail"]))
    o = O.forward(inp, weights, hp, dtype=torch.float32)
    assert H.rel_err(o["embeds"], torch.from_numpy(z["embeds"])) < 1e-5
    assert H.rel_err(o["logits"], torch.from_numpy(z["logits"])) < 1e-4
    assert torch.equal(o["attention_mask"], torch.from_numpy(z["attention_mask"]))
    assert torch.equal(o["labels"], torch.from_numpy(z["labels"]))
    assert abs(float(o["loss"]) - float(z["loss"])) < 1e-4 * abs(float(z["loss"]))
    # prefix lengths follow (tokens - kernel) // stride + 1 with the non-default hyper-parameters
    n_img, n_aud, n_vid = (256 - 40) // 24 + 1, (1500 - 300) // 200 + 1, (3 * 256 - 50) // 45 + 1
    assert o["embeds"].shape[1] == 13 + (n_img + 2) + (n_aud + 2) + (n_vid + 2)


def test_layout_order_and_prefix_lengths(tiny_weights):
    """[BOS, <image> img </image>, <audio> aud </audio>, <video> vid </video>, text[1:]] (SURVEY.md §3.2)."""
    spec, hp, weights = tiny_weights
    case = H.load_case("all3")
    inp = H.case_inputs(spec, case)
    emb, mask, labels = O.prepare_inputs(inp, weights, hp)
    table = weights["llm.model.embed_tokens.weight"]
    n_img = (256 - 48) // 36 + 1
    n_aud = (1500 - 240) // 220 + 1
    n_vid = (spec["n_frames"] * 256 - 36) // 30 + 1
    pos = 1
    for name, n in (("image", n_img), ("audio", n_aud), ("video", n_vid)):
        assert torch.equal(emb[:, pos], table[inp[f"{name}_starts"].long()])
        assert torch.equal(emb[:, pos + n + 1], table[inp[f"{name}_ends"].long()])
        pos += n + 2
    assert emb.shape[1] == pos + inp["input_ids"].shape[1] - 1
    assert torch.equal(emb[:, pos:], table[inp["input_ids"][:, 1:]])
    assert torch.equal(mask[:, : pos - 1], torch.ones(2, pos - 1, dtype=torch.int64))
    assert torch.equal(labels[:, : pos - 1], torch.full((2, pos - 1), -100))


def test_video_pe_fixture():
    ref = np.load(os.path.join(H.GOLDEN, "video_pe_40x24.npz"))["pe"]
    assert np.array_equal(O.video_positional_encoding(40, 24).numpy(), ref)


def test_mha_restatement_vs_torch_module():
    """nn.MultiheadAttention (installed torch) vs the restatement, fp64 — the alignment shape in miniature."""
    torch.manual_seed(0)
    E, Hh, V, B, Lq = 32, 4, 50, 3, 5
    mha = torch.nn.MultiheadAttention(E, Hh, dropout=0.1, add_bias_kv=True, add_zero_attn=True).double().eval()
    with torch.no_grad():
        mha.in_proj_bias.normal_()
        mha.out_proj.bias.normal_()
    table = torch.randn(V, E, dtype=torch.float64)
    q = torch.randn(Lq, B, E, dtype=torch.float64)
    kv = table.unsqueeze(1).repeat(1, B, 1)
    ref = mha(q, kv, kv)[0]
    got = O.mha_forward(q, kv, kv, O._SD(dict(mha.state_dict()), torch.float64), Hh)
    assert float((ref - got).abs().max()) < 1e-12


def test_mha_dropout_restatement_vs_torch_module(monkeypatch):
    """train() mode: torch drops the SOFTMAX PROBABILITIES (all S + 2 keys, bias_k / zero keys included) before P.V
    (functional.py:6640-6645).  nn.MultiheadAttention with F.dropout replaced by an explicit mask vs the restatement with
    the same multipliers: outputs and gradients, fp64."""
    import torch.nn.functional as Fn

    torch.manual_seed(1)
    E, Hh, V, B, Lq, pd = 32, 4, 50, 3, 5, 0.1
    mha = torch.nn.MultiheadAttention(E, Hh, dropout=pd, add_bias_kv=True, add_zero_attn=True).double().train()
    with torch.no_grad():
        mha.in_proj_bias.normal_()
        mha.out_proj.bias.normal_()
    mult = (torch.rand(B * Hh, Lq, V + 2, dtype=torch.float64) >= pd).double() / (1 - pd)
    seen = []

    def fake_dropout(x, p=0.5, training=True, inplace=False):
        assert training and abs(p - pd) < 1e-12 and x.shape == mult.shape
        seen.append(1)
        return x * mult

    monkeypatch.setattr(Fn, "dropout", fake_dropout)
    table = torch.randn(V, E, dtype=torch.float64, requires_grad=True)
    q = torch.randn(Lq, B, E, dtype=torch.float64)
    kv = table.unsqueeze(1).repeat(1, B, 1)
    ref = mha(q, kv, kv)[0]
    assert len(seen) == 1
    w = torch.randn_like(ref)
    (ref * w).sum().backward()
    g_ref = {k: v.grad.clone() for k, v in mha.named_parameters()}
    gt_ref = table.grad.clone()
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in mha.state_dict().items()}
    t2 = table.detach().clone().requires_grad_(True)
    kv2 = t2.unsqueeze(1).expand(-1, B, -1)
    got = O.mha_forward(q, kv2, kv2, O._SD(leaves, torch.float64, keep_graph=True), Hh, dropout_mult=mult)
    assert float((ref - got).detach().abs().max()) < 1e-12
    (got * w).sum().backward()
    assert float((t2.grad - gt_ref).abs().max()) < 1e-10
    for k, g in g_ref.items():
        assert float((leaves[k].grad - g).abs().max()) < 1e-10, k


def test_philox_known_answers():
    """Philox4x32-10 restated in numpy (tests/helpers.py) against the published known-answer vectors of the Random123
    distribution (Salmon et al., SC'11) — the generator csrc/philox.cuh implements; the GPU tier compares the device mask
    with this restatement element by element."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in kat:
        got = H.philox4x32_10(np.array([ctr], dtype=np.uint32), key)
        assert tuple(int(x) for x in got[0]) == want
    m = H.dropout_multipliers(64, 37, 0.1, seed=(7 << 32) | 5, sid=3)
    assert m.shape == (64, 37) and set(np.unique(m)).issubset({0.0, np.float32(1 / 0.9)})
    assert abs(float((m != 0).mean()) - 0.9) < 0.03


def test_oracle_vs_live_reference(tiny_weights):
    """fp32 oracle vs the reference's own fp32 forward of the tiny model on an image+audio batch with labels
    (tests/golden/ref_image_audio.npz, recorded from the unmodified reference by make_golden.reference_outputs)."""
    spec, hp, weights = tiny_weights
    z = np.load(os.path.join(H.GOLDEN, "ref_image_audio.npz"))
    inp = gen.make_inputs(spec, int(z["B"]), int(z["L"]), seed=int(z["seed"]),
                          modalities=tuple(str(m) for m in z["modalities"]), pad_tail=int(z["pad_tail"]))
    o = O.forward(inp, weights, hp)
    assert tuple(o["logits"].shape) == z["logits"].shape
    assert H.rel_err(o["logits"], torch.from_numpy(z["logits"])) < 1e-4
    assert abs(float(o["loss"]) - float(z["loss"])) < 1e-4
