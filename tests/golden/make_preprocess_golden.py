"""Golden vectors for the device-side input pipeline (SURVEY.md §8f rank 3), minted from the THIRD-PARTY code the
reference's `get_self_inputs` calls (llm_trainer.py:151-158, 318-320, 338-345):

  images   torchvision Compose([Resize(224, BICUBIC), CenterCrop(224), ToTensor(), Normalize(CLIP mean/std)]) on PIL images
           (the reference's `_transform(224)`, verbatim)
  audio    whisper.pad_or_trim + whisper.log_mel_spectrogram.  The `whisper` package is absent from this image; its
           30-line implementation is restated here with torch.stft (whisper/audio.py: N_FFT 400, HOP 160, hann window,
           magnitudes = stft[..., :-1].abs()**2, filters @ magnitudes, clamp(1e-10).log10(), max(x, x.max() - 8), (x+4)/4)
           using the mel filter bank of transformers' WhisperFeatureExtractor (an independent implementation of the
           librosa filters whisper ships as assets/mel_filters.npz).

Inputs are synthesised deterministically (tests/golden/gen.py: synth_image / synth_audio), so only the OUTPUTS are stored.
Usage:  python tests/golden/make_preprocess_golden.py
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from tests.golden import gen  # noqa: E402


def reference_transform(n_px=224):
    from PIL import Image
    from torchvision.transforms import CenterCrop, Compose, Normalize, Resize, ToTensor
    from torchvision.transforms import InterpolationMode

    return Compose([
        Resize(n_px, interpolation=InterpolationMode.BICUBIC),
        CenterCrop(n_px),
        lambda im: im.convert("RGB"),
        ToTensor(),
        Normalize((0.48145466, 0.4578275, 0.40821073), (0.26862954, 0.26130258, 0.27577711)),
    ]), Image


def whisper_log_mel(audio: torch.Tensor) -> torch.Tensor:
    from transformers import WhisperFeatureExtractor

    n = 480000
    audio = audio[:n] if audio.shape[0] > n else torch.nn.functional.pad(audio, (0, n - audio.shape[0]))  # pad_or_trim
    window = torch.hann_window(400)
    stft = torch.stft(audio, 400, 160, window=window, return_complex=True)
    magnitudes = stft[..., :-1].abs() ** 2
    filters = torch.from_numpy(WhisperFeatureExtractor().mel_filters.T.astype(np.float32))
    mel_spec = filters @ magnitudes
    log_spec = torch.clamp(mel_spec, min=1e-10).log10()
    log_spec = torch.maximum(log_spec, log_spec.max() - 8.0)
    return (log_spec + 4.0) / 4.0


def mel_frames(i: int) -> np.ndarray:
    """Frames of clip i stored in the fixture: every frame of the padded clip (its silent tail compresses to nothing), a
    seeded sample of 400 of the trimmed clip's 3000 frames (audio everywhere: stored whole it would be ~0.8 MB)."""
    if i == 0:
        return np.arange(3000)
    return np.sort(np.random.default_rng(i).choice(3000, 400, replace=False))


def main():
    tf, Image = reference_transform()
    out = {}
    for i, (h, w) in enumerate(gen.PREPROCESS_IMAGE_SIZES):
        img = gen.synth_image(h, w, seed=i)
        pil = Image.fromarray(img)
        t = tf(pil)
        # the 8-bit resized + cropped image (before ToTensor), via the same two torchvision ops
        from torchvision.transforms import CenterCrop, Resize
        from torchvision.transforms import InterpolationMode

        u8 = np.asarray(CenterCrop(224)(Resize(224, interpolation=InterpolationMode.BICUBIC)(pil)))
        out[f"img{i}_u8"] = u8
        if i == 0:
            out["img0_f32"] = t.numpy()
        assert np.allclose(t.numpy(), ((u8.astype(np.float32) / 255.0).transpose(2, 0, 1)
                                       - np.array([0.48145466, 0.4578275, 0.40821073], np.float32)[:, None, None])
                           / np.array([0.26862954, 0.26130258, 0.27577711], np.float32)[:, None, None], atol=1e-6)
    for i, secs in enumerate(gen.PREPROCESS_AUDIO_SECONDS):
        a = torch.from_numpy(gen.synth_audio(secs, seed=i))
        lm = whisper_log_mel(a)
        assert lm.shape == (80, 3000)
        out[f"mel{i}_cols"] = mel_frames(i)
        out[f"mel{i}"] = lm.numpy().astype(np.float32)[:, out[f"mel{i}_cols"]]
    np.savez_compressed(os.path.join(HERE, "preprocess.npz"), **out)
    print({k: v.shape for k, v in out.items()}, os.path.getsize(os.path.join(HERE, "preprocess.npz")) // 1024, "KiB")


if __name__ == "__main__":
    main()
