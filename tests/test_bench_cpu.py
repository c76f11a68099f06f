"""CPU tier: bench.py plumbing that does not need a GPU — the reference arm's JSON contract (on the tiny stand-in model),
synthetic input shapes, usable-core detection."""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract_small():
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--small", "--seq-len", "16",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "tokens/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and d["gpu_launches"] == 0
    # the arm drives the unmodified reference when oracle/_ref is staged (build container, GPU box), else the port
    from oracle import ref_runner

    assert d["cpu_baseline"]["kind"] == ("reference" if ref_runner.available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_b200_arm_refuses_to_run_without_cuda():
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--small", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_dump_outputs_is_float32_bounded_and_repeatable(tmp_path):
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench

    B, T, V = 3, 50, 1000
    logits = torch.randn(B, T, V, generator=torch.Generator().manual_seed(3)).to(torch.float16)
    for d in ("a", "b"):
        bench.dump_outputs(logits, str(tmp_path / d))
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["logits_last.npy", "logits_sample.npy"]
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "logits_last.npy"), logits[:, -1].float().numpy())
    # every row fits the budget here, so the sorted sample is the whole flattened output in order
    assert np.array_equal(np.load(tmp_path / "a" / "logits_sample.npy"), logits.float().reshape(B * T, V).numpy())
    # at the benchmark's shape the two files stay within 64 MiB
    rows = min(32 * 528, bench.DUMP_SAMPLE_BYTES // (4 * 32000)) + min(32, bench.DUMP_LAST_BYTES // (4 * 32000))
    assert rows * 32000 * 4 <= 64 * 2 ** 20


def test_synth_inputs_and_cores():
    sys.path.insert(0, ROOT)
    import bench

    d = bench.synth_inputs(3, 20, 32000, 224, 3000, seed=1, pin=False)
    assert d["images"].shape == (3, 3, 224, 224) and d["images"].dtype == torch.bfloat16
    assert d["audios"].shape == (3, 80, 3000) and d["videos"] is None
    assert d["input_ids"].shape == (3, 20) and int(d["input_ids"][:, 0].max()) == 1
    assert len({int(d[f"{m}_{s}"][0]) for m in ("image", "audio", "video") for s in ("starts", "ends")}) == 6
    assert 1 <= bench.usable_cores() <= (os.cpu_count() or 1)
    assert 1 <= bench.cpu_threads() <= bench.usable_cores()
    (clip, whisper, llama), hyper = bench.real_configs()
    assert (llama.hidden_size, llama.num_hidden_layers, llama.vocab_size) == (4096, 32, 32000)
    assert (clip.vision_config.hidden_size, clip.projection_dim, whisper.d_model) == (1024, 768, 512)
