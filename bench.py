#!/usr/bin/env python
"""Benchmark of record: multimodal prefill tokens/sec of the MM_LLMs forward (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  # the UNMODIFIED reference modeling.py on the host CPUs (oracle/_ref)

Workload (config.workload): BASELINE config 4 — image + audio + text, CLIP ViT-L/14-224 + Whisper-base encoder +
alignment (32000 x 4096 table, 16 heads) + LLaMA-7B, global batch 32, L = 512 text tokens -> T = 528 positions,
random-init weights, synthetic inputs, labels=None, logits for all positions.  A "step" is one forward over the
global batch; with N ranks the global batch is split by sample (strong scaling, no collective on the data path).

One JSON line is printed by rank 0 (see the field list in DESIGN.md §Measurement).

  python bench.py ... --dump-outputs DIR   # also write what the last timed step computed as DIR/<name>.npy (see dump_outputs)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from untouched (it may be read-only)

import torch  # noqa: E402

METRIC = "multimodal prefill tokens/sec (img+audio+text->LLaMA)"
DEFAULT_DTYPE = "fp16"
UNIT = "tokens/s"


# ---------------------------------------------------------------------------------------------------- configs
def real_configs(small: bool = False):
    from transformers import CLIPConfig, LlamaConfig, WhisperConfig

    if small:  # CI-sized stand-in used by tests (same code path, kernel-compatible widths)
        from tests.golden import gen

        return gen.build_configs(gen.TINY), dict(n_frames=gen.TINY["n_frames"], attention_heads=gen.TINY["attention_heads"])
    clip = CLIPConfig(  # openai/clip-vit-large-patch14
        text_config=dict(hidden_size=768, intermediate_size=3072, num_hidden_layers=12, num_attention_heads=12,
                         projection_dim=768),
        vision_config=dict(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24, num_attention_heads=16,
                           image_size=224, patch_size=14, projection_dim=768, hidden_act="quick_gelu"),
        projection_dim=768)
    whisper = WhisperConfig(  # openai/whisper-base
        d_model=512, encoder_layers=6, encoder_attention_heads=8, encoder_ffn_dim=2048, decoder_layers=6,
        decoder_attention_heads=8, decoder_ffn_dim=2048, num_mel_bins=80, max_source_positions=1500, vocab_size=51865)
    llama = LlamaConfig(hidden_size=4096, intermediate_size=11008, num_hidden_layers=32, num_attention_heads=32,
                        vocab_size=32000, rms_norm_eps=1e-6, max_position_embeddings=2048, pad_token_id=0,
                        bos_token_id=1, eos_token_id=2)
    return (clip, whisper, llama), dict(n_frames=6, attention_heads=8)


def synth_inputs(B, L, V, img, mel_T, seed, dtype=torch.bfloat16, pin=True, video_frames=0):
    """Seeded synthetic host inputs of the reference's `inputs` dict (SURVEY.md §8d).  video_frames > 0: BASELINE config 5
    (a video of that many frames + audio, no image)."""
    g = torch.Generator().manual_seed(seed)
    d = dict(videos=None)
    if video_frames:
        d["images"] = None
        d["videos"] = torch.randn(B, video_frames, 3, img, img, generator=g).to(dtype)
    else:
        d["images"] = torch.randn(B, 3, img, img, generator=g).to(dtype)
    d["audios"] = torch.randn(B, 80, mel_T, generator=g).to(dtype)
    ids = torch.randint(3, V - 6, (B, L), generator=g)
    ids[:, 0] = 1
    d["input_ids"] = ids
    d["attention_mask"] = torch.ones(B, L, dtype=torch.int64)
    sp = [V - 6 + i for i in range(6)]
    for i, name in enumerate(("image", "audio", "video")):
        d[f"{name}_starts"] = torch.full((B,), sp[2 * i], dtype=torch.int32)
        d[f"{name}_ends"] = torch.full((B,), sp[2 * i + 1], dtype=torch.int32)
    if pin and torch.cuda.is_available():
        d = {k: (v.pin_memory() if isinstance(v, torch.Tensor) else v) for k, v in d.items()}
    return d


# ---------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": (statistics.median(sm) if sm else None), "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------- reference arm
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


def usable_cores() -> int:
    """Host threads this process may actually use: min(affinity, cgroup v2 cpu.max quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def physical_cores_one_socket() -> int:
    """Physical cores of socket 0 (hyper-threads and the second socket make the fp32 CPU arm SLOWER: round 1 measured
    56.6 tok/s on a 96-thread box vs 66.4 on a 16-thread one)."""
    try:
        cores, phys, core = set(), None, None
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("physical id"):
                phys = ln.split(":")[1].strip()
            elif ln.startswith("core id"):
                core = ln.split(":")[1].strip()
            elif not ln.strip():
                if phys == "0" and core is not None:
                    cores.add(core)
                phys = core = None
        return len(cores) or (os.cpu_count() or 1)
    except Exception:
        return os.cpu_count() or 1


def cpu_threads() -> int:
    return max(1, min(usable_cores(), physical_cores_one_socket()))


def cpu_reference_sample(cfgs, hyper, L, steps, warmup, seed=1234, state_dict=None, inputs=None):
    """Time the reference's own CPU implementation of the path on a bounded sample of the workload: ONE sample (B=1)
    image+audio+text, full model depth, fp32.

    kind "reference": the UNMODIFIED /root/reference/modeling.py staged under oracle/_ref (oracle/make_ref.py) —
    `MM_LLMs.forward` through its stock code path (per-sample K/V projection of the whole table included).
    kind "port": oracle/macaw_oracle.py, only when oracle/_ref is absent.
    The reference is linear in B (every term is per-sample, SURVEY.md §8d), so tokens/s of one sample is its tokens/s at
    any batch.  Returns timing + the sample's outputs (for the bench line's `parity` block)."""
    import copy

    from oracle import ref_runner as R

    clip, whisper, llama = cfgs
    cores = cpu_threads()
    torch.set_num_threads(cores)
    V = llama.vocab_size
    if inputs is None:
        inputs = synth_inputs(1, L, V, clip.vision_config.image_size, 2 * whisper.max_source_positions, seed,
                              torch.float32, pin=False)
    inputs = {k: (v.float() if isinstance(v, torch.Tensor) and v.is_floating_point() else v) for k, v in inputs.items()}
    if R.available():
        kind = "reference"
        model = R.build_model(copy.deepcopy(clip), copy.deepcopy(whisper), copy.deepcopy(llama), dict(hyper),
                              state_dict=state_dict)

        def run():
            with torch.no_grad():
                emb, _, _ = model.prepare_inputs_for_generation(inputs)
                out = model(inputs)
            return out.logits, emb
        what = "oracle/_ref/modeling.py (unmodified reference, MM_LLMs.forward)"
    else:
        kind = "port"
        from macaw_llm_b200.modeling import MM_LLMs, MM_LLMs_Config
        from oracle import macaw_oracle as O

        cfg = MM_LLMs_Config(clip_config=clip, whisper_config=whisper, llm_config=llama, **hyper)
        hp = O.hp_from_config(cfg)
        if state_dict is None:
            with torch.device("meta"):
                meta = MM_LLMs(cfg)
            state_dict = R.random_state_dict(meta)
        sd = {k: v.detach().to("cpu", torch.float32) for k, v in state_dict.items() if v.is_floating_point()}

        def run():
            o = O.forward(inputs, sd, hp, dtype=torch.float32)
            return o["logits"], o["embeds"]
        what = "oracle/macaw_oracle.py (port; oracle/_ref absent)"
    times, T, out = [], None, None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = run()
        dt = time.perf_counter() - t0
        T = out[0].shape[1]
        if i >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    return dict(value=T / sec, unit=UNIT, cores=cores, kind=kind, steps_timed=len(times), sec_per_step=sec,
                logits=out[0], embeds=out[1],
                sample=f"1 sample (B=1) image+audio+text, L={L} -> T={T}, full depth, fp32, {what}; "
                       f"reference cost is linear in B; {cores} threads (physical cores of one socket, capped by the cgroup)")


# ---------------------------------------------------------------------------------------------------- secondary modes
def run_train(args, cfgs, hyper, rank, local_rank, world):
    """Secondary line: one TRAINING step (SURVEY.md §8f rank 1) = zero_grad + forward + backward + gradient all-reduce +
    fused AdamW on the cfg4 shape at the reference's micro-batch (train.sh: 4 samples per GPU, fp32 master weights).
    Weak scaling: per-GPU work is fixed, the data-parallel group grows."""
    import torch.distributed as dist

    from macaw_llm_b200 import ops
    from macaw_llm_b200.modeling import MM_LLMs, MM_LLMs_Config
    from macaw_llm_b200.training import FusedAdamW, freeze_like_reference, trainable_parameters

    clip, whisper, llama = cfgs
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L, V, Bl = args.seq_len, llama.vocab_size, args.micro_batch
    cfg = MM_LLMs_Config(clip_config=clip, whisper_config=whisper, llm_config=llama, **hyper)
    model = MM_LLMs.build_random(cfg, device=dev, dtype=torch.bfloat16, seed=0)
    freeze_like_reference(model)
    host = synth_inputs(Bl, L, V, clip.vision_config.image_size, 2 * whisper.max_source_positions, 1234 + rank)
    host["labels"] = host["input_ids"].clone()
    inp = {k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in host.items()}
    params = [p for _, p in trainable_parameters(model)]
    opt = FusedAdamW(params, lr=2e-5, weight_decay=0.0)
    model.train()
    model.train_step.set_world(world, overlap=True)
    own_nccl = False
    if world > 1:
        from macaw_llm_b200 import dist as D

        own_nccl = D.init_nccl(dev)  # the kernel library's own communicator (mm_nccl_allreduce)

    def step():
        opt.zero_grad()
        out = model(inp)
        out.loss.backward()
        model.train_step.llama.finish_allreduce()
        opt.step()
        return out.loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    losses = []
    for _ in range(max(args.warmup, 3)):
        losses.append(float(step()))
    barrier()
    ops.launch_count_reset()
    step()
    launches_per_step = ops.launch_count()
    # ---- the whole step (forward, backward, optimizer: ~5000 launches issued from Python) replayed from ONE CUDA graph.
    #      Every step-dependent scalar lives on the device (AdamW step counter, upstream loss gradient), buffers are static.
    # (data-parallel group: the per-layer bucket all-reduces are captured too — NCCL calls on a side stream forked from the
    #  capturing stream — when they go through the library's own communicator; --ddp-graph 0 keeps the host launches)
    use_graph = (world == 1 or (own_nccl and args.ddp_graph)) and not args.no_graphs
    if use_graph:
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        static = {}
        with torch.cuda.graph(graph, capture_error_mode="thread_local"):
            static["loss"] = step()
        eager_step = step

        def step():  # noqa: F811
            graph.replay()
            return static["loss"]

        for _ in range(2):
            losses.append(float(step()))
    barrier()
    if args.kernel_table and rank == 0:  # attribution only (CUPTI trace of one step); printed to stderr, never a bench value
        import collections

        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.synchronize()
        acc = collections.defaultdict(lambda: [0, 0.0])
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                acc[ev.name][0] += 1
                acc[ev.name][1] += ev.device_time
        tot = sum(v[1] for v in acc.values())
        print(f"[train kernel table] kernel time {tot / 1e3:.2f} ms per step", file=sys.stderr)
        for name, (cnt, us) in sorted(acc.items(), key=lambda kv: -kv[1][1])[:28]:
            print(f"{name[:80]:80s} {cnt:6d} {us / cnt:9.1f} us {us / 1e3:8.3f} ms {us / tot:6.1%}", file=sys.stderr)
    ops.launch_count_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step()
    e1.record()
    barrier()
    launches = launches_per_step * args.steps
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / args.steps
    losses.append(float(loss))
    if rank == 0:
        T = L + 16
        n_train = sum(p.numel() for p in params)
        # 6 FLOP per trainable parameter per token (fwd 2 + bwd 4) + the frozen encoders' / alignment forward
        tf = (6.0 * n_train * Bl * T + Bl * (162.4e9 + 87.4e9)) / 1e12
        print(json.dumps({
            "mode": "train", "metric": "multimodal training tokens/sec (img+audio+text->LLaMA, fwd+bwd+all-reduce+AdamW)",
            "value": world * Bl * T / (ms / 1e3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": f"cfg4 shape, micro-batch {Bl}/GPU (train.sh), L={L} -> T={T}, LLaMA-7B + CLIP-L + Whisper-base",
                       "trainable_params": n_train, "optimizer": "fused AdamW, fp32 master + moments",
                       "submission": "cuda_graph_replay of the whole step" if use_graph else "host_launches",
                       "grad_sync": ("flat bf16 buffer, one NCCL all-reduce per decoder layer on a side stream, overlapped with backward ("
                                     + ("mm_nccl_allreduce" if own_nccl else "torch.distributed") + ")") if world > 1 else "none (1 rank)",
                       "differentiable_set": "llm.* + the alignment modules of every modality (incl. the table as the alignment attention's keys/values); video_long_self_attention; encoders frozen; MHA attention dropout p=0.1 live (Philox mask regenerated in backward)"},
            "approx_tflops": tf / (ms / 1e3), "gpu_launches": launches, "loss_first_last": [losses[0], losses[-1]],
            "mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_decode(args, cfgs, hyper, rank, local_rank, world):
    """Secondary line: greedy decoding behind inputs['inference'] = True (SURVEY.md §8f rank 2): image+text, B=8 per GPU,
    prefill + 64 new tokens; reports ms per decode step against the 13.5 GB weight-streaming floor."""
    from macaw_llm_b200.modeling import MM_LLMs, MM_LLMs_Config

    clip, whisper, llama = cfgs
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    V, B, L, n_new = llama.vocab_size, 8, 256, 64
    cfg = MM_LLMs_Config(clip_config=clip, whisper_config=whisper, llm_config=llama, **hyper)
    model = MM_LLMs.build_random(cfg, device=dev, dtype=torch.bfloat16, seed=0)
    host = synth_inputs(B, L, V, clip.vision_config.image_size, 2 * whisper.max_source_positions, 1234 + rank)
    inp = {k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in host.items()}
    inp["audios"] = None
    inp["inference"] = True

    def run(n):
        d = dict(inp, max_new_tokens=n)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        toks = model.engine.generate(d, max_new_tokens=n, eos_token_id=-1)  # eos -1: never stop early (timing)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), toks

    for _ in range(max(1, min(args.warmup, 2))):
        run(n_new)
    t1 = min(run(1)[0] for _ in range(2))           # prefill + first token
    tn = min(run(n_new)[0] for _ in range(args.steps))
    ms_step = (tn - t1) / (n_new - 1)
    hbm, _, _, src = load_peaks()
    wbytes = sum(p.numel() * p.element_size() for n_, p in model.named_parameters() if n_.startswith("llm.model.layers") or n_ == "llm.lm_head.weight")
    floor_ms = wbytes / (hbm * 1e9) * 1e3
    if rank == 0:
        print(json.dumps({
            "mode": "decode", "metric": "greedy decode tokens/sec (image+text prefix, KV cache)", "value": B / (ms_step / 1e3),
            "unit": UNIT, "n_gpus": 1, "higher_is_better": True, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"image+text, B={B}, L={L} -> T={L + 8}, {n_new} new tokens, LLaMA-7B", "submission": "cuda_graph_replay"},
            "prefill_ms": t1, "ms_per_decode_step": ms_step,
            "roofline": {"bound": "hbm", "achieved": wbytes / (ms_step / 1e3) / 1e9, "peak": hbm, "unit": "GB/s",
                         "frac": floor_ms / ms_step, "peak_source": src, "algorithmic_bytes_per_step": wbytes}}), flush=True)


# ---------------------------------------------------------------------------------------------------- output dump
DUMP_SAMPLE_BYTES = 48 * 2 ** 20  # logits_sample.npy
DUMP_LAST_BYTES = 16 * 2 ** 20    # logits_last.npy: 64 MiB in all


def dump_outputs(logits, out_dir: str) -> None:
    """Write the (B, T, V) logits of one prefill step as float32 .npy files under `out_dir`:
      logits_last.npy    (b, V)  next-token logits of the first b = min(B, 16 MiB / (4 V)) samples (all 32 at cfg4);
      logits_sample.npy  (n, V)  n = min(B T, 48 MiB / (4 V)) rows of the (B T, V) logits, flattened batch-major, at the
                                 positions of a seed-0 torch.randperm, sorted (the same rows for the same arguments)."""
    import numpy as np

    B, T, V = logits.shape
    flat = logits.reshape(B * T, V)
    n = min(B * T, DUMP_SAMPLE_BYTES // (4 * V))
    rows = torch.randperm(B * T, generator=torch.Generator().manual_seed(0))[:n].sort().values
    arrays = {"logits_last": logits[: min(B, DUMP_LAST_BYTES // (4 * V)), -1, :],
              "logits_sample": flat[rows.to(flat.device)]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.float().cpu().numpy())


# ---------------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--global-batch", type=int, default=32)
    ap.add_argument("--seq-len", type=int, default=512)
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--small", action="store_true", help="tiny stand-in model (tests only; the result is not a bench value)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graphs", action="store_true", help="launch every kernel from the host instead of replaying a CUDA graph")
    ap.add_argument("--mode", default="prefill", choices=["prefill", "train", "decode"],
                    help="prefill = the benchmark of record; train / decode = secondary lines (SURVEY.md §8f ranks 1, 2)")
    ap.add_argument("--ddp-graph", type=int, default=1, help="--mode train, N > 1: capture the step incl. the NCCL buckets in a CUDA graph")
    ap.add_argument("--kernel-table", action="store_true", help="--mode train: per-kernel time table of one step on stderr")
    ap.add_argument("--micro-batch", type=int, default=4, help="--mode train: samples per GPU per step (train.sh: 4)")
    ap.add_argument("--config", default="cfg4", choices=["cfg4", "cfg5"],
                    help="cfg4 = the benchmark of record (image+audio+text, global batch 32); cfg5 = secondary line: video "
                         "(16 CLIP frames -> 4096 tokens, head_dim-96 self-attention) + audio + text, global batch 16")
    ap.add_argument("--dtype", default=DEFAULT_DTYPE, choices=["bf16", "fp16"],
                    help="storage / tensor-core operand format of the prefill arm (fp32 accumulation either way); the "
                         "reference itself runs fp16 (train.sh --fp16 True)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="prefill: after the timed steps, write what the last one computed (rank 0's logits, float32, a "
                         "fixed seeded sample) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.mode != "prefill"):
        ap.error("--dump-outputs applies to the prefill benchmark of the b200 implementation")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfgs, hyper = real_configs(args.small)
    clip, whisper, llama = cfgs
    vframes = 0
    if args.config == "cfg5":
        vframes = 16
        hyper = dict(hyper, n_frames=16)
        if args.global_batch == 32:
            args.global_batch = 16
    L, V = args.seq_len, llama.vocab_size
    workload = (f"cfg4 image+audio+text: CLIP ViT-L/14-224 + Whisper-base + alignment(V={V},E={llama.hidden_size},"
                f"{hyper['attention_heads'] * 2} heads) + LLaMA-7B, global_batch={args.global_batch}, L={L}")
    if args.config == "cfg5":
        workload = (f"cfg5 video(16 frames)+audio+text: CLIP ViT-L/14-224 x16 frames + video-long self-attention (N=4096, 8x96) + "
                    f"Whisper-base + alignment(V={V},E={llama.hidden_size}) + LLaMA-7B, global_batch={args.global_batch}, L={L}")
    if args.small:
        workload = "SMALL stand-in (tests only) " + workload

    # ------------------------------------------------------------------ reference arm: host CPUs only
    if args.impl == "reference":
        if rank != 0:
            return
        warm = min(args.warmup, 1)
        cb = cpu_reference_sample(cfgs, hyper, L, args.steps, warm)
        line = {
            "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": cb["steps_timed"], "warmup": warm, "ms_per_step": cb["sec_per_step"] * 1e3,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "sample": cb["sample"]},
            "cpu_baseline": {"value": cb["value"], "unit": UNIT, "cores": cb["cores"], "kind": cb["kind"],
                             "sample": cb["sample"]},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line), flush=True)
        return

    # ------------------------------------------------------------------ B200 arm
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    if args.mode == "train":
        return run_train(args, cfgs, hyper, rank, local_rank, world)
    if args.mode == "decode":
        return run_decode(args, cfgs, hyper, rank, local_rank, world)
    import torch.distributed as dist

    from macaw_llm_b200 import ops
    from macaw_llm_b200.modeling import MM_LLMs, MM_LLMs_Config

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.scaling == "strong":
        assert args.global_batch % world == 0, "global batch must divide by the number of ranks"
        B_local, B_global = args.global_batch // world, args.global_batch
    else:
        B_local, B_global = args.global_batch, args.global_batch * world

    cfg = MM_LLMs_Config(clip_config=clip, whisper_config=whisper, llm_config=llama, **hyper)
    tdt = torch.float16 if args.dtype == "fp16" else torch.bfloat16
    model = MM_LLMs.build_random(cfg, device=dev, dtype=tdt, seed=0)  # same seed -> identical replicas
    if args.scaling == "strong":
        # ONE seeded global batch, sharded by sample with the product's own helper: every N runs the same 32 samples
        from macaw_llm_b200 import dist as D

        glob = synth_inputs(B_global, L, V, clip.vision_config.image_size, 2 * whisper.max_source_positions, 1234, dtype=tdt,
                            pin=False, video_frames=vframes)
        host = D.shard_inputs(glob, rank, world)
        host = {k: (v.contiguous().pin_memory() if isinstance(v, torch.Tensor) else v) for k, v in host.items()}
        del glob
    else:
        host = synth_inputs(B_local, L, V, clip.vision_config.image_size, 2 * whisper.max_source_positions, 1234 + rank, dtype=tdt,
                            video_frames=vframes)
    dev_in = {k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in host.items()}

    def step_resident():
        return model(dev_in).logits

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- roofline pass (eager launches, per-launch CUDA events around every GEMM; also builds the weight caches).
    #      The kernels and their launch parameters are exactly those of the timed region below; only the way they are
    #      submitted differs (host launches here, CUDA-graph replay there), so durations are representative.
    for _ in range(2):
        logits = step_resident()
    T = logits.shape[1]
    barrier()
    overlap = model.engine.overlap_encoders
    model.engine.overlap_encoders = False  # per-launch events need the launches serialised on one stream
    ops.PROFILE = []
    ops.launch_count_reset()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(args.steps):
        step_resident()
    p1.record()
    barrier()
    launches = ops.launch_count()
    prof_ms = p0.elapsed_time(p1)
    prof, ops.PROFILE = ops.PROFILE, None
    model.engine.overlap_encoders = overlap

    use_graphs = not args.no_graphs
    if use_graphs:
        model.engine.enable_cuda_graphs(True)
    for _ in range(max(args.warmup, 3)):  # warm-up of the timed path (captures the graph on the first call)
        logits = step_resident()
    barrier()

    # ---- timed region 1: inputs resident in HBM ("value")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        logits = step_resident()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = B_global * T * args.steps / (ms_max / 1e3)
    if args.dump_outputs and rank == 0:  # here: the next region overwrites the CUDA graph's output buffers
        dump_outputs(logits, args.dump_outputs)

    # ---- timed region 2: end to end through the public call with HOST (pinned) buffers: H2D of every input + forward
    #      + D2H of the step's result (next-token logits of every sample)
    out_host = torch.empty((B_local, V), dtype=tdt).pin_memory()

    def step_e2e():
        d = {k: (v.to(dev, non_blocking=True) if isinstance(v, torch.Tensor) else v) for k, v in host.items()}
        lg = model(d).logits
        out_host.copy_(lg[:, -1, :], non_blocking=True)

    step_e2e()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        step_e2e()
    f1.record()
    barrier()
    t2 = torch.tensor([f0.elapsed_time(f1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = B_global * T * args.steps / (float(t2.item()) / 1e3)
    h2d = sum(v.numel() * v.element_size() for v in host.values() if isinstance(v, torch.Tensor)) * world
    d2h = out_host.numel() * out_host.element_size() * world

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- live roofline of the dominant kernel (the tcgen05 GEMM): algorithmic FLOPs / CUDA-event time, all launches
    hbm_peak, tf_burst, tf_sust, peak_src = load_peaks()
    by_tag = {}
    for tag, flops, a, b in prof:
        d = by_tag.setdefault(tag, [0.0, 0.0, 0])
        d[0] += flops
        d[1] += a.elapsed_time(b) * 1e-3
        d[2] += 1
    tot_f = sum(v[0] for v in by_tag.values())
    tot_s = sum(v[1] for v in by_tag.values())
    achieved = tot_f / tot_s / 1e12 if tot_s > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("gemm_dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {
        "kernel": "mm::gemm_bf16_kernel (tcgen05 + TMA), all launches of the step",
        "bound": "tensor", "achieved": achieved, "peak": tf_sust, "unit": "TFLOP/s", "frac": achieved / tf_sust,
        "peak_source": f"{peak_src} bf16_tflops_sustained (kernel timed inside a long step)", "traffic": traffic,
        "share_of_step": tot_s / (prof_ms / 1e3),
        "by_section": {k: {"tflops": v[0] / v[1] / 1e12 if v[1] > 0 else 0.0, "ms_per_step": v[1] * 1e3 / args.steps,
                           "launches_per_step": v[2] / args.steps} for k, v in sorted(by_tag.items())},
    }

    # ---- CPU arm on the SAME weights and the same sample 0 as the GPU arm: a timing baseline AND a full-depth parity
    #      check of the benchmarked configuration (the GPU side re-runs sample 0 alone, eager launches)
    cpu = parity = None
    if not args.no_cpu_baseline and world == 1 and args.config == "cfg4":
        one = {k: (v[:1].clone() if isinstance(v, torch.Tensor) else v) for k, v in host.items()}
        model.engine.enable_cuda_graphs(False)
        with torch.no_grad():
            g_emb, _, _ = model.prepare_inputs_for_generation({k: (v.to(dev) if isinstance(v, torch.Tensor) else v)
                                                               for k, v in one.items()})
            g_log = model({k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in one.items()}).logits
        g_emb, g_log = g_emb.float().cpu(), g_log.float().cpu()
        cb = cpu_reference_sample(cfgs, hyper, L, steps=1, warmup=0, state_dict=model.state_dict(), inputs=one)
        cpu = {"value": cb["value"], "unit": UNIT, "cores": cb["cores"], "kind": cb["kind"], "sample": cb["sample"]}
        r_log, r_emb = cb["logits"].float(), cb["embeds"].float()
        n_prefix = r_emb.shape[1] - L
        # aligned rows only: [BOS, <image>, img x Lq, </image>, <audio>, aud x Lq, </audio>, text...] — the start / end rows
        # are exact table gathers and (with random-init scales) 100x larger than the aligned rows, so they are left out
        lens = model.engine.last_lens
        rows, off = [], 1
        for name in ("image", "audio", "video"):
            if name in lens:
                rows += list(range(off + 1, off + 1 + lens[name]))
                off += lens[name] + 2
        rows = torch.tensor(rows, dtype=torch.long)

        def rel(a, b):
            return float((a - b).norm() / (b.norm() + 1e-30))

        parity = {
            "vs": cb["kind"] + f" fp32 on the GPU arm's {args.dtype} weights, rank-0 sample 0, full depth",
            "embeds_rel": rel(g_emb, r_emb), "prefix_rel": rel(g_emb[:, rows], r_emb[:, rows]),
            "prefix_rows": "the aligned rows of every modality block (start / end token rows are exact gathers)",
            "logits_rel": rel(g_log, r_log),
            "argmax_agree": float((g_log.argmax(-1) == r_log.argmax(-1)).float().mean()),
            "layout_exact": bool(torch.equal(g_emb[:, 1 + n_prefix:], r_emb[:, 1 + n_prefix:].to(tdt).float())),
            "metric": "norm-wise relative error ||gpu - ref|| / ||ref||",
        }

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": workload, "global_batch": B_global, "per_gpu_batch": B_local, "seq_len": L, "T": T,
                   "parallelism": f"dp{world}", "submission": ("cuda_graph_replay" if use_graphs else "host_launches"),
                   "l2": "per-step working set (16 GB of weights) >> 126 MB L2; no flush needed"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "result": f"next-token logits (B, V) {args.dtype} read back to pinned host memory (an inference consumer's result)"},
        "gpu_launches": launches,  # kernels of libmacaw_b200.so per timed region (counted on the eager pass; the graph replays the same nodes)
        "roofline": roofline,
        "cpu_baseline": cpu,
        "parity": parity,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
