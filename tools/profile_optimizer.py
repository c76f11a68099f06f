"""Cost of the training recipe's update on the real trainable set (cfg4: LLaMA-7B + the alignment modules, 7.06e9 bf16
gradients), all timed with CUDA events in one process:

  norm     the mm_grad_norm pass over every gradient, against a device-to-device copy of the same 14.1 GB (alternating);
  step     FusedAdamW.step() as before (host-float lr, no clipping) against the recipe step (clipping at 1.0 + warmup /
           cosine lr + the non-finite check), each replayed from its own CUDA graph, alternating;
  ga3      one optimizer step of train.sh's shape: 3 micro-batches of 4 (L = 512, image + audio + text), no_sync on the
           first two, then the recipe step; the whole step replayed from one CUDA graph.  With >= 2 GPUs visible the
           data-parallel variant is not run by this script (launch one process per GPU for that).

Usage: python tools/profile_optimizer.py [--out FILE] [--reps 10]"""
import argparse
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def card() -> str:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"{torch.cuda.get_device_name(0)} | nvidia-smi: {q}"


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def alternate(fns, reps, rounds=5):
    """ms per call of each fn, interleaved over `rounds` (min and median over rounds)."""
    res = {k: [] for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            res[k].append(timed(f, reps))
    return {k: (min(v), sorted(v)[len(v) // 2]) for k, v in res.items()}


def graph_of(fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, capture_error_mode="thread_local"):
        fn()
    return g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--skip-ga3", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("profile_optimizer: needs a GPU")
    import bench
    from macaw_llm_b200 import ops
    from macaw_llm_b200.modeling import MM_LLMs, MM_LLMs_Config
    from macaw_llm_b200.training import (FusedAdamW, GradBuffer, LRSchedule, freeze_like_reference, trainable_parameters,
                                         warmup_steps)

    lines = []

    def out(s):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out(f"card: {card()}")
    (clip, whisper, llama), hyper = bench.real_configs(False)
    cfg = MM_LLMs_Config(clip_config=clip, whisper_config=whisper, llm_config=llama, **hyper)
    model = MM_LLMs.build_random(cfg, device=dev, dtype=torch.bfloat16, seed=0)
    freeze_like_reference(model)
    params = [p for _, p in trainable_parameters(model)]
    gb = GradBuffer(model)
    gb.attach()
    n = gb.flat.numel()
    nbytes = 2 * n
    gen = torch.Generator(device=dev).manual_seed(0)
    for o in range(0, n, 1 << 28):
        k = min(1 << 28, n - o)
        gb.flat[o:o + k] = (torch.randn(k, device=dev, generator=gen) * 1e-3).to(torch.bfloat16)
    live = [p for p in params if p.grad is not None]
    out(f"trainable set: {len(live)} tensors, {n / 1e9:.3f} e9 bf16 gradients = {nbytes / 1e9:.2f} GB")

    # ---- norm pass vs copy of the same bytes
    total = 1000
    sched = LRSchedule("cosine", num_warmup_steps=warmup_steps(0.03, total), num_training_steps=total)
    table = ops.grad_table([p.grad for p in live])
    st = ops.opt_state(dev)
    parts = torch.zeros(ops.GRAD_NORM_PARTS, device=dev, dtype=torch.float64)
    dst = torch.empty_like(gb.flat)

    def norm():
        ops.grad_norm(table, st, parts, max_norm=1.0, skip_nonfinite=True, base_lr=3e-5, schedule="cosine",
                      warmup_steps=sched.num_warmup_steps, total_steps=total)

    norm(), dst.copy_(gb.flat)
    torch.cuda.synchronize()
    r = alternate({"norm": norm, "copy": lambda: dst.copy_(gb.flat)}, args.reps)
    tn, tc = r["norm"][0], r["copy"][0]
    out(f"norm pass: {tn:.3f} ms (median {r['norm'][1]:.3f}) = {nbytes / tn / 1e9:.2f} TB/s read")
    out(f"d2d copy of the same {nbytes / 1e9:.2f} GB: {tc:.3f} ms (median {r['copy'][1]:.3f}) = "
        f"{2 * nbytes / tc / 1e9:.2f} TB/s read + write, {nbytes / tc / 1e9:.2f} TB/s of source bytes")
    out(f"norm pass / copy time: {tn / tc:.3f}")
    del dst
    torch.cuda.empty_cache()

    # ---- opt.step(): plain vs recipe, one graph each, sharing master / moments
    plain = FusedAdamW(params, lr=3e-5, weight_decay=0.0)
    recipe = FusedAdamW(params, lr=3e-5, weight_decay=0.0, max_grad_norm=1.0, lr_schedule=sched, skip_nonfinite=True)
    plain.step()
    recipe.state = plain.state
    recipe.step()
    torch.cuda.synchronize()
    g_plain, g_recipe = graph_of(plain.step), graph_of(recipe.step)
    r = alternate({"plain": g_plain.replay, "recipe": g_recipe.replay}, max(2, args.reps // 2))
    tp, tr = r["plain"][0], r["recipe"][0]
    adam_bytes = 28 * n  # g 2 + p 2 + master / m / v 3 x (4 read + 4 write)
    out(f"opt.step() plain (graph): {tp:.3f} ms (median {r['plain'][1]:.3f}) = {adam_bytes / tp / 1e9:.2f} TB/s")
    out(f"opt.step() clip 1.0 + cosine + skip check (graph): {tr:.3f} ms (median {r['recipe'][1]:.3f}); "
        f"+{tr - tp:.3f} ms over plain")
    del g_plain, g_recipe, plain
    torch.cuda.synchronize()

    # ---- one optimizer step of train.sh: GA = 3 micro-batches of 4, no_sync on the first two, N = 1
    if not args.skip_ga3:
        L, V = 512, llama.vocab_size
        mbs = []
        for i in range(3):
            h = bench.synth_inputs(4, L, V, clip.vision_config.image_size, 2 * whisper.max_source_positions, 1234 + i)
            h["labels"] = h["input_ids"].clone()
            mbs.append({k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in h.items()})
        model.train()
        ts = model.train_step
        gb.flat.zero_()
        ts.llama.grads = gb

        def ga_step():
            recipe.zero_grad()
            for i, mb in enumerate(mbs):
                if i < 2:
                    with ts.no_sync():
                        (model(mb).loss / 3).backward()
                else:
                    (model(mb).loss / 3).backward()
            recipe.step()

        for _ in range(2):
            ga_step()
        torch.cuda.synchronize()
        g = graph_of(ga_step)
        t_ga = min(timed(g.replay, 1) for _ in range(max(3, args.reps // 3)))
        out(f"GA=3 x micro-batch 4 optimizer step, N=1 (one graph): {t_ga:.1f} ms; recipe update "
            f"{tr:.2f} ms of it ({tr / t_ga:.1%}), norm pass {tn:.2f} ms ({tn / t_ga:.1%})")
        out(f"after the step: grad_norm {float(recipe.grad_norm):.4e}, lr {float(recipe.last_lr):.3e}, "
            f"steps {int(recipe.step_count)}, skipped {int(recipe.skipped_steps)}")
    if torch.cuda.device_count() >= 2:
        out("N = 2 (with / without no_sync): not measured by this single-process script")
    else:
        out("N = 2: not measured (one GPU visible)")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
