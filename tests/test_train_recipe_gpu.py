"""The HF Trainer's update recipe on the B200 (train.sh: gradient accumulation, global-norm clipping at 1.0, warmup +
cosine learning rate, overflow-skipped steps): the deterministic gradient-norm kernel against an fp64 norm, the skip of a
non-finite step, whole trajectories against torch (clip_grad_norm_ + torch.optim.AdamW + LambdaLR), gradient
accumulation under `no_sync` against the oracle, one CUDA graph of a whole accumulated step, and two data-parallel ranks.

The learning-rate lambdas of the torch runs are `LRSchedule.lam`, which tests/test_train_recipe_cpu.py pins to
transformers' schedules."""
import contextlib
import copy
import os

import pytest
import torch

from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _ops():
    from macaw_llm_b200 import ops

    return ops


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def norm64(ts):
    return float(sum(t.double().pow(2).sum() for t in ts).sqrt())


def words(st):
    return st.cpu().tolist()


def f32(st, i):
    return float(st.view(torch.float32)[i])


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def bf16_randn(n, seed, scale=1.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(n, device=DEV, generator=g) * scale).to(torch.bfloat16)


# ---------------------------------------------------------------------------------------------------- 1. norm kernel
def test_grad_norm_kernel_sizes_unaligned_and_determinism():
    ops = _ops()
    ts = [bf16_randn(n, seed=i) for i, n in enumerate((1, 7, 8, 4097, 10 ** 6 + 3))]
    base = bf16_randn(10000, seed=9)
    ts += [base[1:4002], base[5003:5003 + 999], base[3:4]]  # 2-, 6- and 6-byte offsets: scalar path
    st, parts = ops.opt_state(DEV), torch.zeros(ops.GRAD_NORM_PARTS, device=DEV, dtype=torch.float64)
    table = ops.grad_table(ts)
    ops.grad_norm(table, st, parts, max_norm=1.0, skip_nonfinite=True, base_lr=1.0)
    ref = norm64(ts)
    got = f32(st, ops.OPT_GRAD_NORM)
    print(f"\n[grad_norm] {got:.9e} vs fp64 {ref:.9e} rel {abs(got - ref) / ref:.2e}")
    assert abs(got - ref) <= 1e-6 * ref
    n32 = torch.tensor(got, dtype=torch.float32)
    assert f32(st, ops.OPT_CLIP_COEF) == float(torch.clamp(1.0 / (n32 + 1e-6), max=1.0))
    assert int(st[ops.OPT_FINITE]) == 1 and int(st[ops.OPT_STEP]) == 1 and int(st[ops.OPT_ARRIVED]) == 0
    bits = int(st[ops.OPT_GRAD_NORM])
    for _ in range(5):  # repeated launches: bit-identical
        ops.grad_norm(table, st, parts, max_norm=1.0, skip_nonfinite=True, base_lr=1.0)
        assert int(st[ops.OPT_GRAD_NORM]) == bits
    # under graph replay
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.grad_norm(table, st, parts, max_norm=1.0, skip_nonfinite=True, base_lr=1.0)
    torch.cuda.current_stream().wait_stream(s)
    with torch.cuda.graph(g):
        ops.grad_norm(table, st, parts, max_norm=1.0, skip_nonfinite=True, base_lr=1.0)
    before = int(st[ops.OPT_STEP])
    for _ in range(3):
        g.replay()
    assert int(st[ops.OPT_GRAD_NORM]) == bits and int(st[ops.OPT_STEP]) == before + 3
    # without clipping and without the finiteness check there is no pass: only the step bookkeeping
    st2 = ops.opt_state(DEV)
    ops.grad_norm(None, st2, parts, base_lr=2.0)
    assert int(st2[ops.OPT_STEP]) == 1 and f32(st2, ops.OPT_LR) == 2.0 and f32(st2, ops.OPT_CLIP_COEF) == 1.0


def test_grad_norm_kernel_int64_indexing():
    """One tensor of 2^31 + 17 elements (4.3 GB of bf16): the elements past index 2^31 are counted."""
    ops = _ops()
    n = (1 << 31) + 17
    big = torch.empty(n, device=DEV, dtype=torch.bfloat16)
    step = 1 << 28
    for i, o in enumerate(range(0, n, step)):
        k = min(step, n - o)
        big[o:o + k] = bf16_randn(k, seed=100 + i, scale=0.01)
    big[-1] = 1000.0  # its square is ~0.5 % of the whole sum
    ref = sum(float(big[o:o + step].float().pow(2).sum(dtype=torch.float64)) for o in range(0, n, step)) ** 0.5
    st, parts = ops.opt_state(DEV), torch.zeros(ops.GRAD_NORM_PARTS, device=DEV, dtype=torch.float64)
    ops.grad_norm(ops.grad_table([big]), st, parts, max_norm=1.0)
    got = f32(st, ops.OPT_GRAD_NORM)
    print(f"\n[grad_norm 2^31+17] {got:.9e} vs fp64 {ref:.9e} rel {abs(got - ref) / ref:.2e}")
    assert abs(got - ref) <= 1e-6 * ref


def test_grad_norm_excludes_none_grads_and_stale_views(tiny_train):
    from macaw_llm_b200.training import FusedAdamW, trainable_parameters
    from tests.golden import gen

    a = torch.nn.Parameter(bf16_randn(300, seed=1))
    b = torch.nn.Parameter(bf16_randn(300, seed=2))
    a.grad, b.grad = bf16_randn(300, seed=3), None
    opt = FusedAdamW([a, b], lr=1e-3, max_grad_norm=1.0)
    opt.step()
    assert abs(float(opt.grad_norm) - norm64([a.grad])) <= 1e-6 * norm64([a.grad])

    model0, spec, hp, weights = tiny_train
    model = copy.deepcopy(model0)
    params = [p for _, p in trainable_parameters(model)]
    opt = FusedAdamW(params, lr=1e-3, max_grad_norm=1.0)
    model.train()
    model.train_step.attention_dropout = False
    for mods, seed in ((("image",), 11), ((), 12)):
        inp = _dev(gen.make_inputs(spec, 2, 16, seed=seed, modalities=mods, with_labels=True))
        opt.zero_grad()
        model(inp).loss.backward()
        opt.step()
    live = [p.grad for p in params if p.grad is not None]
    stale = model.train_step.llama.grads.views[id(model.project_image.weight)]
    assert model.project_image.weight.grad is None and float(stale.float().abs().sum()) > 0
    ref = norm64(live)
    print(f"\n[grad_norm tiny text-only after image] {float(opt.grad_norm):.6e} vs {ref:.6e}; with stale views "
          f"{norm64(live + [stale]):.6e}")
    assert abs(float(opt.grad_norm) - ref) <= 1e-6 * ref


# ---------------------------------------------------------------------------------------------------- torch reference
SHAPES = [(1000, 64), (37,), (4097,), (513, 8)]


def _grads(k, scale=1.0):
    return [bf16_randn(int(torch.tensor(s).prod()), seed=1000 * k + i, scale=scale).view(s) for i, s in enumerate(SHAPES)]


def _params():
    return [torch.nn.Parameter(bf16_randn(int(torch.tensor(s).prod()), seed=77 + i).view(s)) for i, s in enumerate(SHAPES)]


def _torch_run(p0, grad_seq, *, lr, sched, max_norm, wd=0.0, betas=(0.9, 0.999)):
    """clip_grad_norm_ on fp32 copies, torch.optim.AdamW, LambdaLR(sched.lam): master weights, lr per step, norms."""
    ref = [torch.nn.Parameter(p.detach().float().clone()) for p in p0]
    topt = torch.optim.AdamW(ref, lr=lr, betas=betas, eps=1e-8, weight_decay=wd)
    ls = torch.optim.lr_scheduler.LambdaLR(topt, sched.lam)
    lrs, norms = [], []
    for gs in grad_seq:
        for r, g in zip(ref, gs):
            r.grad = g.float().clone()
        norms.append(float(torch.nn.utils.clip_grad_norm_(ref, max_norm)))
        lrs.append(topt.param_groups[0]["lr"])
        topt.step()
        ls.step()
    return ref, lrs, norms


@pytest.mark.parametrize("schedule", ["cosine", "linear", "constant_with_warmup"])
@pytest.mark.parametrize("max_norm", [1e-3, 1e9])
def test_trajectory_matches_torch(schedule, max_norm):
    """12 steps, warmup 3 of 10 (the run goes past the end), clipping every step or never."""
    from macaw_llm_b200.training import FusedAdamW, LRSchedule

    ops = _ops()
    sched = LRSchedule(schedule, num_warmup_steps=3, num_training_steps=10)
    ps = _params()
    init = [p.detach().float().clone() for p in ps]
    seq = [_grads(k) for k in range(12)]
    ref, lrs, norms = _torch_run(ps, seq, lr=1e-2, sched=sched, max_norm=max_norm, wd=0.1, betas=(0.9, 0.95))
    opt = FusedAdamW(ps, lr=1e-2, betas=(0.9, 0.95), weight_decay=0.1, max_grad_norm=max_norm, lr_schedule=sched)
    for k, gs in enumerate(seq):
        for p, g in zip(ps, gs):
            p.grad = g.clone()
        opt.step()
        got_lr = float(opt.last_lr)
        assert abs(got_lr - lrs[k]) <= 1e-7 * abs(lrs[k]), (k, got_lr, lrs[k])
        assert abs(float(opt.grad_norm) - norms[k]) <= 1e-6 * norms[k]
        if k == 0:  # warmup: the first update runs at lr = 0 exactly; the moments still move
            assert got_lr == 0.0
            assert all(torch.equal(opt.state[id(p)][0], w) for p, w in zip(ps, init))
            assert all(float(opt.state[id(p)][1].abs().sum()) > 0 for p in ps)
    assert int(opt.step_count) == 12 and int(opt.skipped_steps) == 0
    errs = [rel(opt.state[id(p)][0], r.detach()) for p, r in zip(ps, ref)]
    clipped = f32(opt.opt_state, ops.OPT_CLIP_COEF)
    print(f"\n[trajectory {schedule} max_norm {max_norm:g}] master rel err {max(errs):.2e}; last clip coef {clipped:.3e}")
    assert max(errs) <= 1e-6
    assert (clipped < 1.0) == (max_norm < 1.0)


# ---------------------------------------------------------------------------------------------------- 2. non-finite
@pytest.mark.parametrize("where", ["inf_last", "nan_mid"])
def test_nonfinite_step_is_skipped(where):
    from macaw_llm_b200.training import FusedAdamW, LRSchedule

    ops = _ops()
    sched = LRSchedule("cosine", num_warmup_steps=2, num_training_steps=8)
    ps = _params()
    seq = [_grads(k) for k in range(6)]
    bad = [g.clone() for g in seq[3]]
    if where == "inf_last":
        bad[-1].view(-1)[-1] = float("inf")
    else:
        bad[1].view(-1)[18] = float("nan")
    ref, lrs, _ = _torch_run(ps, seq[:3] + seq[4:], lr=1e-2, sched=sched, max_norm=1.0)
    opt = FusedAdamW(ps, lr=1e-2, max_grad_norm=1.0, lr_schedule=sched, skip_nonfinite=True)
    for k in range(6):
        for p, g in zip(ps, bad if k == 3 else seq[k]):
            p.grad = g.clone()
        if k == 3:
            snap = [(p.detach().clone(), *(t.clone() for t in opt.state[id(p)])) for p in ps]
            st0 = words(opt.opt_state)
        opt.step()
        if k == 3:
            st1 = words(opt.opt_state)
            assert st1[ops.OPT_FINITE] == 0 and st1[ops.OPT_SKIPPED] == 1 and st1[ops.OPT_APPLY] == 0
            assert st1[ops.OPT_STEP] == st0[ops.OPT_STEP] and st1[ops.OPT_LR] == st0[ops.OPT_LR]
            for p, s in zip(ps, snap):
                now = (p.detach(), *opt.state[id(p)])
                assert all(torch.equal(_bits(a), _bits(b)) for a, b in zip(now, s))
    assert int(opt.step_count) == 5 and int(opt.skipped_steps) == 1
    assert abs(float(opt.last_lr) - lrs[-1]) <= 1e-7 * lrs[-1]
    errs = [rel(opt.state[id(p)][0], r.detach()) for p, r in zip(ps, ref)]
    print(f"\n[skip {where}] master rel err vs torch without that step {max(errs):.2e}")
    assert max(errs) <= 1e-6


# ---------------------------------------------------------------------------------------------------- tiny model
@pytest.fixture(scope="module")
def tiny_train():
    return H.build_tiny_model("cuda", torch.bfloat16)


def _dev(inp):
    return {k: (v.to(torch.bfloat16).cuda() if isinstance(v, torch.Tensor) and v.is_floating_point() else
                (v.cuda() if isinstance(v, torch.Tensor) else v)) for k, v in inp.items()}


def _micro_batches(spec, seeds, mods=("image", "audio")):
    from tests.golden import gen

    return [gen.make_inputs(spec, 2, 14, seed=s, modalities=mods, pad_tail=2, with_labels=True) for s in seeds]


def _accumulate(model, mbs, sync_last=True):
    n = len(mbs)
    for i, mb in enumerate(mbs):
        last = i == n - 1 and sync_last
        with model.train_step.no_sync() if not last else contextlib.nullcontext():
            (model(mb).loss / n).backward()


# ---------------------------------------------------------------------------------------------------- 4. accumulation
def test_accumulation_under_no_sync_matches_oracle(tiny_train, monkeypatch):
    from oracle import macaw_oracle as O
    from macaw_llm_b200 import training

    model0, spec, hp, weights = tiny_train
    model = copy.deepcopy(model0)
    host = _micro_batches(spec, (201, 202, 203))
    mbs = [_dev(h) for h in host]
    model.train()
    model.train_step.attention_dropout = False
    for p in model.parameters():
        p.grad = None
    _accumulate(model, mbs)
    torch.cuda.synchronize()
    sd = H.bf16_round(weights)
    mean = {}
    for h in host:
        h32 = {k: (v.to(torch.bfloat16).float() if isinstance(v, torch.Tensor) and v.is_floating_point() else v)
               for k, v in h.items()}
        _, gr = O.full_loss_and_grads(h32, sd, hp)
        for k, g in gr.items():
            if g is not None:  # modules of modalities absent from the batch
                mean[k] = mean.get(k, 0) + g / len(host)
    named = dict(model.named_parameters())
    worst = {True: ("", 0.0), False: ("", 0.0)}
    for k, g in mean.items():
        is_align = not k.startswith("llm.")
        if is_align and not k.startswith(("project_image.", "transform_image_to_hidden.", "image_align_attention.",
                                          "project_audio.", "transform_audio_to_hidden.", "audio_align_attention.")):
            continue
        e = rel(named[k].grad, g)
        if e > worst[is_align][1]:
            worst[is_align] = (k, e)
        assert e < (5e-2 if is_align else 3e-2), (k, e)
    print(f"\n[accumulation GA=3] worst gradient rel err: llm {worst[False][1]:.3e} ({worst[False][0]}), alignment "
          f"{worst[True][1]:.3e} ({worst[True][0]})")
    # collective count with a 2-rank world: none under no_sync, one per bucket on the boundary micro-batch
    calls = []
    monkeypatch.setattr(training, "allreduce_grads", lambda buf, world, bucket=None, async_op=False: calls.append(bucket))
    model.train_step.set_world(2)
    try:
        with model.train_step.no_sync():
            (model(mbs[0]).loss / 2).backward()
        assert calls == []
        (model(mbs[1]).loss / 2).backward()
        assert sorted(calls) == list(range(len(model.train_step.llama.grads.buckets)))
        model.train_step.finish_allreduce()
    finally:
        model.train_step.set_world(1)
        model.eval()


# ---------------------------------------------------------------------------------------------------- 5. graph
def test_whole_accumulated_step_in_one_graph(tiny_train):
    """zero_grad + 2 x (forward, backward) with no_sync on the first + clipped, cosine-scheduled step, captured once and
    replayed 5 times, against 5 eager steps on a deep copy."""
    from macaw_llm_b200.training import FusedAdamW, LRSchedule, trainable_parameters

    ops = _ops()
    model0, spec, hp, weights = tiny_train
    mbs = [_dev(h) for h in _micro_batches(spec, (301, 302))]
    runs = []
    for _ in range(2):
        m = copy.deepcopy(model0)
        m.train()
        m.train_step.attention_dropout = False
        params = [p for _, p in trainable_parameters(m)]
        opt = FusedAdamW(params, lr=1e-3, max_grad_norm=0.5, lr_schedule=LRSchedule("cosine", 2, 6))
        runs.append((m, params, opt, [p.detach().float().clone() for p in params]))

    def step(m, opt):
        opt.zero_grad()
        _accumulate(m, mbs)
        opt.step()

    (ma, pa, oa, ia), (mb, pb, ob, ib) = runs
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step(ma, oa)  # eager warm-up: builds the norm table, the moments, the optimizer state
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, capture_error_mode="thread_local"):
        step(ma, oa)
    # the capture enqueued nothing: the state is still the warm-up step's
    assert int(oa.step_count) == 1
    step(mb, ob)
    for i in range(5):
        graph.replay()
        step(mb, ob)
        torch.cuda.synchronize()
        wa, wb = words(oa.opt_state), words(ob.opt_state)
        for f in (ops.OPT_STEP, ops.OPT_LR, ops.OPT_SKIPPED):
            assert wa[f] == wb[f], (i, f, wa, wb)
    assert int(oa.step_count) == 6
    worst = ("", 0.0)
    for (n, _), p_a, p_b, w0 in zip(trainable_parameters(ma), pa, pb, ia):
        if id(p_a) not in oa.state:
            continue
        e = rel(oa.state[id(p_a)][0] - w0, ob.state[id(p_b)][0] - w0)
        worst = max(worst, (n, e), key=lambda t: t[1])
    print(f"\n[graph GA=2] graph vs eager: worst relative difference of the accumulated update {worst[1]:.2e} ({worst[0]})")
    # Only atomics make the step non-deterministic: the bf16 atomics of the embedding-table scatter (and the order of
    # fp32 column-sum atomics).  A last-bit gradient difference changes AdamW's normalised update of most elements by
    # about one bf16 ulp (4e-3), but an element whose gradient sits near zero can change its update by up to 2 lr, and
    # the weights then differ in every later forward.  Measured on a B200: 1.4e-3 and 1.5e-2 after 6 steps in two runs; bar 5e-2.
    assert worst[1] < 5e-2


def test_optimizer_graph_is_bit_exact():
    from macaw_llm_b200.training import FusedAdamW, LRSchedule

    sched = LRSchedule("cosine", 2, 6)
    runs = []
    for _ in range(2):
        ps = _params()
        for p, g in zip(ps, _grads(0)):
            p.grad = g
        runs.append((ps, FusedAdamW(ps, lr=1e-2, max_grad_norm=1.0, lr_schedule=sched, skip_nonfinite=True)))
    (pa, oa), (pb, ob) = runs
    oa.step()
    ob.step()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        oa.step()
    for _ in range(4):
        g.replay()
        ob.step()
    assert words(oa.opt_state) == words(ob.opt_state)
    for x, y in zip(pa, pb):
        assert torch.equal(x.detach().view(torch.int16), y.detach().view(torch.int16))
        for s, t in zip(oa.state[id(x)], ob.state[id(y)]):
            assert torch.equal(s.view(torch.int32), t.view(torch.int32))


def test_plain_optimizer_launches_unchanged():
    """Without the recipe arguments: one mm_adamw per tensor, exactly as before."""
    from macaw_llm_b200.training import FusedAdamW

    ops = _ops()
    ps = _params()
    for p, g in zip(ps, _grads(0)):
        p.grad = g
    opt = FusedAdamW(ps, lr=1e-3)
    opt.step()
    torch.cuda.synchronize()
    ops.launch_count_reset()
    opt.step()
    assert ops.launch_count() == len(ps) and opt.opt_state is None
    sch = FusedAdamW(ps, lr=1e-3, max_grad_norm=1.0)
    sch.step()
    ops.launch_count_reset()
    sch.step()
    assert ops.launch_count() == len(ps) + 1


# ---------------------------------------------------------------------------------------------------- 6. two GPUs
def _dp_worker(rank, world, port, out_dir):
    import torch.distributed as dist

    from macaw_llm_b200.training import FusedAdamW, trainable_parameters

    torch.cuda.set_device(rank)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        model, spec, hp, weights = H.build_tiny_model(f"cuda:{rank}", torch.bfloat16)
        model.train()
        model.train_step.attention_dropout = False
        model.train_step.set_world(world)
        mbs = [_dev_on(h, rank) for h in _micro_batches(spec, (401 + 2 * rank, 402 + 2 * rank))]
        params = [p for _, p in trainable_parameters(model)]
        opt = FusedAdamW(params, lr=1e-3, max_grad_norm=0.5)
        opt.zero_grad()
        _accumulate(model, mbs)
        opt.step()  # orders itself after the bucket all-reduces
        torch.cuda.synchronize()
        names = [n for n, _ in trainable_parameters(model)]
        torch.save({"grad_norm": opt.opt_state.cpu(),
                    "master": {n: opt.state[id(p)][0].cpu() for n, p in zip(names, params) if id(p) in opt.state},
                    "grads": {n: p.grad.float().cpu() for n, p in zip(names, params) if p.grad is not None}},
                   os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


def _dev_on(inp, rank):
    return {k: (v.to(torch.bfloat16).to(f"cuda:{rank}") if isinstance(v, torch.Tensor) and v.is_floating_point() else
                (v.to(f"cuda:{rank}") if isinstance(v, torch.Tensor) else v)) for k, v in inp.items()}


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two visible GPUs")
def test_two_ranks_agree_bitwise_and_match_single_process(tmp_path, tiny_train):
    import socket

    import torch.multiprocessing as mp

    from macaw_llm_b200.training import FusedAdamW, trainable_parameters

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_dp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = (torch.load(os.path.join(tmp_path, f"rank{r}.pt")) for r in range(2))
    assert torch.equal(r0["grad_norm"], r1["grad_norm"])
    assert r0["master"].keys() == r1["master"].keys()
    for k in r0["master"]:
        assert torch.equal(r0["master"][k].view(torch.int32), r1["master"][k].view(torch.int32)), k
    # one process on the union of the batches: GA = 4, each loss / 4
    model0, spec, hp, weights = tiny_train
    model = copy.deepcopy(model0)
    model.train()
    model.train_step.attention_dropout = False
    params = [p for _, p in trainable_parameters(model)]
    opt = FusedAdamW(params, lr=1e-3, max_grad_norm=0.5)
    opt.zero_grad()
    _accumulate(model, [_dev(h) for h in _micro_batches(spec, (401, 402, 403, 404))])
    named = dict(trainable_parameters(model))
    for k, g in r0["grads"].items():
        e = rel(g, named[k].grad)
        assert e < (5e-2 if not k.startswith("llm.") else 3e-2), (k, e)
