"""CPU tier: the training recipe's host side.  The learning-rate lambdas of `training.LRSchedule` (which the device
restates in mm_grad_norm) equal transformers' schedules step for step; `warmup_steps` equals
TrainingArguments.get_warmup_steps; the new entry points are declared in the header and bound in _lib.SIGNATURES."""
import inspect
import os
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CASES = [(0, 10), (3, 10), (1, 1), (10, 10), (12, 10), (4, 100), (0, 0), (5, 0)]


def _hf_scheduler(name, warmup, total):
    torch = pytest.importorskip("torch")
    opt_mod = pytest.importorskip("transformers.optimization")
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([p], lr=1.0)
    if name == "constant":
        return opt, opt_mod.get_constant_schedule(opt)
    if name == "constant_with_warmup":
        return opt, opt_mod.get_constant_schedule_with_warmup(opt, num_warmup_steps=warmup)
    fn = {"linear": opt_mod.get_linear_schedule_with_warmup, "cosine": opt_mod.get_cosine_schedule_with_warmup}[name]
    return opt, fn(opt, num_warmup_steps=warmup, num_training_steps=total)


@pytest.mark.parametrize("name", ["constant", "constant_with_warmup", "linear", "cosine"])
@pytest.mark.parametrize("warmup,total", CASES)
def test_lambda_equals_transformers(name, warmup, total):
    """Every step up to twice past the end: lam(k) is the factor LambdaLR applies after k scheduler steps."""
    from macaw_llm_b200.training import LRSchedule

    if name in ("linear", "cosine") and total == 0:
        with pytest.raises(ValueError):
            LRSchedule(name, warmup, total)
        return
    sch = LRSchedule(name, num_warmup_steps=warmup, num_training_steps=total)
    opt, hf = _hf_scheduler(name, warmup, total)
    for k in range(2 * max(total, warmup) + 3):
        assert sch.lam(k) == opt.param_groups[0]["lr"], (name, warmup, total, k)
        opt.step()
        hf.step()


def _hf_warmup_steps(ratio, total):
    ta = pytest.importorskip("transformers").TrainingArguments
    src = inspect.getsource(ta.get_warmup_steps)
    # older releases keep the ratio in `warmup_ratio`; newer ones accept a ratio < 1 in `warmup_steps`
    ns = (types.SimpleNamespace(warmup_steps=0, warmup_ratio=ratio) if "warmup_ratio" in src
          else types.SimpleNamespace(warmup_steps=ratio, warmup_ratio=ratio))
    return ta.get_warmup_steps(ns, total)


@pytest.mark.parametrize("ratio", [0.0, 0.03, 0.1, 0.5, 0.999])
@pytest.mark.parametrize("total", [1, 7, 33, 100, 1000, 12345])
def test_warmup_steps_equals_training_arguments(ratio, total):
    from macaw_llm_b200.training import warmup_steps

    assert warmup_steps(ratio, total) == _hf_warmup_steps(ratio, total)


def test_new_symbols_are_declared_and_bound():
    from macaw_llm_b200 import _lib, ops
    from tests.test_abi import header_symbols

    syms = header_symbols()
    for s in ("mm_grad_norm", "mm_adamw_sched"):
        assert s in syms and s in _lib.SIGNATURES, s
    hdr = open(os.path.join(ROOT, "include", "macaw_b200.h")).read()
    assert f"#define MM_GRAD_NORM_PARTS {ops.GRAD_NORM_PARTS}" in hdr
    for name, i in ops.SCHEDULES.items():
        assert f"#define MM_SCHED_{name.upper()} {i}" in hdr


def test_opt_state_layout_matches_header():
    """ops.opt_state's word offsets mirror `mm_opt_state` (checked by compiling a probe), and a fresh state is the
    documented initial one."""
    import ctypes  # noqa: F401
    import subprocess
    import tempfile

    import torch

    from macaw_llm_b200 import ops

    probe = r'''
#include <stdio.h>
#include <stddef.h>
#include "macaw_b200.h"
int main(void){ printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(mm_opt_state), offsetof(mm_opt_state, step),
  offsetof(mm_opt_state, skipped), offsetof(mm_opt_state, lr), offsetof(mm_opt_state, clip_coef),
  offsetof(mm_opt_state, grad_norm), offsetof(mm_opt_state, finite), offsetof(mm_opt_state, apply),
  offsetof(mm_opt_state, arrived)); return 0; }
'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "p.c")
        open(c, "w").write(probe)
        exe = os.path.join(d, "p")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        got = list(map(int, subprocess.run([exe], capture_output=True, text=True).stdout.split()))
    want = [4 * i for i in (ops.OPT_STEP, ops.OPT_SKIPPED, ops.OPT_LR, ops.OPT_CLIP_COEF, ops.OPT_GRAD_NORM, ops.OPT_FINITE,
                            ops.OPT_APPLY, ops.OPT_ARRIVED)]
    assert got == [32] + want
    st = ops.opt_state("cpu")
    assert st.dtype == torch.int32 and st.numel() == 8
    assert st.view(torch.float32)[ops.OPT_CLIP_COEF] == 1.0 and st[ops.OPT_FINITE] == 1
    assert int(st[ops.OPT_STEP]) == int(st[ops.OPT_SKIPPED]) == int(st[ops.OPT_APPLY]) == int(st[ops.OPT_ARRIVED]) == 0


def test_unscheduled_optimizer_keeps_its_plain_step():
    """FusedAdamW without the recipe arguments is the plain optimizer (host-float lr, no device state)."""
    import torch

    from macaw_llm_b200.training import FusedAdamW, LRSchedule

    p = torch.nn.Parameter(torch.zeros(4))
    assert not FusedAdamW([p], lr=1e-3).scheduled
    assert FusedAdamW([p], max_grad_norm=1.0).scheduled
    assert FusedAdamW([p], lr_schedule=LRSchedule("cosine", 3, 10)).scheduled
    assert FusedAdamW([p], skip_nonfinite=True).scheduled
    with pytest.raises(ValueError):
        LRSchedule("polynomial")


def test_no_sync_suppresses_bucket_allreduce(monkeypatch):
    """Inside TrainStep.no_sync() a bucket sync launches nothing; outside it, one collective per bucket, and
    finish_allreduce is idempotent."""
    from macaw_llm_b200 import training

    calls = []
    monkeypatch.setattr(training, "allreduce_grads", lambda buf, world, bucket=None, async_op=False: calls.append(bucket))
    ts = training.TrainStep.__new__(training.TrainStep)
    ts.llama = training.LlamaTrainer.__new__(training.LlamaTrainer)
    ts.llama.__init__(None)
    ts.llama.grads = types.SimpleNamespace(flat=types.SimpleNamespace(is_cuda=False))
    ts.set_world(2)
    with ts.no_sync():
        for i in range(3):
            ts.llama._sync_bucket(i)
    assert calls == [] and ts.llama.sync_gradients
    for i in range(3):
        ts.llama._sync_bucket(i)
    assert calls == [0, 1, 2]
    ts.set_world(2, overlap=False)
    ts.llama._sync_bucket(0)
    ts.finish_allreduce()
    ts.finish_allreduce()
    assert calls == [0, 1, 2, None]
