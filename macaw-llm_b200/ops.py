"""torch-tensor front end of the C ABI (include/macaw_b200.h).

torch is used only for device memory and streams; every function here launches kernels from libmacaw_b200.so on
torch's current CUDA stream and raises if an operand is not a CUDA tensor (there is no CPU or eager fallback).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from ._lib import AlignArgs, AttnArgs, GemmArgs

ACT_NONE, ACT_GELU, ACT_QUICK_GELU, ACT_SILU = 0, 1, 2, 3
EPI_STD, EPI_SWIGLU, EPI_ROPE = 0, 1, 2

_BF16 = torch.bfloat16
_F16 = torch.float16
_ACT_DTYPE = torch.bfloat16


def ACT():
    """16-bit storage dtype of activations / parameters of the model being run (see set_act_format)."""
    return _ACT_DTYPE


def set_act_format(dtype) -> None:
    """Select the activation format (torch.bfloat16 | torch.float16) for this thread: the Python-side dtype checks and
    the kernel library's thread-local format (mm_set_act_format) move together."""
    global _ACT_DTYPE
    if dtype not in _16BIT:
        raise TypeError(f"macaw_b200: activation format must be bf16 or fp16, got {dtype}")
    if dtype != _ACT_DTYPE or int(_lib.load().mm_get_act_format()) != int(dtype == _F16):
        _lib.load().mm_set_act_format(int(dtype == _F16))
        _ACT_DTYPE = dtype
_16BIT = (torch.bfloat16, torch.float16)


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed (rc={rc}): {_lib.last_error()}")


def _cuda(t: torch.Tensor, dtype=None, name: str = "tensor") -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"macaw_b200: {name} must be a CUDA tensor (no CPU fallback exists)")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"macaw_b200: {name} must be {dtype}, got {t.dtype}")
    if t.device.index != torch.cuda.current_device():
        # kernels are launched on the CURRENT device's stream: a tensor of another GPU would be used with the wrong stream
        raise RuntimeError(f"macaw_b200: {name} lives on {t.device} but the current CUDA device is "
                           f"cuda:{torch.cuda.current_device()}; wrap the call in torch.cuda.device(...)")
    return t


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


# Optional per-launch CUDA-event profiling of the GEMM kernel (bench.py's live roofline): when PROFILE is a list, every
# mm_gemm_fwd launch appends (TAG, flops, start_event, end_event) recorded on the launching stream.
PROFILE = None
TAG = "gemm"


def launch_count() -> int:
    return int(_lib.load().mm_launch_count())


def launch_count_reset() -> None:
    _lib.load().mm_launch_count_reset()


# ---------------------------------------------------------------------------------------------------- GEMM
def gemm_raw(*, M, N, K, A, lda, B, ldb, Cout, ldc, batch=1, a_bs=0, b_bs=0, c_bs=0, batch2=1, a_bs2=0, b_bs2=0,
             c_bs2=0, b_mn_major=False, c_fp32=False, epi=EPI_STD, act=ACT_NONE, alpha=1.0, bias=None, bias_bs=0,
             row_scale=None, residual=None, ldr=0, r_bs=0, r_bs2=0, res_row_mod=0, rope_cos=None, rope_sin=None,
             rope_T=0, rope_cols=0, rope_pos=None, c_trans=False, a_fp16=None, b_fp16=None, c_fp16=None,
             bias_rs=None, bias2=None, bias2_rs=None, a_mn_major=False, sumsq_out=None, rs_sumsq=None, rs_parts=0,
             rs_eps=0.0, streamk: Optional[torch.Tensor] = None) -> None:
    """Direct binding of mm_gemm_fwd; pointers are ints (data_ptr() + byte offsets).  Operand / output formats default to
    the current activation format (ACT()): fp16 for an fp16 model, bf16 otherwise."""
    f16 = ACT() == _F16
    a_fp16 = f16 if a_fp16 is None else a_fp16
    b_fp16 = f16 if b_fp16 is None else b_fp16
    c_fp16 = (f16 and not c_fp32) if c_fp16 is None else c_fp16
    a = GemmArgs(M, N, K, batch, batch2, A, lda, a_bs, a_bs2, B, ldb, b_bs, b_bs2, int(b_mn_major), Cout, ldc, c_bs,
                 c_bs2, int(c_fp32), epi, act, float(alpha), bias, bias_bs, row_scale, residual, ldr, r_bs, r_bs2,
                 res_row_mod, rope_cos, rope_sin, rope_T, rope_cols, rope_pos, int(c_trans), int(a_fp16), int(b_fp16), int(c_fp16),
                 bias_rs, bias2, bias2_rs, int(a_mn_major), sumsq_out, rs_sumsq, int(rs_parts), float(rs_eps),
                 None if streamk is None else streamk.data_ptr(), 0 if streamk is None else streamk.numel() * streamk.element_size())
    if PROFILE is None:
        _check(_lib.load().mm_gemm_fwd(C.byref(a), _stream()), "mm_gemm_fwd")
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _check(_lib.load().mm_gemm_fwd(C.byref(a), _stream()), "mm_gemm_fwd")
    e1.record()
    PROFILE.append((TAG, 2.0 * M * N * K * batch * max(1, batch2), e0, e1))


def gemm_plan(*, M: int, N: int, K: int, batch: int = 1, batch2: int = 1, epi: int = EPI_STD, b_mn_major: bool = False,
              a_mn_major: bool = False, c_fp32: bool = False, c_trans: bool = False, fp16: bool = False,
              streamk: bool = False) -> dict:
    """The schedule mm_gemm_fwd would pick for a dense, 16-byte-aligned GEMM of this shape (mm_gemm_plan: the host-side
    dispatch run without touching memory or launching — works without a GPU, where the library assumes 148 SMs).
    `streamk=True` hands the dispatcher a stream-K workspace, as the LLaMA stack does."""
    lib = _lib.load()
    fake = 1 << 20  # operand addresses are only checked for null / alignment
    lda = M if a_mn_major else K
    ldb = N if b_mn_major else K
    n_out = N // 2 if epi == EPI_SWIGLU else N
    ldc = M if c_trans else n_out
    ws = int(lib.mm_gemm_streamk_workspace_bytes()) if streamk else 0
    rope = dict(rope_cos=fake, rope_sin=fake, rope_T=max(1, M), rope_cols=(N // 128) * 128) if epi == EPI_ROPE else {}
    kw = dict(M=M, N=N, K=K, batch=batch, batch2=batch2, A=fake, lda=lda, a_bs=M * K, a_bs2=M * K * batch, B=fake, ldb=ldb,
              b_bs=N * K, b_bs2=N * K * batch, b_mn_major=int(b_mn_major), C=fake, ldc=ldc, c_bs=M * n_out,
              c_bs2=M * n_out * batch, c_fp32=int(c_fp32), epi=epi, act=ACT_NONE, alpha=1.0, c_trans=int(c_trans),
              a_fp16=int(fp16), b_fp16=int(fp16), c_fp16=int(fp16 and not c_fp32), a_mn_major=int(a_mn_major),
              sk_workspace=fake if streamk else None, sk_workspace_bytes=ws, **rope)
    a = GemmArgs(**kw)
    plan = _lib.GemmPlan()
    _check(lib.mm_gemm_plan(C.byref(a), C.byref(plan)), "mm_gemm_plan")
    d = {name: int(getattr(plan, name)) for name, _ in _lib.GemmPlan._fields_}
    d["fill"] = d["units"] / float(d["waves"] * d["workers"])  # share of the scheduled tile slots that carry work
    return d


def linear(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, *, act: int = ACT_NONE,
           residual: Optional[torch.Tensor] = None, res_row_mod: int = 0, out: Optional[torch.Tensor] = None,
           out_fp32: bool = False, alpha: float = 1.0, row_scale: Optional[torch.Tensor] = None, epi: int = EPI_STD,
           rope=None, out_dtype=None, sumsq_out: Optional[torch.Tensor] = None, rms_from=None) -> torch.Tensor:
    """out = epilogue(alpha * x @ w.T): x (M, K) bf16 or fp16 with unit inner stride, w (N, K) bf16 or fp16 (an nn.Linear
    weight); out bf16 (default), fp16 or fp32 (`out_dtype` / the dtype of `out`)."""
    _cuda(x, None, "x"); _cuda(w, None, "w")
    assert x.dtype in _16BIT and w.dtype in _16BIT, (x.dtype, w.dtype)
    assert x.dim() == 2 and w.dim() == 2 and x.shape[1] == w.shape[1], (x.shape, w.shape)
    assert x.stride(1) == 1 and w.stride(1) == 1
    M, K = x.shape
    N = w.shape[0]
    n_out = N // 2 if epi == EPI_SWIGLU else N
    if out is None:
        out = torch.empty((M, n_out), device=x.device,
                          dtype=out_dtype if out_dtype is not None else (torch.float32 if out_fp32 else ACT()))
    assert out.shape[0] == M and out.shape[1] == n_out and out.stride(1) == 1
    kw = {}
    if residual is not None:
        _cuda(residual, ACT(), "residual")
        assert residual.stride(-1) == 1
        kw.update(residual=residual.data_ptr(), ldr=residual.stride(0), res_row_mod=res_row_mod)
    if rope is not None:
        cos, sin, T, cols = rope[:4]
        kw.update(rope_cos=cos.data_ptr(), rope_sin=sin.data_ptr(), rope_T=T, rope_cols=cols)
        if len(rope) > 4 and rope[4] is not None:  # device-side position offset (int32 tensor)
            kw.update(rope_pos=rope[4].data_ptr())
    if sumsq_out is not None:  # (M, N/32) fp32: per-chunk sums of squares of the stored outputs (next RMSNorm's statistic)
        assert sumsq_out.dtype == torch.float32 and sumsq_out.is_contiguous() and sumsq_out.shape == (M, (N + 31) // 32)
        kw.update(sumsq_out=sumsq_out.data_ptr())
    if rms_from is not None:   # (partials (M, parts) fp32, eps): RMSNorm row scale derived in this GEMM's epilogue
        parts, eps = rms_from
        assert parts.dtype == torch.float32 and parts.is_contiguous() and parts.shape[0] == M and row_scale is None
        kw.update(rs_sumsq=parts.data_ptr(), rs_parts=parts.shape[1], rs_eps=eps)
    if STREAMK is not None and STREAMK.device == x.device:
        kw.update(streamk=STREAMK)
    gemm_raw(M=M, N=N, K=K, A=x.data_ptr(), lda=x.stride(0), B=w.data_ptr(), ldb=w.stride(0), Cout=out.data_ptr(),
             ldc=out.stride(0), c_fp32=out.dtype == torch.float32, c_fp16=out.dtype == _F16, a_fp16=x.dtype == _F16,
             b_fp16=w.dtype == _F16, epi=epi, act=act, alpha=alpha, bias=_ptr(bias), row_scale=_ptr(row_scale), **kw)
    return out


# Stream-K workspace handed to every `linear()` launch while set (see mm_gemm_args.sk_workspace).  The OWNER sets it
# around a section whose GEMMs run one after another on a single stream (the LLaMA stack) and clears it afterwards: two
# GEMMs sharing one workspace must never run concurrently.
STREAMK: Optional[torch.Tensor] = None


def streamk_workspace(device) -> torch.Tensor:
    """A zero-initialised stream-K workspace (flags + one fp32 accumulator slot per SM) on `device`."""
    _lib.load()
    with torch.cuda.device(device):
        n = int(_lib.load().mm_gemm_streamk_workspace_bytes())
    return torch.zeros((n + 15) // 16 * 4, device=device, dtype=torch.int32)


def linear_thin(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, *, act: int = ACT_NONE,
                residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                row_scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = epilogue(x @ w.T) for a THIN x (a few rows, e.g. one decode step): operands are swapped so the weight rows
    fill the 128-row MMA tile (weight-streaming regime) and the epilogue stores transposed.  Same semantics as `linear`
    with the standard epilogue: row_scale scales rows of x, bias is per output feature, residual/out are (M, N)."""
    _cuda(x, ACT(), "x"); _cuda(w, ACT(), "w")
    M, K = x.shape
    N = w.shape[0]
    assert x.stride(1) == 1 and w.stride(1) == 1 and w.shape[1] == K
    if out is None:
        out = torch.empty((M, N), device=x.device, dtype=ACT())
    assert out.shape == (M, N) and out.stride(1) == 1
    kw = {}
    if residual is not None:
        assert residual.stride(1) == 1
        kw.update(residual=residual.data_ptr(), ldr=residual.stride(0))
    # swapped problem: M' = N (weight rows), N' = M (activation rows)
    if STREAMK is not None and STREAMK.device == x.device:
        kw.update(streamk=STREAMK)
    gemm_raw(M=N, N=M, K=K, A=w.data_ptr(), lda=w.stride(0), B=x.data_ptr(), ldb=x.stride(0), Cout=out.data_ptr(),
             ldc=out.stride(0), c_fp32=out.dtype == torch.float32, act=act, bias=_ptr(bias), row_scale=_ptr(row_scale),
             c_trans=True, **kw)
    return out


THIN_SPLITS = 4  # K slices of a thin (decode) GEMM: 32..172-tile grids become 128..688 units on 148 SMs


def linear_thin_splitk(x: torch.Tensor, w: torch.Tensor, *, residual: Optional[torch.Tensor] = None,
                       out: Optional[torch.Tensor] = None, row_scale: Optional[torch.Tensor] = None,
                       splits: Optional[int] = None) -> torch.Tensor:
    """`linear_thin` (no bias / activation) with the K dimension split over `splits` CTAs per weight tile: fp32 partials +
    mm_thin_reduce.  Falls back to `linear_thin` when K does not split into 64-element multiples."""
    _cuda(x, ACT(), "x"); _cuda(w, ACT(), "w")
    M, K = x.shape
    N = w.shape[0]
    S = THIN_SPLITS if splits is None else int(splits)
    if S <= 1 or K % (S * 64) != 0:
        return linear_thin(x, w, residual=residual, out=out, row_scale=row_scale)
    assert x.stride(1) == 1 and w.stride(1) == 1 and w.shape[1] == K
    Kc = K // S
    Mp = (M + 3) // 4 * 4
    part = torch.empty((S, N, Mp), device=x.device, dtype=torch.float32)
    gemm_raw(M=N, N=M, K=Kc, batch=S, A=w.data_ptr(), lda=w.stride(0), a_bs=Kc, B=x.data_ptr(), ldb=x.stride(0), b_bs=Kc,
             Cout=part.data_ptr(), ldc=Mp, c_bs=N * Mp, c_fp32=True)
    if out is None:
        out = torch.empty((M, N), device=x.device, dtype=ACT())
    assert out.shape == (M, N) and out.stride(1) == 1
    _check(_lib.load().mm_thin_reduce(part.data_ptr(), S, N, M, Mp, _ptr(row_scale), _ptr(residual),
                                      0 if residual is None else residual.stride(0), out.data_ptr(), out.stride(0),
                                      _stream()), "mm_thin_reduce")
    return out


THIN_RES, THIN_SWIGLU, THIN_QKV = 0, 1, 2


def linear_thin_fused(x: torch.Tensor, w: torch.Tensor, mode: int, *, row_scale: Optional[torch.Tensor] = None,
                      rms_from=None, residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                      sumsq_out: Optional[torch.Tensor] = None, rope=None, cache: Optional[torch.Tensor] = None, t0: int = 0,
                      t0_dev: Optional[torch.Tensor] = None, splits: Optional[int] = None) -> torch.Tensor:
    """Decode-step GEMM x (M <= 64, K) @ w (N, K)^T with K split over `splits` CTAs per weight tile (fp32 partials) and ONE
    fused tail kernel (mm_thin_fused):
      THIN_RES     out = rs * xW^T + residual (in place allowed); sumsq_out (M, N/32) fp32 receives the next RMSNorm's statistic
      THIN_SWIGLU  out (M, N/2) = silu(gate) * up of the [32 gate | 32 up]-interleaved fused weight
      THIN_QKV     N = 3E: RoPE on q / k (rope = (cos, sin, pos_dev | None)), q -> out (M, 3E) columns [0, E), k / v -> `cache`
                   (B, Tmax, 2, E) at slot t0 / *t0_dev
    rs: `row_scale` (M,) fp32, or rms_from = (partials (M, parts) fp32, eps): rsqrt(mean(x^2) + eps) from a THIN_RES pass."""
    _cuda(x, ACT(), "x"); _cuda(w, ACT(), "w")
    M, K = x.shape
    N = w.shape[0]
    assert x.stride(1) == 1 and w.stride(1) == 1 and w.shape[1] == K and M <= 64
    sk = None  # stream-K needs a full wave of tiles to hide its hand-over behind: a decode GEMM has 32..172 tiles
    S = THIN_SPLITS if splits is None else int(splits)
    if S < 1 or K % (S * 64) != 0:
        S = 1
    Kc = K // S
    Mp = (M + 3) // 4 * 4
    dev = x.device
    part = torch.empty((S, N, Mp), device=dev, dtype=torch.float32)
    # fixed split-K factor; the tail kernel adds the partial sums up
    gemm_raw(M=N, N=M, K=Kc, batch=S, A=w.data_ptr(), lda=w.stride(0), a_bs=Kc, B=x.data_ptr(), ldb=x.stride(0), b_bs=Kc,
             Cout=part.data_ptr(), ldc=Mp, c_bs=N * Mp, c_fp32=True, streamk=sk)
    n_out = N // 2 if mode == THIN_SWIGLU else N
    if out is None:
        out = torch.empty((M, n_out), device=dev, dtype=ACT())
    assert out.shape == (M, n_out) and out.stride(1) == 1
    a = _lib.ThinArgs()
    a.part, a.splits, a.N, a.M, a.ldp, a.mode = part.data_ptr(), S, N, M, Mp, int(mode)
    a.row_scale = _ptr(row_scale)
    if rms_from is not None:
        parts, eps = rms_from
        assert row_scale is None and parts.dtype == torch.float32 and parts.is_contiguous() and parts.shape[0] == M
        a.rs_sumsq, a.rs_parts, a.rs_K, a.rs_eps = parts.data_ptr(), parts.shape[1], K, float(eps)
    if residual is not None:
        _cuda(residual, ACT(), "residual")
        assert mode == THIN_RES and residual.stride(1) == 1
        a.residual, a.ldr = residual.data_ptr(), residual.stride(0)
    a.out, a.ldo = out.data_ptr(), out.stride(0)
    if sumsq_out is not None:
        assert mode == THIN_RES and sumsq_out.dtype == torch.float32 and sumsq_out.is_contiguous() and sumsq_out.shape == (M, N // 32)
        a.sumsq_out = sumsq_out.data_ptr()
    if mode == THIN_QKV:
        cos, sin, pos_dev = rope
        _cuda(cache, ACT(), "cache")
        E = N // 3
        assert cache.is_contiguous() and cache.dim() == 4 and cache.shape[0] == M and cache.shape[2] == 2 and cache.shape[3] == E
        a.rope_cos, a.rope_sin, a.pos_dev, a.E = cos.data_ptr(), sin.data_ptr(), _ptr(pos_dev), E
        a.cache, a.Tmax, a.t0, a.t0_dev = cache.data_ptr(), cache.shape[1], int(t0), _ptr(t0_dev)
    _check(_lib.load().mm_thin_fused(C.byref(a), _stream()), "mm_thin_fused")
    return out


def splitk_reduce(partial: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor) -> torch.Tensor:
    _cuda(partial, torch.float32, "partial"); _cuda(out, None, "out")
    assert out.dtype in _16BIT
    S, M, N = partial.shape
    _check(_lib.load().mm_splitk_reduce(partial.data_ptr(), S, M, N, _ptr(bias), out.data_ptr(), out.stride(0),
                                        int(out.dtype == _F16), _stream()), "mm_splitk_reduce")
    return out


# ---------------------------------------------------------------------------------------------------- attention
def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, scale: float, causal: bool = False,
              key_mask: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None, impl: int = 0,
              tk_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
    """q (B, Tq, H, hd), k/v (B, Tk, H, hd) bf16 views (hd contiguous, arbitrary other strides) -> (B, Tq, H, hd)."""
    for n, t in (("q", q), ("k", k), ("v", v)):
        _cuda(t, ACT(), n)
        assert t.dim() == 4 and t.stride(3) == 1
    B, Tq, H, hd = q.shape
    Tk = k.shape[1]
    if out is None:
        out = torch.empty((B, Tq, H, hd), device=q.device, dtype=ACT())
    if key_mask is not None:
        _cuda(key_mask, torch.int32, "key_mask")
        assert key_mask.shape == (B, Tk) and key_mask.is_contiguous()
    a = AttnArgs(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), B, H, Tq, Tk, hd,
                 q.stride(0), q.stride(1), q.stride(2), k.stride(0), k.stride(1), k.stride(2),
                 v.stride(0), v.stride(1), v.stride(2), out.stride(0), out.stride(1), out.stride(2),
                 _ptr(key_mask), int(causal), float(scale), int(impl), _ptr(tk_dev))
    _check(_lib.load().mm_attn_fwd(C.byref(a), _stream()), "mm_attn_fwd")
    return out


# ---------------------------------------------------------------------------------------------------- norms
def rmsnorm(x: torch.Tensor, w: torch.Tensor, eps: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _cuda(x, ACT(), "x"); _cuda(w, ACT(), "w")
    assert x.is_contiguous()
    cols = x.shape[-1]
    rows = x.numel() // cols
    if out is None:
        out = torch.empty_like(x)
    _check(_lib.load().mm_rmsnorm_fwd(x.data_ptr(), w.data_ptr(), out.data_ptr(), rows, cols, float(eps), _stream()),
           "mm_rmsnorm_fwd")
    return out


def rms_rstd(x: torch.Tensor, eps: float) -> torch.Tensor:
    """fp32 rsqrt(mean(x^2) + eps) per row of a contiguous bf16 (rows, cols) tensor."""
    _cuda(x, ACT(), "x")
    assert x.is_contiguous()
    cols = x.shape[-1]
    rows = x.numel() // cols
    out = torch.empty((rows,), device=x.device, dtype=torch.float32)
    _check(_lib.load().mm_rms_rstd(x.data_ptr(), out.data_ptr(), rows, cols, float(eps), _stream()), "mm_rms_rstd")
    return out


def layernorm(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, eps: float,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x (rows, cols) bf16 with unit inner stride (row stride free)."""
    _cuda(x, ACT(), "x"); _cuda(w, ACT(), "w"); _cuda(b, ACT(), "b")
    assert x.dim() == 2 and x.stride(1) == 1
    rows, cols = x.shape
    if out is None:
        out = torch.empty((rows, cols), device=x.device, dtype=ACT())
    _check(_lib.load().mm_layernorm_fwd(x.data_ptr(), x.stride(0), w.data_ptr(), b.data_ptr(), out.data_ptr(),
                                        out.stride(0), rows, cols, float(eps), _stream()), "mm_layernorm_fwd")
    return out


# ---------------------------------------------------------------------------------------------------- gathers / layout
def embed_gather(table: torch.Tensor, ids: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[i] = table[ids[i]]; ids any integer dtype (converted to int64 on device), out (n, dim) row stride free."""
    _cuda(table, ACT(), "table"); _cuda(ids, None, "ids")
    ids64 = ids.reshape(-1).to(torch.int64).contiguous()  # (a strided 1-D view survives reshape(-1))
    n, dim = ids64.numel(), table.shape[1]
    if out is None:
        out = torch.empty((n, dim), device=table.device, dtype=ACT())
    assert out.stride(-1) == 1
    _check(_lib.load().mm_embed_gather(table.data_ptr(), table.shape[0], dim, ids64.data_ptr(), n, out.data_ptr(),
                                       out.stride(0), _stream()), "mm_embed_gather")
    return out


def splice_prefix(text: torch.Tensor, prefix: Optional[torch.Tensor], mask_in: Optional[torch.Tensor],
                  labels_in: Optional[torch.Tensor]):
    """text (B, L, E), prefix (B, P, E) -> embeds (B, P + L, E), mask (B, P + L) | None, labels (B, P + L) | None."""
    _cuda(text, ACT(), "text")
    B, L, E = text.shape
    P = 0 if prefix is None else prefix.shape[1]
    assert text.is_contiguous() and (prefix is None or prefix.is_contiguous())
    dst = torch.empty((B, P + L, E), device=text.device, dtype=ACT())
    mask_out = labels_out = None
    if mask_in is not None:
        mask_in = _cuda(mask_in, None, "attention_mask").to(torch.int64).contiguous()
        mask_out = torch.empty((B, P + L), device=text.device, dtype=torch.int64)
    if labels_in is not None:
        labels_in = _cuda(labels_in, None, "labels").to(torch.int64).contiguous()
        labels_out = torch.empty((B, P + L), device=text.device, dtype=torch.int64)
    _check(_lib.load().mm_splice_prefix(text.data_ptr(), _ptr(prefix), dst.data_ptr(), B, L, P, E, _ptr(mask_in),
                                        _ptr(mask_out), _ptr(labels_in), _ptr(labels_out), _stream()),
           "mm_splice_prefix")
    return dst, mask_out, labels_out


def patchify(images: torch.Tensor, patch: int, ldo: int) -> torch.Tensor:
    _cuda(images, ACT(), "images")
    assert images.is_contiguous()
    B, Cc, H, W = images.shape
    out = torch.empty((B * (H // patch) * (W // patch), ldo), device=images.device, dtype=ACT())
    _check(_lib.load().mm_patchify(images.data_ptr(), B, Cc, H, W, patch, out.data_ptr(), ldo, _stream()),
           "mm_patchify")
    return out


def transpose_pad(x: torch.Tensor, pad: int) -> torch.Tensor:
    """(B, C, T) -> (B, T + 2 pad, C) with zero pad rows."""
    _cuda(x, ACT(), "x")
    assert x.is_contiguous()
    B, Cc, T = x.shape
    out = torch.empty((B, T + 2 * pad, Cc), device=x.device, dtype=ACT())
    _check(_lib.load().mm_transpose_pad(x.data_ptr(), B, Cc, T, pad, out.data_ptr(), _stream()), "mm_transpose_pad")
    return out


def cast_f16(x: torch.Tensor) -> torch.Tensor:
    """bf16 (..., cols) contiguous -> fp16 copy (mm_cast_bf16_f16)."""
    _cuda(x, torch.bfloat16, "x")
    assert x.is_contiguous()
    cols = x.shape[-1]
    rows = x.numel() // cols
    y = torch.empty(x.shape, device=x.device, dtype=_F16)
    _check(_lib.load().mm_cast_bf16_f16(x.data_ptr(), cols, y.data_ptr(), cols, rows, cols, _stream()), "mm_cast_bf16_f16")
    return y


def add_rows(x: torch.Tensor, add: Optional[torch.Tensor], out: torch.Tensor) -> torch.Tensor:
    """out[r] = x[r] + add[r % add.shape[0]] over 2-D bf16 views with unit inner stride."""
    _cuda(x, ACT(), "x"); _cuda(out, ACT(), "out")
    rows, cols = x.shape
    assert x.stride(1) == 1 and out.stride(1) == 1 and out.shape == x.shape
    if add is None:
        _check(_lib.load().mm_copy_rows(x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0), rows, cols,
                                        _stream()), "mm_copy_rows")
    else:
        _cuda(add, ACT(), "add")
        assert add.stride(1) == 1 and add.shape[1] == cols
        _check(_lib.load().mm_add_rows(x.data_ptr(), x.stride(0), add.data_ptr(), add.stride(0), add.shape[0],
                                       out.data_ptr(), out.stride(0), rows, cols, _stream()), "mm_add_rows")
    return out


# ---------------------------------------------------------------------------------------------------- alignment
ALIGN_MODE = 0  # 0: one cooperative launch with grid-wide barriers between the phases; 1: three stream-ordered launches


def align_fused(table: torch.Tensor, qt: torch.Tensor, stats: torch.Tensor, out: Optional[torch.Tensor] = None,
                mode: Optional[int] = None, keep: Optional[dict] = None):
    """Fused absorbed-form alignment attention (mm_align_fwd).  table (V, E) fp16; qt (R, E) fp16 absorbed queries;
    stats (R, 2) fp32 = [row_bias, extra score] -> (ctx~ (R, E) fp16, p_sum_real (R,), p_extra (R,))."""
    _cuda(table, _F16, "table"); _cuda(qt, _F16, "qt"); _cuda(stats, torch.float32, "stats")
    R, E = qt.shape
    V = table.shape[0]
    assert table.shape[1] == E and table.stride(1) == 1 and qt.stride(1) == 1 and stats.shape == (R, 2) and stats.is_contiguous()
    dev = qt.device
    if out is None:
        out = torch.empty((R, E), device=dev, dtype=_F16)
    assert out.shape == (R, E) and out.stride(1) == 1 and out.dtype == _F16
    Vp = (V + 7) // 8 * 8
    P = torch.empty((R, Vp), device=dev, dtype=_F16)
    lib = _lib.load()
    ws = torch.empty((int(lib.mm_align_workspace_bytes(R, V)) + 15) // 16 * 4, device=dev, dtype=torch.int32)
    psum = torch.empty((R,), device=dev, dtype=torch.float32)
    pext = torch.empty((R,), device=dev, dtype=torch.float32)
    inv_l = torch.empty((R,), device=dev, dtype=torch.float32) if keep is not None else None
    a = AlignArgs(table.data_ptr(), V, E, table.stride(0), qt.data_ptr(), R, qt.stride(0), stats.data_ptr(),
                  stats.data_ptr() + 4, 2, out.data_ptr(), out.stride(0), psum.data_ptr(), pext.data_ptr(), P.data_ptr(), Vp,
                  ws.data_ptr(), ALIGN_MODE if mode is None else int(mode), _ptr(inv_l))
    if keep is not None:  # the training step keeps the un-normalised probabilities and 1 / l for the backward pass
        keep.update(P=P, inv_l=inv_l)
    if PROFILE is None:
        _check(lib.mm_align_fwd(C.byref(a), _stream()), "mm_align_fwd")
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _check(lib.mm_align_fwd(C.byref(a), _stream()), "mm_align_fwd")
        e1.record()
        PROFILE.append(("align.fused", 4.0 * R * V * E, e0, e1))
    return out, psum, pext


def align_softmax(scores: torch.Tensor, stats: torch.Tensor, P: torch.Tensor, V: int):
    """scores fp32 (R, >=V); stats fp32 (R, 2) = [row_bias, extra_score]; P bf16 (R, ldp) -> (p_sum_real, p_extra)."""
    _cuda(scores, torch.float32, "scores"); _cuda(stats, torch.float32, "stats"); _cuda(P, ACT(), "P")
    R = scores.shape[0]
    assert stats.shape == (R, 2) and stats.is_contiguous() and P.shape[0] == R
    psum = torch.empty((R,), device=scores.device, dtype=torch.float32)
    pext = torch.empty((R,), device=scores.device, dtype=torch.float32)
    _check(_lib.load().mm_align_softmax(scores.data_ptr(), scores.stride(0), stats.data_ptr(), stats.data_ptr() + 4, 2,
                                        P.data_ptr(), P.stride(0), psum.data_ptr(), pext.data_ptr(), R, V, _stream()),
           "mm_align_softmax")
    return psum, pext


def align_ctx_fixup(ctx: torch.Tensor, psum: torch.Tensor, pext: torch.Tensor, b_v: torch.Tensor,
                    bias_v: torch.Tensor, head_dim: int) -> torch.Tensor:
    _cuda(ctx, ACT(), "ctx")
    Nq, E = ctx.shape
    _check(_lib.load().mm_align_ctx_fixup(ctx.data_ptr(), ctx.stride(0), psum.data_ptr(), pext.data_ptr(),
                                          b_v.data_ptr(), bias_v.data_ptr(), Nq, E, head_dim, _stream()),
           "mm_align_ctx_fixup")
    return ctx


# ---------------------------------------------------------------------------------------------------- decode helpers
def kv_append(qkv: torch.Tensor, B: int, T_new: int, cache: torch.Tensor, t0: int,
              t0_dev: Optional[torch.Tensor] = None) -> None:
    """qkv (B*T_new, 3E) fused activation -> cache (B, Tmax, 2, E) at positions t0 .. t0+T_new-1 (K and V thirds)."""
    _cuda(qkv, ACT(), "qkv"); _cuda(cache, ACT(), "cache")
    E = cache.shape[-1]
    assert qkv.shape == (B * T_new, 3 * E) and qkv.stride(1) == 1 and cache.is_contiguous() and cache.shape[2] == 2
    _check(_lib.load().mm_kv_append(qkv.data_ptr(), qkv.stride(0), B, T_new, E, cache.data_ptr(), cache.shape[1], t0,
                                    _ptr(t0_dev), _stream()), "mm_kv_append")


def rope_rows(x: torch.Tensor, rot_cols: int, cos: torch.Tensor, sin: torch.Tensor, rope_T: int,
              pos_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
    """In-place rotate-half RoPE (head_dim 128) on the first rot_cols columns of thin bf16 rows."""
    _cuda(x, ACT(), "x")
    assert x.dim() == 2 and x.stride(1) == 1
    _check(_lib.load().mm_rope_rows(x.data_ptr(), x.stride(0), x.shape[0], rot_cols, cos.data_ptr(), sin.data_ptr(), rope_T,
                                    _ptr(pos_dev), _stream()), "mm_rope_rows")
    return x


def swiglu_rows(gu: torch.Tensor, I: int) -> torch.Tensor:
    """(rows, 2I) [32 gate | 32 up]-interleaved product -> (rows, I) silu(gate) * up."""
    _cuda(gu, ACT(), "gu")
    assert gu.dim() == 2 and gu.stride(1) == 1 and gu.shape[1] == 2 * I
    out = torch.empty((gu.shape[0], I), device=gu.device, dtype=ACT())
    _check(_lib.load().mm_swiglu_rows(gu.data_ptr(), gu.stride(0), gu.shape[0], I, out.data_ptr(), out.stride(0),
                                      _stream()), "mm_swiglu_rows")
    return out


def argmax_rows(logits: torch.Tensor) -> torch.Tensor:
    """Greedy token per row of bf16 logits (rows, V) with unit inner stride -> int64 (rows,)."""
    _cuda(logits, ACT(), "logits")
    assert logits.dim() == 2 and logits.stride(1) == 1
    out = torch.empty((logits.shape[0],), device=logits.device, dtype=torch.int64)
    _check(_lib.load().mm_argmax_rows(logits.data_ptr(), logits.stride(0), logits.shape[0], logits.shape[1],
                                      out.data_ptr(), _stream()), "mm_argmax_rows")
    return out


# ---------------------------------------------------------------------------------------------------- loss
def ce_loss(logits: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
    """Shifted CE (mean over labels != -100) of bf16 logits (B, T, V) against int64 labels (B, T); returns fp32 scalar."""
    _cuda(logits, ACT(), "logits"); _cuda(labels, torch.int64, "labels")
    assert logits.is_contiguous() and labels.is_contiguous()
    B, T, V = logits.shape
    acc = torch.zeros((2,), device=logits.device, dtype=torch.float32)
    cnt = acc[1:].view(torch.int32)
    _check(_lib.load().mm_ce_loss(logits.data_ptr(), labels.data_ptr(), B, T, V, acc.data_ptr(), cnt.data_ptr(),
                                  _stream()), "mm_ce_loss")
    return acc[0] / cnt[0].to(torch.float32)


# ---------------------------------------------------------------------------------------------------- training step
def gemm_dx(dy: torch.Tensor, w: torch.Tensor, out: Optional[torch.Tensor] = None, accumulate: bool = False) -> torch.Tensor:
    """Input gradient of y = x @ w.T:  dx (M, K) = dy (M, N) @ w (N, K) — w is read as an MN-major B operand in place."""
    _cuda(dy, ACT(), "dy"); _cuda(w, ACT(), "w")
    M, N = dy.shape
    K = w.shape[1]
    assert w.shape[0] == N and dy.stride(1) == 1 and w.stride(1) == 1
    if out is None:
        assert not accumulate
        out = torch.empty((M, K), device=dy.device, dtype=ACT())
    kw = dict(residual=out.data_ptr(), ldr=out.stride(0)) if accumulate else {}
    gemm_raw(M=M, N=K, K=N, A=dy.data_ptr(), lda=dy.stride(0), B=w.data_ptr(), ldb=w.stride(0), b_mn_major=True,
             Cout=out.data_ptr(), ldc=out.stride(0), **kw)
    return out


def gemm_dw(dy: torch.Tensor, x: torch.Tensor, out: torch.Tensor, accumulate: bool) -> torch.Tensor:
    """Weight gradient of y = x @ w.T:  dw (N, K) (+)= dy (M, N).T @ x (M, K) — both activations are read as stored
    (MN-major A and B operands), no transposes."""
    _cuda(dy, ACT(), "dy"); _cuda(x, ACT(), "x"); _cuda(out, ACT(), "dw")
    M, N = dy.shape
    K = x.shape[1]
    assert x.shape[0] == M and out.shape == (N, K) and dy.stride(1) == 1 and x.stride(1) == 1 and out.stride(1) == 1
    kw = dict(residual=out.data_ptr(), ldr=out.stride(0)) if accumulate else {}
    gemm_raw(M=N, N=K, K=M, A=dy.data_ptr(), lda=dy.stride(0), a_mn_major=True, B=x.data_ptr(), ldb=x.stride(0),
             b_mn_major=True, Cout=out.data_ptr(), ldc=out.stride(0), **kw)
    return out


def rmsnorm_bwd(dy: torch.Tensor, x: torch.Tensor, rstd: torch.Tensor, g: torch.Tensor, dres: Optional[torch.Tensor],
                dg: Optional[torch.Tensor]) -> torch.Tensor:
    """dx of y = x * rstd * g (+ dres); dg (fp32, cols) is accumulated in place."""
    _cuda(dy, ACT(), "dy"); _cuda(x, ACT(), "x"); _cuda(rstd, torch.float32, "rstd"); _cuda(g, ACT(), "g")
    assert dy.is_contiguous() and x.is_contiguous() and (dres is None or dres.is_contiguous())
    rows, cols = x.shape
    dx = torch.empty_like(x)
    lib = _lib.load()
    parts = None
    if dg is not None:  # per-CTA partial column sums, reduced in a fixed order (no atomics)
        with torch.cuda.device(x.device):
            parts = torch.empty((int(lib.mm_rmsnorm_bwd_parts(rows)), cols), device=x.device, dtype=torch.float32)
    _check(lib.mm_rmsnorm_bwd(dy.data_ptr(), x.data_ptr(), rstd.data_ptr(), g.data_ptr(), _ptr(dres), dx.data_ptr(),
                              _ptr(dg), _ptr(parts), rows, cols, _stream()), "mm_rmsnorm_bwd")
    return dx


def swiglu_fwd(gate: torch.Tensor, up: torch.Tensor) -> torch.Tensor:
    _cuda(gate, ACT(), "gate"); _cuda(up, ACT(), "up")
    assert gate.is_contiguous() and up.is_contiguous() and gate.shape == up.shape
    h = torch.empty_like(gate)
    _check(_lib.load().mm_swiglu_fwd(gate.data_ptr(), up.data_ptr(), h.data_ptr(), gate.numel(), _stream()), "mm_swiglu_fwd")
    return h


def swiglu_bwd(dh: torch.Tensor, gate: torch.Tensor, up: torch.Tensor):
    _cuda(dh, ACT(), "dh")
    assert dh.is_contiguous() and gate.is_contiguous() and up.is_contiguous()
    dg, du = torch.empty_like(gate), torch.empty_like(up)
    _check(_lib.load().mm_swiglu_bwd(dh.data_ptr(), gate.data_ptr(), up.data_ptr(), dg.data_ptr(), du.data_ptr(), dh.numel(),
                                     _stream()), "mm_swiglu_bwd")
    return dg, du


def _drop_args(dropout):
    """dropout = None | (p, seed_dev int64 1-element CUDA tensor, stream id) -> (p, seed pointer, sid) for the C ABI."""
    if dropout is None:
        return 0.0, None, 0
    p, seed, sid = dropout
    if float(p) <= 0.0:
        return 0.0, None, 0
    assert seed.is_cuda and seed.dtype == torch.int64 and seed.numel() == 1
    return float(p), seed.data_ptr(), int(sid)


def dropout_mask(rows: int, cols: int, dropout, device) -> torch.Tensor:
    """fp32 (rows, cols) multipliers (0 or 1/(1-p)) the dropout kernels apply for this (seed, stream id): tests only."""
    p, seed, sid = _drop_args(dropout)
    out = torch.empty((rows, cols), device=device, dtype=torch.float32)
    _check(_lib.load().mm_dropout_mask(out.data_ptr(), cols, rows, cols, p, seed, sid, _stream()), "mm_dropout_mask")
    return out


def attention_train_fwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, scale: float, causal: bool = False,
                        key_mask: Optional[torch.Tensor] = None, dropout=None) -> torch.Tensor:
    """Training-mode forward of a DROPOUT attention (the flash kernel has no dropout): S = q k^T (fp32, batched tcgen05
    GEMM), Pd = dropout(softmax(scale S)) (one row-wise kernel, Philox mask), O = Pd v.  Same operand conventions as
    attention_bwd; returns O (B, Tq, H, hd) contiguous."""
    for n, t in (("q", q), ("k", k), ("v", v)):
        _cuda(t, ACT(), n)
        assert t.dim() == 4 and t.stride(3) == 1
    assert ACT() == torch.bfloat16, "the training step computes in bf16"
    B, Tq, H, hd = q.shape
    Tk = k.shape[1]
    dev = q.device
    Tp = (Tk + 7) // 8 * 8
    S = torch.empty((B, H, Tq, Tp), device=dev, dtype=torch.float32)
    gemm_raw(M=Tq, N=Tk, K=hd, batch=H, batch2=B, A=q.data_ptr(), lda=q.stride(1), a_bs=q.stride(2), a_bs2=q.stride(0),
             B=k.data_ptr(), ldb=k.stride(1), b_bs=k.stride(2), b_bs2=k.stride(0), Cout=S.data_ptr(), ldc=Tp, c_bs=Tq * Tp,
             c_bs2=H * Tq * Tp, c_fp32=True)
    P = torch.empty((B, H, Tq, Tp), device=dev, dtype=ACT())
    if key_mask is not None:
        _cuda(key_mask, torch.int32, "key_mask")
    pd, seed, sid = _drop_args(dropout)
    _check(_lib.load().mm_attn_softmax_fwd(S.data_ptr(), P.data_ptr(), B, H, Tq, Tk, Tp, float(scale), int(causal),
                                           _ptr(key_mask), pd, seed, sid, _stream()), "mm_attn_softmax_fwd")
    del S
    o = torch.empty((B, Tq, H, hd), device=dev, dtype=ACT())
    gemm_raw(M=Tq, N=hd, K=Tk, batch=H, batch2=B, A=P.data_ptr(), lda=Tp, a_bs=Tq * Tp, a_bs2=H * Tq * Tp,
             B=v.data_ptr(), ldb=v.stride(1), b_bs=v.stride(2), b_bs2=v.stride(0), b_mn_major=True, Cout=o.data_ptr(),
             ldc=o.stride(1), c_bs=o.stride(2), c_bs2=o.stride(0))
    return o


def attention_bwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, do: torch.Tensor, *, scale: float, causal: bool,
                  key_mask: Optional[torch.Tensor] = None, dropout=None):
    """Backward of mm_attn_fwd composed from tcgen05 GEMMs: S = q k^T and dP = dO v^T (fp32, batched over (b, h)), one
    row-wise softmax-backward kernel (P, dS in bf16), then dV = P^T dO, dK = dS^T q (MN-major A), dQ = dS k.
    q / do (B, Tq, H, hd), k / v (B, Tk, H, hd): bf16 views with unit head-dim stride.  Returns contiguous dq, dk, dv.
    dropout = (p, seed_dev, sid): backward of attention_train_fwd with the same mask (regenerated, not stored)."""
    for n, t in (("q", q), ("k", k), ("v", v), ("do", do)):
        _cuda(t, ACT(), n)
        assert t.dim() == 4 and t.stride(3) == 1
    B, Tq, H, hd = q.shape
    Tk = k.shape[1]
    dev = q.device
    Tp = (Tk + 7) // 8 * 8
    S = torch.empty((B, H, Tq, Tp), device=dev, dtype=torch.float32)
    dP = torch.empty((B, H, Tq, Tp), device=dev, dtype=torch.float32)

    def bat(t):  # (lda, head stride, sample stride) of a (B, T, H, hd) view
        return dict(ld=t.stride(1), bs=t.stride(2), bs2=t.stride(0))

    def scores(a, b, out):
        sa, sb = bat(a), bat(b)
        gemm_raw(M=Tq, N=Tk, K=hd, batch=H, batch2=B, A=a.data_ptr(), lda=sa["ld"], a_bs=sa["bs"], a_bs2=sa["bs2"],
                 B=b.data_ptr(), ldb=sb["ld"], b_bs=sb["bs"], b_bs2=sb["bs2"], Cout=out.data_ptr(), ldc=Tp, c_bs=Tq * Tp,
                 c_bs2=H * Tq * Tp, c_fp32=True)

    scores(q, k, S)
    scores(do, v, dP)
    P = torch.empty((B, H, Tq, Tp), device=dev, dtype=ACT())
    dS = torch.empty((B, H, Tq, Tp), device=dev, dtype=ACT())
    if key_mask is not None:
        _cuda(key_mask, torch.int32, "key_mask")
    pd, seed, sid = _drop_args(dropout)
    _check(_lib.load().mm_attn_softmax_bwd(S.data_ptr(), dP.data_ptr(), P.data_ptr(), dS.data_ptr(), B, H, Tq, Tk, Tp,
                                           float(scale), int(causal), _ptr(key_mask), pd, seed, sid, _stream()),
           "mm_attn_softmax_bwd")
    del S, dP
    dq = torch.empty((B, Tq, H, hd), device=dev, dtype=ACT())
    dk = torch.empty((B, Tk, H, hd), device=dev, dtype=ACT())
    dv = torch.empty((B, Tk, H, hd), device=dev, dtype=ACT())

    def pt_x(p_, x_, out):  # out_bh (Tk, hd) = p_bh^T (Tk x Tq) @ x_bh (Tq, hd)
        sx, so = bat(x_), bat(out)
        gemm_raw(M=Tk, N=hd, K=Tq, batch=H, batch2=B, A=p_.data_ptr(), lda=Tp, a_bs=Tq * Tp, a_bs2=H * Tq * Tp,
                 a_mn_major=True, B=x_.data_ptr(), ldb=sx["ld"], b_bs=sx["bs"], b_bs2=sx["bs2"], b_mn_major=True,
                 Cout=out.data_ptr(), ldc=so["ld"], c_bs=so["bs"], c_bs2=so["bs2"])

    pt_x(P, do, dv)
    pt_x(dS, q, dk)
    sk, so = bat(k), bat(dq)
    gemm_raw(M=Tq, N=hd, K=Tk, batch=H, batch2=B, A=dS.data_ptr(), lda=Tp, a_bs=Tq * Tp, a_bs2=H * Tq * Tp,
             B=k.data_ptr(), ldb=sk["ld"], b_bs=sk["bs"], b_bs2=sk["bs2"], b_mn_major=True, Cout=dq.data_ptr(),
             ldc=so["ld"], c_bs=so["bs"], c_bs2=so["bs2"])
    return dq, dk, dv


def ce_loss_with_count(logits: torch.Tensor, labels: torch.Tensor):
    """mm_ce_loss -> (loss fp32 scalar tensor, n_valid int32 1-element tensor)."""
    _cuda(logits, ACT(), "logits"); _cuda(labels, torch.int64, "labels")
    assert logits.is_contiguous() and labels.is_contiguous()
    B, T, V = logits.shape
    acc = torch.zeros((2,), device=logits.device, dtype=torch.float32)
    cnt = acc[1:].view(torch.int32)
    _check(_lib.load().mm_ce_loss(logits.data_ptr(), labels.data_ptr(), B, T, V, acc.data_ptr(), cnt.data_ptr(),
                                  _stream()), "mm_ce_loss")
    return acc[0] / cnt[0].to(torch.float32), cnt


def ce_bwd(logits: torch.Tensor, labels: torch.Tensor, n_valid: torch.Tensor, grad_scale=1.0) -> torch.Tensor:
    """d loss / d logits, written IN PLACE over the bf16 logits.  grad_scale: python float or a device fp32 scalar tensor
    (the upstream gradient of the loss, read by the kernel — no host sync, CUDA-graph capturable)."""
    B, T, V = logits.shape
    gs_dev = None
    if isinstance(grad_scale, torch.Tensor):
        gs_dev = _cuda(grad_scale.reshape(1).to(torch.float32), torch.float32, "grad_scale")
        grad_scale = 1.0
    _check(_lib.load().mm_ce_bwd(logits.data_ptr(), labels.data_ptr(), logits.data_ptr(), B, T, V, n_valid.data_ptr(),
                                 float(grad_scale), _ptr(gs_dev), _stream()), "mm_ce_bwd")
    return logits


def embed_scatter_add(dx: torch.Tensor, ids: torch.Tensor, dtable: torch.Tensor) -> None:
    """dtable[ids[i]] += dx[i] for bf16 rows dx (n, dim) with unit inner stride."""
    _cuda(dx, ACT(), "dx"); _cuda(dtable, ACT(), "dtable")
    ids64 = ids.reshape(-1).to(torch.int64).contiguous()  # (a strided 1-D view survives reshape(-1))
    assert dx.dim() == 2 and dx.stride(1) == 1 and dx.shape[0] == ids64.numel() and dtable.is_contiguous()
    _check(_lib.load().mm_embed_scatter_add(dx.data_ptr(), dx.stride(0), ids64.data_ptr(), ids64.numel(), dx.shape[1],
                                            dtable.shape[0], dtable.data_ptr(), _stream()), "mm_embed_scatter_add")


def colsum(x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    _cuda(x, ACT(), "x"); _cuda(out, torch.float32, "out")
    assert x.dim() == 2 and x.stride(1) == 1 and out.numel() == x.shape[1]
    _check(_lib.load().mm_colsum(x.data_ptr(), x.stride(0), x.shape[0], x.shape[1], out.data_ptr(), _stream()), "mm_colsum")
    return out


def adamw(p: torch.Tensor, g: torch.Tensor, master: torch.Tensor, m: torch.Tensor, v: torch.Tensor, *, lr: float,
          beta1: float, beta2: float, eps: float, weight_decay: float, step: int, grad_scale: float = 1.0,
          step_dev: Optional[torch.Tensor] = None) -> None:
    _cuda(p, ACT(), "p"); _cuda(g, ACT(), "g")
    assert p.is_contiguous() and g.is_contiguous() and master.numel() == p.numel()
    _check(_lib.load().mm_adamw(p.data_ptr(), g.data_ptr(), master.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(),
                                float(lr), float(beta1), float(beta2), float(eps), float(weight_decay), int(step),
                                _ptr(step_dev), float(grad_scale), _stream()), "mm_adamw")


# mm_opt_state (include/macaw_b200.h) as 8 int32 words; float fields are read through .view(torch.float32)
OPT_STEP, OPT_SKIPPED, OPT_LR, OPT_CLIP_COEF, OPT_GRAD_NORM, OPT_FINITE, OPT_APPLY, OPT_ARRIVED = range(8)
SCHEDULES = {"constant": 0, "constant_with_warmup": 1, "linear": 2, "cosine": 3}
GRAD_NORM_PARTS = 1024  # MM_GRAD_NORM_PARTS


def opt_state(device) -> torch.Tensor:
    """A fresh mm_opt_state: step 0, nothing skipped, clip_coef 1, finite."""
    st = torch.zeros((8,), dtype=torch.int32)
    st.view(torch.float32)[OPT_CLIP_COEF] = 1.0
    st[OPT_FINITE] = 1
    return st.to(device)


def grad_table(grads) -> torch.Tensor:
    """Device int64 (n, 2) table of (address, numel) of contiguous bf16 gradients (the input of grad_norm)."""
    rows = []
    for g in grads:
        _cuda(g, _BF16, "gradient")
        if not g.is_contiguous():
            raise RuntimeError("macaw_b200: grad_norm needs contiguous gradients")
        rows.append((g.data_ptr(), g.numel()))
    return torch.tensor(rows, dtype=torch.int64).reshape(-1, 2).to(torch.cuda.current_device())


def grad_norm(table: Optional[torch.Tensor], state: torch.Tensor, partials: torch.Tensor, *, max_norm: float = 0.0,
              skip_nonfinite: bool = False, base_lr: float = 0.0, schedule: str = "constant", warmup_steps: int = 0,
              total_steps: int = 0) -> None:
    """mm_grad_norm: global L2 norm of the gradients in `table` (None / empty: no pass) into the optimizer state, then the
    step's clip coefficient, step count and learning rate (see include/macaw_b200.h)."""
    _cuda(state, torch.int32, "state"); _cuda(partials, torch.float64, "partials")
    assert state.numel() == 8 and partials.numel() >= GRAD_NORM_PARTS
    n = 0 if table is None else table.shape[0]
    if n:
        _cuda(table, torch.int64, "table")
        assert table.is_contiguous() and table.shape[1] == 2
    _check(_lib.load().mm_grad_norm(_ptr(table) if n else None, n, partials.data_ptr(), state.data_ptr(), float(max_norm),
                                    int(bool(skip_nonfinite)), float(base_lr), SCHEDULES[schedule], int(warmup_steps),
                                    int(total_steps), _stream()), "mm_grad_norm")


def adamw_sched(p: torch.Tensor, g: torch.Tensor, master: torch.Tensor, m: torch.Tensor, v: torch.Tensor, *, beta1: float,
                beta2: float, eps: float, weight_decay: float, state: torch.Tensor) -> None:
    """mm_adamw_sched: AdamW with lr, gradient multiplier, step and skip flag read from the device optimizer state."""
    _cuda(p, ACT(), "p"); _cuda(g, ACT(), "g"); _cuda(state, torch.int32, "state")
    assert p.is_contiguous() and g.is_contiguous() and master.numel() == p.numel() and g.numel() == p.numel()
    _check(_lib.load().mm_adamw_sched(p.data_ptr(), g.data_ptr(), master.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(),
                                      float(beta1), float(beta2), float(eps), float(weight_decay), state.data_ptr(),
                                      _stream()), "mm_adamw_sched")


def cast_bf16(x: torch.Tensor) -> torch.Tensor:
    """fp16 contiguous tensor -> bf16 copy (mm_cast_f16_bf16): the alignment backward runs in bf16 (gradient range)."""
    _cuda(x, _F16, "x")
    assert x.is_contiguous()
    cols = x.shape[-1]
    rows = x.numel() // cols
    y = torch.empty(x.shape, device=x.device, dtype=torch.bfloat16)
    _check(_lib.load().mm_cast_f16_bf16(x.data_ptr(), cols, y.data_ptr(), cols, rows, cols, _stream()), "mm_cast_f16_bf16")
    return y


def align_dropout_fwd(P_unnorm: torch.Tensor, inv_l: torch.Tensor, pe: torch.Tensor, V: int, dropout):
    """Training-mode dropout of the alignment probabilities -> (Pm fp16 (R, ldp) kept entries, rs (R,) = (1/l)/(1-p),
    p_sum_real_d (R,), p_extra_d (R,)); see mm_align_dropout_fwd."""
    _cuda(P_unnorm, _F16, "P")
    R, ldp = P_unnorm.shape
    dev = P_unnorm.device
    Pm = torch.empty_like(P_unnorm)
    rs, psum_d, pext_d = (torch.empty((R,), device=dev, dtype=torch.float32) for _ in range(3))
    pd, seed, sid = _drop_args(dropout)
    _check(_lib.load().mm_align_dropout_fwd(P_unnorm.data_ptr(), Pm.data_ptr(), ldp, inv_l.data_ptr(), pe.data_ptr(),
                                            rs.data_ptr(), psum_d.data_ptr(), pext_d.data_ptr(), R, V, pd, seed, sid,
                                            _stream()), "mm_align_dropout_fwd")
    return Pm, rs, psum_d, pext_d


def align_softmax_bwd(G: torch.Tensor, P_unnorm: torch.Tensor, inv_l: torch.Tensor, dpsr: torch.Tensor, pe: torch.Tensor,
                      dpe: torch.Tensor, gscale: float, V: int, dropout=None):
    """-> (Pd bf16 (R, ldp), dS bf16 (R, ldp), dstats fp32 (2, R)); see mm_align_softmax_bwd."""
    _cuda(G, torch.float32, "G"); _cuda(P_unnorm, _F16, "P")
    R, ldp = P_unnorm.shape
    assert G.shape[0] == R and G.stride(1) == 1 and P_unnorm.stride(1) == 1
    for t in (inv_l, dpsr, pe, dpe):
        assert t.dtype == torch.float32 and t.is_contiguous() and t.numel() == R
    P = torch.empty((R, ldp), device=G.device, dtype=ACT())
    dS = torch.empty((R, ldp), device=G.device, dtype=ACT())
    dstats = torch.empty((2, R), device=G.device, dtype=torch.float32)
    pd, seed, sid = _drop_args(dropout)
    _check(_lib.load().mm_align_softmax_bwd(G.data_ptr(), G.stride(0), P_unnorm.data_ptr(), ldp, inv_l.data_ptr(), dpsr.data_ptr(),
                                            pe.data_ptr(), dpe.data_ptr(), float(gscale), P.data_ptr(), dS.data_ptr(), ldp,
                                            dstats.data_ptr(), R, V, pd, seed, sid, _stream()), "mm_align_softmax_bwd")
    return P, dS, dstats


def head_weighted_colsum(x: torch.Tensor, w: torch.Tensor, head_dim: int, out: torch.Tensor) -> torch.Tensor:
    """out[h*hd + d] += sum_n w[h, n] * x[n, h*hd + d]; x (Nq, E) bf16 / fp16, w (H*Nq,) fp32 contiguous, out fp32 (E,)."""
    _cuda(x, None, "x"); _cuda(w, torch.float32, "w"); _cuda(out, torch.float32, "out")
    assert x.dtype in _16BIT and x.stride(1) == 1 and w.is_contiguous()
    Nq, E = x.shape
    assert w.numel() == (E // head_dim) * Nq and out.numel() == E
    _check(_lib.load().mm_head_weighted_colsum(x.data_ptr(), x.stride(0), int(x.dtype == _F16), w.data_ptr(), 1, Nq, E,
                                               head_dim, out.data_ptr(), _stream()), "mm_head_weighted_colsum")
    return out


def window_gather_add(dwin: torch.Tensor, B: int, N: int, C: int, Lq: int, kk: int, ss: int) -> torch.Tensor:
    """Conv1d data gradient: dwin (B*Lq, kk*C) bf16 -> dfeats (B, N, C) bf16 (mm_window_gather_add)."""
    _cuda(dwin, torch.bfloat16, "dwin")
    assert dwin.is_contiguous() and dwin.shape == (B * Lq, kk * C)
    out = torch.empty((B, N, C), device=dwin.device, dtype=torch.bfloat16)
    _check(_lib.load().mm_window_gather_add(dwin.data_ptr(), B, N, C, Lq, kk, ss, out.data_ptr(), _stream()),
           "mm_window_gather_add")
    return out
