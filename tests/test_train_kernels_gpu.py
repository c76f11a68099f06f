"""The kernels of the training step one by one, at the real model's shapes, against fp64 autograd of the FORWARD op
they differentiate (never a restatement of the kernel's own backward formula), plus one real-width gradient test of the
alignment + video-long backward through `model(inputs).loss.backward()`.

Conventions:
  * references run in fp64 (on the GPU: fp64 matmuls never use TF32) on the same 16-bit tensors the kernel reads;
  * errors are norm-wise relative; every test prints its measured errors beside its bars;
  * bars are built from the storage format of the result and of the intermediates: one bf16 rounding costs about
    BF16 = 2e-3 norm-wise, one fp16 rounding FP16 = 2.5e-4, fp32 outputs are held much tighter; a bar is the sum of
    the roundings on the path (independent errors add in quadrature, so the sum leaves headroom without being loose);
  * every test starts from poisoned scratch memory (a large block filled with 0xFF bytes, NaN in every float format,
    then freed), and the padding columns of the buffers a test allocates itself are NaN: a kernel or GEMM that reads an
    element it should not fails on NaN instead of passing on zeros left behind by an earlier test;
  * dropout masks come from `ops.dropout_mask` with the same (p, seed, stream id), which tests/test_train_gpu.py pins
    bit-exact to the numpy Philox restatement.
"""
import math
import time

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"
BF16 = 2e-3    # one bf16 rounding of a result, norm-wise
FP16 = 2.5e-4  # one fp16 rounding of a result, norm-wise
P_DROP = 0.1   # the MHAs' attention dropout (nn.MultiheadAttention(dropout=0.1))


def _ops():
    from macaw_llm_b200 import ops

    return ops


def rel(a, b) -> float:
    a, b = a.detach().double(), b.detach().double().to(a.device)
    return float((a - b).norm() / (b.norm() + 1e-300))


def _gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def _seed_dev(value=0x5EED0123):
    return torch.tensor([value], dtype=torch.int64, device=DEV)


@pytest.fixture(autouse=True)
def _poisoned_scratch():
    """Hand every test NaN-filled memory from the caching allocator: release what is cached, then fill and free one
    large block (large pool) and a set of 1 MiB blocks (small pool)."""
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    big = torch.empty(min(16 << 30, free // 2), dtype=torch.uint8, device=DEV)
    big.fill_(0xFF)
    small = [torch.empty(1 << 20, dtype=torch.uint8, device=DEV).fill_(0xFF) for _ in range(64)]
    torch.cuda.synchronize()
    del big, small
    yield


# ------------------------------------------------------------------------------------------------ alignment softmax
# (R, V, E, kind).  R = 16 heads x 13 query rows (ragged), the real table (V = 32000) and the resized one (V = 32007:
# V % 4 = 3, so column V -- the bias_k key -- is word 3 of its Philox group and Vp = 32008), the small odd table, the
# overflow case of test_align_fused (real scores far above the synthetic keys -> exact-max re-run of phase 1) and the
# case where all mass sits on the synthetic keys (every real P' underflows to 0).
ALIGN_CASES = [
    (16 * 13, 32000, 4096, "real"),
    (16 * 13, 32007, 4096, "resized"),
    (300, 519, 256, "small"),
    (130, 2048, 256, "overflow"),
    (64, 2048, 256, "synthetic"),
]


def _align_inputs(R, V, E, kind):
    """table16 (V, E) fp16 (exact copy of a bf16 table), qt (R, E) fp16, stats (R, 2) fp32 = [row bias, extra score] and
    the fp64 real scores S = qt . table^T (without the row bias)."""
    g = _gen(R * 7 + V)
    table16 = (torch.randn(V, E, generator=g) * 0.5).to(torch.bfloat16).to(torch.float16).to(DEV)
    qs = 40.0 if kind == "overflow" else 1.0
    qt = (torch.randn(R, E, generator=g) * (qs * 2.0 / math.sqrt(E))).to(torch.float16).to(DEV)
    S = qt.double() @ table16.double().t()
    rb = torch.randn(R, generator=g, dtype=torch.float64).to(DEV)
    noise = torch.randn(R, generator=g, dtype=torch.float64).to(DEV)
    if kind == "synthetic":
        rb = torch.full_like(rb, -60.0)  # every real score ~60 nats below the zero key
        extra = noise
    elif kind == "overflow":
        # real maxima ~12 nats above the bias_k key (> 2^15 in P' -> flag -> exact-max re-run); p_extra stays ~1e-5
        extra = (S + rb[:, None]).max(1).values - 12.0 + 0.3 * noise
    else:
        # the bias_k key carries a few percent of the mass (p_extra ~ 0.01 .. 0.3), so its terms of D and of dstats[1]
        # are far above the rounding noise of the real keys
        extra = torch.logsumexp(S + rb[:, None], 1) - 3.0 + noise
    stats = torch.stack([rb, extra], 1).float().contiguous()
    return table16, qt, stats, S


def _align_softmax_ref(S, stats, mult):
    """fp64 softmax over the V + 2 keys [real ; bias_k ; zero] with the dropout multipliers `mult` (R, V + 1) applied
    to the real keys and the bias_k key -> (S leaf, extra leaf, Pd (R, V), pext_d (R,))."""
    R, V = S.shape
    S = S.clone().requires_grad_(True)
    ex = stats[:, 1].double().clone().requires_grad_(True)
    full = torch.cat([S + stats[:, :1].double(), ex[:, None], torch.zeros_like(ex)[:, None]], 1)
    p = torch.softmax(full, -1)
    return S, ex, p[:, :V] * mult[:, :V], p[:, V] * mult[:, V]


def _drop(dropout, sid=1):
    return (P_DROP, _seed_dev(), sid) if dropout else None


def _mult(R, V, drop):
    if drop is None:
        return torch.ones(R, V + 1, dtype=torch.float64, device=DEV)
    m = _ops().dropout_mask(R, V + 1, drop, DEV).double()
    assert abs(float((m != 0).double().mean()) - (1 - P_DROP)) < 0.01
    return m


def _nan_pad(t, V):
    if t.shape[1] > V:
        t[:, V:] = float("nan")
    return t


@pytest.mark.parametrize("dropout", [False, True])
@pytest.mark.parametrize("R,V,E,kind", ALIGN_CASES)
def test_align_softmax_bwd(R, V, E, kind, dropout):
    """mm_align_softmax_bwd on the P' / 1 / l that align_fused(keep=) saved, vs fp64 autograd of
    L = sum_v Pd_v (G_v + dpsr) + pext_d dpe,  Pd = m . softmax([q~ table^T + rb ; extra ; 0])[:V],  pext_d = m_V p_V,
    differentiated w.r.t. the real scores (dS; dstats[0] is their sum) and the extra score (dstats[1])."""
    ops = _ops()
    table16, qt, stats, S = _align_inputs(R, V, E, kind)
    keep = {}
    _, psum, pext = ops.align_fused(table16, qt, stats, keep=keep)
    Pp, inv_l = keep["P"], keep["inv_l"]
    Vp = Pp.shape[1]
    assert Vp == (V + 7) // 8 * 8 and inv_l.shape == (R,)
    _nan_pad(Pp, V)
    if kind == "overflow":  # the exact-max re-run ran: every row's largest P' is exactly 2^0
        assert torch.equal(Pp[:, :V].float().max(1).values, torch.ones(R, device=DEV))
    g = _gen(V + R)
    G = _nan_pad(torch.randn(R, Vp, generator=g).to(DEV), V)
    dpsr, dpe = torch.randn(R, generator=g).to(DEV), torch.randn(R, generator=g).to(DEV)
    drop = _drop(dropout)
    P, dS, dstats = ops.align_softmax_bwd(G, Pp, inv_l, dpsr, pext, dpe, 1.0, V, dropout=drop)
    torch.cuda.synchronize()

    mult = _mult(R, V, drop)
    Sl, ex, Pd, pext_d = _align_softmax_ref(S, stats, mult)
    L = (Pd * (G[:, :V].double() + dpsr.double()[:, None])).sum() + (pext_d * dpe.double()).sum()
    L.backward()
    dS_ref, ds1_ref = Sl.grad, ex.grad
    ds0_ref = dS_ref.sum(1)
    P, dS = P[:, :V], dS[:, :V]
    assert torch.isfinite(P).all() and torch.isfinite(dS).all() and torch.isfinite(dstats).all()
    e1 = rel(dstats[1], ds1_ref)
    tag = f"[align_softmax_bwd {kind} R{R} V{V}{' +dropout' if dropout else ''}]"
    if kind == "synthetic":
        # real probabilities ~e^-60: P' underflows to exactly 0 in fp16, so P, dS and their row sums are exact zeros
        assert float(Pd.detach().abs().max()) < 1e-20
        assert int(torch.count_nonzero(P)) == 0 and int(torch.count_nonzero(dS)) == 0
        assert int(torch.count_nonzero(dstats[0])) == 0
        print(f"\n{tag} P, dS, dstats[0] exact zeros; dstats[1] {e1:.2e} (bar {FP16:.1e})")
        assert e1 < FP16
        return
    eP, edS = rel(P, Pd), rel(dS, dS_ref)
    # dstats[0] = sum_v dS_v cancels (the softmax Jacobian's rows sum to ~0): measure its error against the norm of the
    # summands, sum_v |dS_v| per row
    e0 = float((dstats[0].double() - ds0_ref).norm() / dS_ref.abs().sum(1).norm())
    print(f"\n{tag} P {eP:.2e} dS {edS:.2e} (bars {FP16 + BF16:.2e}); dstats[0] {e0:.2e} (vs sum|dS|), "
          f"dstats[1] {e1:.2e} (bars {FP16:.1e})")
    # P, dS: the fp16 P' (one fp16 rounding) times fp32 math, stored once in bf16
    assert eP < FP16 + BF16 and edS < FP16 + BF16
    # dstats: fp32 outputs whose only 16-bit input is P'
    assert e0 < FP16 and e1 < FP16


@pytest.mark.parametrize("R,V,E,kind", ALIGN_CASES)
def test_align_dropout_fwd_and_masked_context(R, V, E, kind):
    """mm_align_dropout_fwd, then the masked P'.table GEMM with `row_scale` exactly as the training forward runs it
    (engine.py: ctx~ = rs . (Pm . table)), vs the fp64 dropped softmax."""
    ops = _ops()
    table16, qt, stats, S = _align_inputs(R, V, E, kind)
    keep = {}
    _, psum, pext = ops.align_fused(table16, qt, stats, keep=keep)
    Pp, inv_l = keep["P"], keep["inv_l"]
    Vp = Pp.shape[1]
    _nan_pad(Pp, V)
    drop = _drop(True, sid=2)
    Pm, rs, psum_d, pext_d = ops.align_dropout_fwd(Pp, inv_l, pext, V, drop)
    ctxt = torch.empty((R, E), device=DEV, dtype=torch.float16)
    ops.gemm_raw(M=R, N=E, K=V, A=Pm.data_ptr(), lda=Vp, B=table16.data_ptr(), ldb=table16.stride(0), b_mn_major=True,
                 Cout=ctxt.data_ptr(), ldc=E, row_scale=rs.data_ptr(), c_fp16=True, a_fp16=True, b_fp16=True)
    torch.cuda.synchronize()

    mult = _mult(R, V, drop)
    # bit-exact: kept entries are P' itself, dropped ones +0 (unscaled: the 1 / (1 - p) rides rs)
    want = torch.where(mult[:, :V] != 0, Pp[:, :V], torch.zeros((), dtype=torch.float16, device=DEV))
    assert torch.equal(Pm[:, :V].view(torch.int16), want.view(torch.int16))
    one = torch.ones((), dtype=torch.float32, device=DEV)
    assert torch.equal(rs, inv_l * (one / (one - torch.tensor(P_DROP, dtype=torch.float32, device=DEV))))
    with torch.no_grad():
        _, _, Pd, pext_ref = _align_softmax_ref(S, stats, mult)
        psum_ref = Pd.sum(1)
        ctx_ref = Pd @ table16.double()
        p_scaled = rs.double()[:, None] * Pp[:, :V].double()  # = P / (1 - p)
        p_scaled_ref = _align_softmax_ref(S, stats, torch.ones_like(mult))[2] / (1 - P_DROP)
    e_ext = rel(pext_d, pext_ref)
    tag = f"[align_dropout_fwd {kind} R{R} V{V}]"
    if kind == "synthetic":
        assert int(torch.count_nonzero(ctxt)) == 0 and int(torch.count_nonzero(psum_d)) == 0
        print(f"\n{tag} ctx~ and p_sum_real_d exact zeros; p_extra_d {e_ext:.2e} (bar {FP16:.1e})")
        assert e_ext < FP16
        return
    e_rs, e_sum, e_ctx = rel(p_scaled, p_scaled_ref), rel(psum_d, psum_ref), rel(ctxt, ctx_ref)
    print(f"\n{tag} rs.P' {e_rs:.2e} p_sum_real_d {e_sum:.2e} p_extra_d {e_ext:.2e} (bars {FP16:.1e}); "
          f"ctx~ {e_ctx:.2e} (bar {2 * FP16:.1e})")
    assert e_rs < FP16 and e_sum < FP16 and e_ext < FP16
    # ctx~: the fp16 P' and the fp16 output, two fp16 roundings
    assert e_ctx < 2 * FP16


# ------------------------------------------------------------------------------------------------ bias-gradient column sums
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("E,hd,Nq", [(4096, 256, 1), (4096, 256, 13), (4096, 256, 300), (768, 96, 300)])
def test_head_weighted_colsum(E, hd, Nq, dtype):
    """out[h*hd + d] += sum_n w[h, n] x[n, h*hd + d]: the bias gradients of b_k / b_v / bias_k / bias_v (16 heads of
    256; 8 heads of 96 is the video-long shape), accumulating into a non-zero fp32 `out`; x is a row-strided view."""
    ops = _ops()
    H = E // hd
    g = _gen(E + Nq)
    buf = torch.full((Nq, E + 64), float("nan"), dtype=dtype, device=DEV)
    x = buf[:, :E]
    x.copy_(torch.randn(Nq, E, generator=g).to(dtype))
    w = torch.randn(H * Nq, generator=g).to(DEV)
    out0 = torch.randn(E, generator=g).to(DEV)
    out = ops.head_weighted_colsum(x, w, hd, out0.clone())
    ref = out0.double() + torch.einsum("hn,nhd->hd", w.double().view(H, Nq), x.double().view(Nq, H, hd)).reshape(E)
    e = rel(out, ref)
    # fp32 accumulation of <= 300 products of 16-bit inputs: ~sqrt(300) * 2^-24 ~ 1e-6
    print(f"\n[head_weighted_colsum E{E} hd{hd} Nq{Nq} {str(dtype)[6:]}] {e:.2e} (bar 1e-5)")
    assert e < 1e-5


# ------------------------------------------------------------------------------------------------ fp16 -> bf16
@pytest.mark.parametrize("rows,cols", [(3, 5), (10007, 96)])
def test_cast_bf16_every_fp16_value(rows, cols):
    """mm_cast_f16_bf16 over every one of the 65536 fp16 bit patterns (subnormals, +-65504, values whose rounding
    carries into the exponent, ties, +-inf, NaN), tiled over a shape whose element count does not fill the kernel's
    grid-stride loop evenly; bit-exact against torch's conversion.  NaN payloads are not part of that contract (torch's
    CPU and GPU conversions differ there): a NaN must stay a NaN."""
    ops = _ops()
    n = rows * cols
    pat = torch.arange(n, dtype=torch.int64).remainder(65536).to(torch.int32)
    pat = torch.where(pat >= 32768, pat - 65536, pat).to(torch.int16)
    x16 = pat.view(torch.float16).view(rows, cols)
    y = ops.cast_bf16(x16.to(DEV)).cpu()
    want = x16.to(torch.bfloat16)
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(y), nan)
    assert torch.equal(y.view(torch.int16)[~nan], want.view(torch.int16)[~nan])
    if n >= 65536:
        spot = {0x7BFF: 65536.0, 0xFBFF: -65536.0, 0x3BFF: 1.0, 0x0001: 2.0 ** -24, 0x03FF: 1023 * 2.0 ** -24,
                0x7C00: math.inf, 0xFC00: -math.inf}
        for bits, val in spot.items():
            b = bits - 65536 if bits >= 32768 else bits
            got = y.view(-1)[int((pat == b).nonzero()[0])]
            assert float(got) == torch.tensor(val).to(torch.bfloat16).item(), (hex(bits), float(got))
    print(f"\n[cast_bf16 {rows}x{cols}] bit-exact over {min(n, 65536)} fp16 patterns")


# ------------------------------------------------------------------------------------------------ Conv1d data gradient
# (B, N, C, kernel, stride): the image / video / audio down-samplers, a stride > kernel case (tokens in no window) and
# shapes with (N - k) % s != 0 (trailing tokens in no window: image, video N = 4096, audio, the gap case).
WINDOW_CASES = [
    (2, 257, 768, 48, 36, "image"),
    (2, 1536, 768, 36, 30, "video 6 frames"),
    (2, 4096, 768, 36, 30, "video 16 frames"),
    (2, 1500, 512, 240, 220, "audio"),
    (2, 300, 64, 20, 30, "stride > kernel"),
]


@pytest.mark.parametrize("B,N,C,kk,ss,kind", WINDOW_CASES)
def test_window_gather_add(B, N, C, kk, ss, kind):
    """mm_window_gather_add (col2im) vs the input gradient of an fp64 F.conv1d: a grouped one-hot Conv1d is exactly the
    window extraction of the strided Conv1d's GEMM (y[b, c*k + j, l] = x[b, c, l*s + j]), so its data gradient given
    d(window) is the reference."""
    ops = _ops()
    Lq = (N - kk) // ss + 1
    dwin = torch.randn(B * Lq, kk * C, generator=_gen(N + kk)).to(torch.bfloat16).to(DEV)
    out = ops.window_gather_add(dwin, B, N, C, Lq, kk, ss)
    torch.cuda.synchronize()
    w = torch.zeros(C * kk, 1, kk, dtype=torch.float64, device=DEV)
    w[torch.arange(C * kk), 0, torch.arange(C * kk) % kk] = 1.0
    x = torch.zeros(B, C, N, dtype=torch.float64, device=DEV, requires_grad=True)
    y = F.conv1d(x, w, stride=ss, groups=C)
    assert y.shape == (B, C * kk, Lq)
    y.backward(dwin.double().view(B, Lq, kk, C).permute(0, 3, 2, 1).reshape(B, C * kk, Lq))
    ref = x.grad.permute(0, 2, 1)
    covered = torch.zeros(N, dtype=torch.bool)
    for l in range(Lq):
        covered[l * ss:l * ss + kk] = True
    if kind == "stride > kernel" or (N - kk) % ss != 0:
        assert not bool(covered.all())  # the case has tokens in no window
    e = rel(out, ref)
    # at most ceil(k / s) bf16 terms summed in fp32, stored once in bf16
    print(f"\n[window_gather_add {kind} N{N} C{C} k{kk} s{ss}] {e:.2e} (bar {BF16:.0e}); "
          f"{int((~covered).sum())} tokens in no window")
    assert e < BF16
    assert int(torch.count_nonzero(out[:, ~covered.to(DEV)])) == 0


# ------------------------------------------------------------------------------------------------ attention, training
def _strided_qkv(B, Tq, Tk, H, hd, seed):
    """q / k / v as strided views of ONE (B, Tk, 3 P) buffer, as Engine.encode_video_long builds them (q: the first Tq
    rows; the last key / value row is the zero key).  q, k ~ N(0, 1.4^2): scores of standard deviation 2, so the
    probabilities are far from uniform and every term of the softmax backward matters."""
    P = H * hd
    g = _gen(seed)
    qkv = torch.randn(B, Tk, 3, H, hd, generator=g)
    qkv[:, :, :2] *= 1.4
    qkv[:, Tk - 1, 1:] = 0.0
    qkv = qkv.view(B, Tk, 3 * P).to(torch.bfloat16).to(DEV)
    q5 = qkv.view(B, Tk, 3, H, hd)
    do = torch.randn(B, Tq, H, hd, generator=g).to(torch.bfloat16).to(DEV)
    return q5[:, :Tq, 0], q5[:, :, 1], q5[:, :, 2], do


def _attn_ref(q, k, v, do, scale, causal, key_mask, mult):
    """fp64 autograd of O = (m . softmax(scale q k^T + mask)) v; a query row with no visible key gives zeros (DESIGN §4)."""
    qf, kf, vf = (t.double().permute(0, 2, 1, 3).requires_grad_(True) for t in (q, k, v))
    Tq, Tk = q.shape[1], k.shape[1]
    s = (qf @ kf.transpose(-1, -2)) * scale
    vis = torch.ones(Tq, Tk, dtype=torch.bool, device=DEV)
    if causal:
        vis = torch.arange(Tk, device=DEV)[None, :] <= torch.arange(Tq, device=DEV)[:, None] + (Tk - Tq)
    vis = vis[None, None].expand(q.shape[0], 1, Tq, Tk)
    if key_mask is not None:
        vis = vis & (key_mask[:, None, None, :] != 0)
    any_vis = vis.any(-1, keepdim=True)
    p = torch.softmax(s.masked_fill(~(vis | ~any_vis), float("-inf")), -1) * any_vis
    if mult is not None:
        p = p * mult
    o = p @ vf
    o.backward(do.double().permute(0, 2, 1, 3))
    back = lambda t: t.permute(0, 2, 1, 3)  # noqa: E731
    return back(o.detach()), back(qf.grad), back(kf.grad), back(vf.grad), any_vis[:, 0, :, 0]


def _check_attention(B, H, hd, Tq, Tk, causal, key_mask, dropout, tag, seed):
    ops = _ops()
    q, k, v, do = _strided_qkv(B, Tq, Tk, H, hd, seed)
    scale = hd ** -0.5
    drop = (P_DROP, _seed_dev(0x0123456789), 4) if dropout else None
    o = ops.attention_train_fwd(q, k, v, scale=scale, causal=causal, key_mask=key_mask, dropout=drop)
    dq, dk, dv = ops.attention_bwd(q, k, v, do, scale=scale, causal=causal, key_mask=key_mask, dropout=drop)
    torch.cuda.synchronize()
    mult = ops.dropout_mask(B * H * Tq, Tk, drop, DEV).view(B, H, Tq, Tk).double() if dropout else None
    ro, rq, rk, rv, any_vis = _attn_ref(q, k, v, do, scale, causal, key_mask, mult)
    del mult
    e = dict(o=rel(o, ro), dq=rel(dq, rq), dk=rel(dk, rk), dv=rel(dv, rv))
    # P / dS stored once in bf16 (GEMM operands), the result stored once in bf16
    bar = 2 * BF16
    print(f"\n[{tag}] " + " ".join(f"{n} {x:.2e}" for n, x in e.items()) + f" (bar {bar:.0e})")
    assert max(e.values()) < bar, e
    if key_mask is not None:
        dead = ~any_vis  # (B, Tq): query rows that see only masked keys
        assert bool(dead.any())
        assert int(torch.count_nonzero(o[dead])) == 0 and int(torch.count_nonzero(dq[dead])) == 0
        padded = key_mask == 0
        assert int(torch.count_nonzero(dk[padded])) == 0 and int(torch.count_nonzero(dv[padded])) == 0


@pytest.mark.parametrize("dropout", [False, True])
@pytest.mark.parametrize("N", [1536, 4096])
def test_video_long_attention_train(N, dropout):
    """attention_train_fwd + attention_bwd at the video-long shape (B = 2, 8 heads of 96, Tq = N, Tk = N + 2; 6 frames
    -> N = 1536, 16 frames -> 4096): Tk > 1024 runs the CTA-per-row softmax kernels."""
    _check_attention(2, 8, 96, N, N + 2, False, None, dropout, f"video-long attention N{N}{' +dropout' if dropout else ''}",
                     seed=N)


@pytest.mark.parametrize("variant", ["full", "causal_leftpad_dropout"])
@pytest.mark.parametrize("Tk", [512, 513, 640, 641, 1024, 1025])
def test_attention_softmax_kernel_boundaries(Tk, variant):
    """Every softmax-backward instantiation at its boundary: Tk = 512 / 513 / 640 / 641 / 1024 select the warp kernels
    with 16 / 17 / 20 / 24 / 32 columns per lane, 1025 the first CTA-per-row shape.  Tq = Tk - 2.  `causal_leftpad_dropout`:
    causal with a left-padded key mask (the first query rows of each sample see only padding: their outputs and
    gradients must be zeros and no padded key may receive a gradient) and attention dropout."""
    B, H, hd, Tq = 2, 8, 96, Tk - 2
    km = None
    causal = dropout = variant != "full"
    if causal:
        km = torch.ones(B, Tk, dtype=torch.int32, device=DEV)
        km[0, :100] = 0
        km[1, :7] = 0
    _check_attention(B, H, hd, Tq, Tk, causal, km, dropout, f"attention softmax Tk{Tk} {variant}", seed=Tk)


# ------------------------------------------------------------------------------------------------ cross-entropy
@pytest.mark.parametrize("gs_kind", ["float", "device"])
@pytest.mark.parametrize("V", [32000, 32007])
def test_ce_loss_and_backward(V, gs_kind):
    """ce_loss_with_count / ce_bwd at the lm_head shape (B = 4, T = 528) vs fp64 autograd of the shifted cross entropy,
    with long runs of ignored labels (-100) and the upstream gradient as a Python float and as a device scalar."""
    ops = _ops()
    B, T = 4, 528
    g = _gen(V)
    logits = (torch.randn(B, T, V, generator=g) * 2.0).to(torch.bfloat16).to(DEV)
    labels = torch.randint(0, V, (B, T), generator=g)
    labels[0, :400] = -100
    labels[1, 100:300] = -100
    labels[2, :-5] = -100
    labels[3, 500:] = -100
    labels = labels.to(DEV)
    gs = 0.37 if gs_kind == "float" else torch.tensor(1.7, device=DEV)
    loss, cnt = ops.ce_loss_with_count(logits, labels)
    d = ops.ce_bwd(logits.clone(), labels, cnt, gs)
    torch.cuda.synchronize()
    lf = logits.double().requires_grad_(True)
    ref = F.cross_entropy(lf[:, :-1].reshape(-1, V), labels[:, 1:].reshape(-1), ignore_index=-100)
    (ref * float(gs)).backward()
    assert int(cnt) == int((labels[:, 1:] != -100).sum())
    el, ed = abs(float(loss) - float(ref)) / float(ref), rel(d, lf.grad)
    # loss: fp32 sum of ~1500 row losses, each good to ~1e-6; gradient: fp32 softmax stored once in bf16
    print(f"\n[ce V{V} grad_scale {gs_kind}] loss {el:.2e} (bar 3e-5) dlogits {ed:.2e} (bar {BF16:.0e})")
    assert el < 3e-5 and ed < BF16
    dead = torch.ones(B, T, dtype=torch.bool, device=DEV)
    dead[:, :-1] = labels[:, 1:] == -100
    assert int(torch.count_nonzero(d[dead])) == 0


# ------------------------------------------------------------------------------------------------ embedding gradient
def test_embed_scatter_add_repeated_ids():
    """embed_scatter_add at E = 4096, V = 32000 over 2 x 528 ids into a non-zero table gradient: one id ~300 times,
    the BOS id once per sample, ids of -1 (skipped), every other id once; dx is a row-strided view.

    Each add is a bf16 atomic: c adds round c partial sums whose norms grow like sqrt(j), so the rounding errors add up
    in quadrature to about BF16 * sqrt((c + 1) / 2) of the result -> bar(c) = BF16 * sqrt(c)."""
    ops = _ops()
    E, V, n = 4096, 32000, 2 * 528
    g = _gen(11)
    REP, BOS = 777, 1
    pool = torch.randperm(V - 3, generator=g)[: n + 1] + 3
    ids = pool[pool != REP][:n].clone()
    pos = torch.randperm(n, generator=g)
    ids[pos[:300]] = REP
    ids[pos[300:320]] = -1
    ids[0], ids[528] = BOS, BOS
    counts = torch.bincount(ids[ids >= 0], minlength=V)
    assert int(counts[REP]) == 300 - int((pos[:300] == 0).sum() + (pos[:300] == 528).sum()) and int(counts[BOS]) == 2
    buf = torch.full((n, E + 128), float("nan"), dtype=torch.bfloat16, device=DEV)
    dx = buf[:, :E]
    dx.copy_(torch.randn(n, E, generator=g).to(torch.bfloat16))
    init = torch.randn(V, E, generator=g).to(torch.bfloat16).to(DEV)
    table_g = init.clone()
    ops.embed_scatter_add(dx, ids.to(DEV), table_g)
    torch.cuda.synchronize()
    ref = init.double()
    keep = ids >= 0
    ref.index_add_(0, ids[keep].to(DEV), dx[keep.to(DEV)].double())
    counts = counts.to(DEV)
    assert torch.equal(table_g[counts == 0].view(torch.int16), init[counts == 0].view(torch.int16))
    once = counts == 1
    e1, e_bos, e_rep = rel(table_g[once], ref[once]), rel(table_g[BOS], ref[BOS]), rel(table_g[REP], ref[REP])
    c_rep = int(counts[REP])
    print(f"\n[embed_scatter_add] unrepeated rows {e1:.2e} (bar {BF16:.0e}); BOS x2 {e_bos:.2e} "
          f"(bar {BF16 * math.sqrt(2):.1e}); id x{c_rep} {e_rep:.2e} (bar {BF16 * math.sqrt(c_rep):.1e})")
    assert e1 < BF16 and e_bos < BF16 * math.sqrt(2) and e_rep < BF16 * math.sqrt(c_rep)


# ------------------------------------------------------------------------------------------------ AdamW
@pytest.mark.parametrize("n,offset", [(4097, 0), (7, 0), (4097, 1)])
def test_adamw_scalar_and_tail_paths(n, offset):
    """ops.adamw over 3 steps with a device step counter (the host `step` argument is left stale at 1) and
    grad_scale = 0.25, vs torch.optim.AdamW in fp64 on the hand-scaled gradient.  n = 4097: the vec8 kernel plus a
    one-element scalar tail; n = 7: scalar only; offset 1: views one element into larger buffers (not 16-byte aligned)
    -> the scalar kernel over everything.  Elements outside the views must not be touched."""
    ops = _ops()
    lr, betas, eps, wd, gs = 1e-2, (0.9, 0.95), 1e-8, 0.1, 0.25
    g = _gen(n + offset)
    w0 = torch.randn(n, generator=g).to(torch.bfloat16).double()  # bf16-representable start: p and master agree

    def view(dtype, fill):
        buf = torch.full((n + 16,), fill, dtype=dtype, device=DEV)
        return buf, buf[offset:offset + n]

    pb, p = view(torch.bfloat16, 7.0)
    gb, gv = view(torch.bfloat16, 7.0)
    wb, w = view(torch.float32, 7.0)
    mb, m = view(torch.float32, 0.0)
    vb, v = view(torch.float32, 0.0)
    p.copy_(w0.to(torch.bfloat16))
    w.copy_(w0.float())
    m.zero_()
    v.zero_()
    guards = [(t.clone(), t) for t in (pb, gb, wb, mb, vb)]
    ref = torch.nn.Parameter(w0.clone())
    opt = torch.optim.AdamW([ref], lr=lr, betas=betas, eps=eps, weight_decay=wd)
    step_dev = torch.zeros(1, dtype=torch.int32, device=DEV)
    for _ in range(3):
        gr = (torch.randn(n, generator=g) * 3.0).to(torch.bfloat16)
        gv.copy_(gr)
        guards[1] = (gb.clone(), gb)
        step_dev += 1
        ops.adamw(p, gv, w, m, v, lr=lr, beta1=betas[0], beta2=betas[1], eps=eps, weight_decay=wd, step=1,
                  grad_scale=gs, step_dev=step_dev)
        ref.grad = gr.double() * gs
        opt.step()
    torch.cuda.synchronize()
    st = opt.state[ref]
    ew, em, ev = rel(w, ref.detach()), rel(m, st["exp_avg"]), rel(v, st["exp_avg_sq"])
    eu = rel(w.double().cpu() - w0, ref.detach() - w0)
    # fp32 state: a few roundings of |w| ~ 1 per step (2^-24 each); the update itself (~lr) to ~1e-5
    print(f"\n[adamw n{n} offset{offset}] master {ew:.2e} m {em:.2e} v {ev:.2e} (bars 1e-6); update {eu:.2e} (bar 2e-5)")
    assert ew < 1e-6 and em < 1e-6 and ev < 1e-6 and eu < 2e-5
    assert torch.equal(p.view(torch.int16), w.to(torch.bfloat16).view(torch.int16))
    for before, after in guards:
        outside = torch.ones(n + 16, dtype=torch.bool, device=DEV)
        outside[offset:offset + n] = False
        assert torch.equal(after[outside], before[outside])


# ------------------------------------------------------------------------------------------------ real-width gradients
def _real_width_model():
    import bench
    from macaw_llm_b200.modeling import MM_LLMs, MM_LLMs_Config

    (clip, whisper, llama), hyper = bench.real_configs()  # n_frames = 6 -> video-long N = 1536, Tk = 1538
    clip.vision_config.num_hidden_layers = 1
    whisper.encoder_layers = 1
    llama.num_hidden_layers = 1
    cfg = MM_LLMs_Config(clip_config=clip, whisper_config=whisper, llm_config=llama, **hyper)
    return MM_LLMs.build_random(cfg, device="cuda", dtype=torch.bfloat16, seed=3), cfg


def test_real_width_alignment_and_video_long_gradients():
    """`model.train(); model(inputs).loss.backward()` at REAL widths (CLIP-L/14, LLaMA-7B width, V = 32000, 6 frames
    -> video-long Tk = 1538, alignment R = 16 heads x B x Lq; depths cut to one layer) vs autograd of the fp32 CPU oracle
    on the same bf16-rounded weights: every alignment parameter of image, audio and video, `video_long_self_attention.*`,
    the embedding table (gathered rows + keys / values of the alignment attention at V = 32000) and the LLaMA layer.
    Bar 2e-2 per tensor; the CPU oracle (it projects the 32000-row table once per modality) takes ~20 s."""
    from oracle import macaw_oracle as O

    model, cfg = _real_width_model()
    g = _gen(9)
    B, L, V = 2, 64, cfg.llm_config.vocab_size
    inp = dict(images=torch.randn(B, 3, 224, 224, generator=g).to(torch.bfloat16),
               audios=torch.randn(B, 80, 3000, generator=g).to(torch.bfloat16),
               videos=torch.randn(B, 6, 3, 224, 224, generator=g).to(torch.bfloat16),
               input_ids=torch.randint(3, V - 6, (B, L), generator=g), attention_mask=torch.ones(B, L, dtype=torch.int64))
    inp["input_ids"][:, 0] = 1
    labels = inp["input_ids"].clone()
    labels[:, :5] = -100
    inp["labels"] = labels
    for i, name in enumerate(("image", "audio", "video")):
        inp[f"{name}_starts"] = torch.full((B,), V - 6 + 2 * i, dtype=torch.int32)
        inp[f"{name}_ends"] = torch.full((B,), V - 5 + 2 * i, dtype=torch.int32)
    model.train()
    model.train_step.attention_dropout = False
    try:
        for p in model.parameters():
            p.grad = None
        out = model({k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in inp.items()})
        out.loss.backward()
        torch.cuda.synchronize()
    finally:
        model.train_step.attention_dropout = True
        model.eval()
    named = dict(model.named_parameters())
    grads = {k: p.grad.float().cpu() for k, p in named.items() if p.grad is not None}
    sd = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
    del model, out
    torch.cuda.empty_cache()
    t0 = time.time()
    loss_ref, grads_ref = O.full_loss_and_grads(
        {k: (v.float() if isinstance(v, torch.Tensor) and v.is_floating_point() else v) for k, v in inp.items()}, sd,
        O.hp_from_config(cfg))
    print(f"\n[real-width grads] CPU oracle {time.time() - t0:.0f} s; loss {float(loss_ref):.5f}")
    checked = [k for k in grads_ref if k.startswith(O.ALIGN_PREFIXES + ("llm.",))]
    assert "llm.model.embed_tokens.weight" in checked and "video_long_self_attention.bias_k" in checked
    assert "audio_align_attention.bias_k" in checked and len(checked) == len(grads_ref)
    errs = {}
    for k in checked:
        assert k in grads, k
        errs[k] = rel(grads[k], grads_ref[k])
    for k, e in sorted(errs.items(), key=lambda kv: -kv[1]):
        print(f"[real-width grads] {k:60s} {e:.3e}")
    bad = {k: e for k, e in errs.items() if not e < 2e-2}
    assert not bad, bad


def test_align_training_forward_needs_one_row_chunk():
    """A train-mode forward whose alignment block would be split into row chunks (engine.align_max_rows) raises
    NotImplementedError instead of training on partial activations, and leaves no gradient behind."""
    from tests import helpers as H
    from tests.golden import gen

    model, spec, hp, weights = H.build_tiny_model("cuda", torch.bfloat16)
    inp = gen.make_inputs(spec, 2, 16, seed=5, modalities=("image",), with_labels=True)
    inp = {k: (v.to(torch.bfloat16).cuda() if isinstance(v, torch.Tensor) and v.is_floating_point() else
               (v.cuda() if isinstance(v, torch.Tensor) else v)) for k, v in inp.items()}
    model.engine.align_max_rows = 1
    model.train()
    try:
        with pytest.raises(NotImplementedError):
            model(inp).loss.backward()
    finally:
        model.engine.align_max_rows = None
        model.eval()
    assert all(p.grad is None for p in model.parameters())
