// HBM-bound kernels of the training step (SURVEY.md §8f rank 1): the backward halves of RMSNorm / SwiGLU / softmax /
// cross-entropy, the embedding-gradient scatter and the fused AdamW update.  The contractions of the backward pass run on
// the tcgen05 GEMM (dX = dY W with an MN-major B operand, dW = dY^T X with MN-major A and B operands).
//
// Reference: autograd of the vendored LLaMA in /root/reference/modeling.py (LlamaRMSNorm :302-319, LlamaMLP :126-140,
// LlamaAttention :143-231, shifted CE :597-610) driven by llm_trainer.py:184-188 (compute_loss -> loss.backward()) and the
// optimizer of train.sh / configs/deepspeed_config.json (AdamW, fp32 master weights).
#include "common.cuh"
#include <cuda_fp16.h>
#include "ptx.cuh"
#include "philox.cuh"
#include "../../include/macaw_b200.h"

namespace mm {

#define ST(s) reinterpret_cast<cudaStream_t>(s)

__device__ __forceinline__ void unpack8f(const uint4& u, float (&f)[8]) {
  f[0] = bf16lo(u.x); f[1] = bf16hi(u.x); f[2] = bf16lo(u.y); f[3] = bf16hi(u.y);
  f[4] = bf16lo(u.z); f[5] = bf16hi(u.z); f[6] = bf16lo(u.w); f[7] = bf16hi(u.w);
}
__device__ __forceinline__ uint4 pack8f(const float (&f)[8]) {
  return make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// block-wide sum; `sh` holds >= 32 floats; every thread gets the result
__device__ __forceinline__ float block_sum(float v, float* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  float t = lane < nw ? sh[lane] : 0.f;
  return warp_sum(t);
}
__device__ __forceinline__ float block_max(float v, float* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  float t = lane < nw ? sh[lane] : -INFINITY;
  return warp_max(t);
}

// ------------------------------------------------------------------------------------------------ RMSNorm backward
// y = x * rstd * g.   dx = rstd * (g*dy) - rstd^3/cols * x * sum(g*dy*x) (+ dres);   dg += sum_rows dy * x * rstd.
// One CTA walks `rows_per_cta` rows; each thread owns a fixed set of 8-column chunks, so the dg partial sums stay in
// registers across the CTA's rows and cost one fp32 atomicAdd per column per CTA.
constexpr int kNormMaxChunks = 4;  // cols <= 256 threads * 8 * 4 = 8192
// NCH = 8-column chunks per thread (cols <= 256 * 8 * NCH): a template parameter so that the register budget follows the row
// width (the fixed 4-chunk version needed 162 registers -> ONE CTA per SM at cols = 4096: 55 us per launch).
template <int NCH>
__global__ void __launch_bounds__(256) rmsnorm_bwd_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ x,
                                                          const float* __restrict__ rstd, const bf16* __restrict__ g,
                                                          const bf16* __restrict__ dres, bf16* __restrict__ dx,
                                                          float* __restrict__ dg, float* __restrict__ dg_part, int rows,
                                                          int cols, int rows_per_cta) {
  __shared__ float sh[32];
  const int nch = cols >> 3;
  float gacc[NCH][8];
  float gv[NCH][8];
#pragma unroll
  for (int k = 0; k < NCH; ++k) {
    const int c = threadIdx.x + k * blockDim.x;
#pragma unroll
    for (int i = 0; i < 8; ++i) gacc[k][i] = 0.f;
    if (c < nch) unpack8f(__ldg(reinterpret_cast<const uint4*>(g + c * 8)), gv[k]);
  }
  const int r0 = blockIdx.x * rows_per_cta, r1 = min(rows, r0 + rows_per_cta);
  for (int r = r0; r < r1; ++r) {
    const float rs = rstd[r];
    float xv[NCH][8], tv[NCH][8];
    uint4 dru[NCH];  // the residual-branch gradient is fetched with the other operands, not after the reduction
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = threadIdx.x + k * blockDim.x;
      dru[k] = make_uint4(0u, 0u, 0u, 0u);
      if (c < nch && dres != nullptr) dru[k] = *reinterpret_cast<const uint4*>(dres + static_cast<long long>(r) * cols + c * 8);
    }
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = threadIdx.x + k * blockDim.x;
      if (c < nch) {
        float dv[8];
        unpack8f(*reinterpret_cast<const uint4*>(dy + static_cast<long long>(r) * cols + c * 8), dv);
        unpack8f(*reinterpret_cast<const uint4*>(x + static_cast<long long>(r) * cols + c * 8), xv[k]);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          tv[k][i] = dv[i] * gv[k][i];
          dot += tv[k][i] * xv[k][i];
          gacc[k][i] += dv[i] * xv[k][i] * rs;
        }
      }
    }
    dot = block_sum(dot, sh);
    const float coef = rs * rs * rs * dot / static_cast<float>(cols);
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = threadIdx.x + k * blockDim.x;
      if (c < nch) {
        float o[8];
        unpack8f(dru[k], o);  // zeros when there is no residual-branch gradient
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] += rs * tv[k][i] - coef * xv[k][i];
        *reinterpret_cast<uint4*>(dx + static_cast<long long>(r) * cols + c * 8) = pack8f(o);
      }
    }
  }
  if (dg_part != nullptr) {
    // deterministic two-stage reduction: this CTA's partial column sums, summed over CTAs by dg_reduce_kernel (the
    // atomics below put grid-size-way contention on every one of the `cols` addresses)
    float* dst = dg_part + static_cast<long long>(blockIdx.x) * cols;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = threadIdx.x + k * blockDim.x;
      if (c < nch) {
        reinterpret_cast<float4*>(dst + c * 8)[0] = make_float4(gacc[k][0], gacc[k][1], gacc[k][2], gacc[k][3]);
        reinterpret_cast<float4*>(dst + c * 8)[1] = make_float4(gacc[k][4], gacc[k][5], gacc[k][6], gacc[k][7]);
      }
    }
  } else if (dg != nullptr) {
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = threadIdx.x + k * blockDim.x;
      if (c < nch) {
#pragma unroll
        for (int i = 0; i < 8; ++i) atomicAdd(&dg[c * 8 + i], gacc[k][i]);
      }
    }
  }
}

// dg[c] += sum_b part[b][c] in a fixed order.  CTA = 32 columns x 8 slices of the partials (slice s takes b = s, s + 8, ...:
// 128-byte coalesced loads, 8x the loads in flight of a thread-per-column loop), slices combined through shared memory.
__global__ void __launch_bounds__(256) dg_reduce_kernel(const float* __restrict__ part, int n_parts, int cols,
                                                        float* __restrict__ dg) {
  __shared__ float sh[8][32];
  const int lane = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float a0 = 0.f, a1 = 0.f;
  if (c < cols) {
    int b = sl;
    for (; b + 8 < n_parts; b += 16) {
      a0 += part[static_cast<long long>(b) * cols + c];
      a1 += part[static_cast<long long>(b + 8) * cols + c];
    }
    if (b < n_parts) a0 += part[static_cast<long long>(b) * cols + c];
  }
  sh[sl][lane] = a0 + a1;
  __syncthreads();
  if (sl == 0 && c < cols) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sh[k][lane];
    dg[c] += t;
  }
}

// ------------------------------------------------------------------------------------------------ SwiGLU
__global__ void swiglu_fwd_kernel(const bf16* __restrict__ gate, const bf16* __restrict__ up, bf16* __restrict__ h,
                                  long long n8) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float a[8], b[8], o[8];
    unpack8f(reinterpret_cast<const uint4*>(gate)[i], a);
    unpack8f(reinterpret_cast<const uint4*>(up)[i], b);
#pragma unroll
    for (int k = 0; k < 8; ++k) o[k] = a[k] / (1.f + __expf(-a[k])) * b[k];
    reinterpret_cast<uint4*>(h)[i] = pack8f(o);
  }
}
// dgate = dh * up * d silu(gate),  dup = dh * silu(gate);   d silu(a) = s (1 + a (1 - s)),  s = sigmoid(a)
__global__ void swiglu_bwd_kernel(const bf16* __restrict__ dh, const bf16* __restrict__ gate, const bf16* __restrict__ up,
                                  bf16* __restrict__ dgate, bf16* __restrict__ dup, long long n8) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float d[8], a[8], b[8], og[8], ou[8];
    unpack8f(reinterpret_cast<const uint4*>(dh)[i], d);
    unpack8f(reinterpret_cast<const uint4*>(gate)[i], a);
    unpack8f(reinterpret_cast<const uint4*>(up)[i], b);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float s = 1.f / (1.f + __expf(-a[k]));
      ou[k] = d[k] * a[k] * s;
      og[k] = d[k] * b[k] * s * (1.f + a[k] * (1.f - s));
    }
    reinterpret_cast<uint4*>(dgate)[i] = pack8f(og);
    reinterpret_cast<uint4*>(dup)[i] = pack8f(ou);
  }
}

// ------------------------------------------------------------------------------------------------ attention softmax (training)
// One CTA per (b, h, query) row of the score matrices: S (pre-scale logits q.k) and dP = dO V^T, both fp32.
//   P = softmax(scale * S + mask),  Pd = m . P  (m: dropout multipliers, 0 or 1/(1-p); all ones when dropout is off),
//   dP <- m . dP,  D = sum_j P_j dP_j,  dS = scale * P (dP - D).
// Pd and dS are written as bf16 (A operands of dV = Pd^T dO, dK = dS^T Q, dQ = dS K).  Mask semantics match the forward
// kernel: key j visible to query i iff j <= i + (Tk - Tq) (causal) and key_mask[b][j] != 0; fully masked rows give zeros.
// Dropout element index: (row = blockIdx.x, col = j) of stream `sid` (philox.cuh).
__global__ void __launch_bounds__(256) attn_softmax_bwd_kernel(const float* __restrict__ S, const float* __restrict__ dP,
                                                               bf16* __restrict__ P, bf16* __restrict__ dS, int H, int Tq,
                                                               int Tk, long long ld, float scale, int causal,
                                                               const int* __restrict__ key_mask, float p_drop,
                                                               const unsigned long long* __restrict__ seed_dev, uint32_t sid) {
  __shared__ float sh[32];
  const long long row = blockIdx.x;
  const int i = static_cast<int>(row % Tq);
  const int b = static_cast<int>(row / (static_cast<long long>(Tq) * H));
  const float* s = S + row * ld;
  const float* dp = dP + row * ld;
  bf16* p = P + row * ld;
  bf16* ds = dS + row * ld;
  const int* km = key_mask ? key_mask + static_cast<long long>(b) * Tk : nullptr;
  const int lim = causal ? i + (Tk - Tq) : Tk - 1;
  const DropCfg dc = drop_cfg(p_drop, seed_dev, sid);
  const int n4 = (Tk + 3) >> 2;
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < Tk; j += blockDim.x) {
    const bool ok = j <= lim && (km == nullptr || km[j] != 0);
    if (ok) mx = fmaxf(mx, s[j] * scale);
  }
  mx = block_max(mx, sh);
  float sum = 0.f, dsum = 0.f;
  for (int j4 = threadIdx.x; j4 < n4; j4 += blockDim.x) {
    float m[4];
    drop_mult4(dc, static_cast<uint32_t>(row), static_cast<uint32_t>(j4), m);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = 4 * j4 + u;
      if (j >= Tk) break;
      const bool ok = j <= lim && (km == nullptr || km[j] != 0);
      const float e = ok ? __expf(s[j] * scale - mx) : 0.f;
      sum += e;
      dsum += e * m[u] * dp[j];
    }
  }
  sum = block_sum(sum, sh);
  dsum = block_sum(dsum, sh);
  const float inv = sum > 0.f ? 1.f / sum : 0.f;
  const float D = dsum * inv;
  for (int j4 = threadIdx.x; j4 < n4; j4 += blockDim.x) {
    float m[4];
    drop_mult4(dc, static_cast<uint32_t>(row), static_cast<uint32_t>(j4), m);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = 4 * j4 + u;
      if (j >= Tk) break;
      const bool ok = j <= lim && (km == nullptr || km[j] != 0);
      const float pj = ok ? __expf(s[j] * scale - mx) * inv : 0.f;
      p[j] = __float2bfloat16(pj * m[u]);
      ds[j] = __float2bfloat16(scale * pj * (m[u] * dp[j] - D));
    }
  }
}

// Same computation, ONE WARP per row with the row held in registers (Tk <= 32 * NV): both inputs are read once with every
// load in flight, the three reductions are shuffles, no __syncthreads.  Lane l owns columns l, l + 32, ... (coalesced).
// History (profiles/r2_ncu_softmax_bwd.txt): the block-per-row kernel above takes 377 us per LLaMA layer at T = 528; the
// first warp-per-row version (NV = 24, 126 registers -> 16 warps / SM) took 357 us at 14 % of the DRAM rate with
// long-scoreboard stalls: too few loads in flight.  Hence NV is matched to Tk (17 at T = 528), the visibility mask is one
// bit word instead of an array, and the register budget is capped so that 32 warps are resident.
template <int NV>
__global__ void __launch_bounds__(256, (NV <= 20 ? 4 : 2))
attn_softmax_bwd_warp_kernel(const float* __restrict__ S, const float* __restrict__ dP, bf16* __restrict__ P,
                             bf16* __restrict__ dS, long long rows, int H, int Tq, int Tk, long long ld, float scale,
                             int causal, const int* __restrict__ key_mask, float p_drop,
                             const unsigned long long* __restrict__ seed_dev, uint32_t sid) {
  const int lane = threadIdx.x & 31;
  const long long row = blockIdx.x * static_cast<long long>(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int i = static_cast<int>(row % Tq);
  const int b = static_cast<int>(row / (static_cast<long long>(Tq) * H));
  const float* s = S + row * ld;
  const float* dp = dP + row * ld;
  const int lim = causal ? min(Tk - 1, i + (Tk - Tq)) : Tk - 1;
  const DropCfg dc = drop_cfg(p_drop, seed_dev, sid);
  float sv[NV], dv[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int j = lane + 32 * k;
    sv[k] = j < Tk ? s[j] : 0.f;
  }
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int j = lane + 32 * k;
    dv[k] = j < Tk ? dp[j] : 0.f;
  }
  uint32_t okb = 0u;  // bit k: column lane + 32 k is visible
  if (key_mask != nullptr) {
    const int* km = key_mask + static_cast<long long>(b) * Tk;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int j = lane + 32 * k;
      if (j <= lim && km[j] != 0) okb |= 1u << k;
    }
  } else {
#pragma unroll
    for (int k = 0; k < NV; ++k)
      if (lane + 32 * k <= lim) okb |= 1u << k;
  }
  float mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    sv[k] *= scale;
    if (okb & (1u << k)) mx = fmaxf(mx, sv[k]);
  }
  mx = warp_max(mx);
  float sum = 0.f, dsum = 0.f;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const float e = (okb & (1u << k)) ? __expf(sv[k] - mx) : 0.f;
    if (dc.on) dv[k] *= drop_mult1(dc, static_cast<uint32_t>(row), static_cast<uint32_t>(lane + 32 * k));
    sv[k] = e;
    sum += e;
    dsum += e * dv[k];
  }
  sum = warp_sum(sum);
  dsum = warp_sum(dsum);
  const float inv = sum > 0.f ? 1.f / sum : 0.f;
  const float D = dsum * inv;
  bf16* p = P + row * ld;
  bf16* ds = dS + row * ld;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int j = lane + 32 * k;
    if (j < Tk) {
      const float pj = sv[k] * inv;
      const float mj = dc.on ? drop_mult1(dc, static_cast<uint32_t>(row), static_cast<uint32_t>(j)) : 1.0f;
      p[j] = __float2bfloat16(pj * mj);
      ds[j] = __float2bfloat16(scale * pj * (dv[k] - D));
    }
  }
}

// Forward half for the training step of a dropout attention (video_long_self_attention in train() mode): S fp32 ->
// Pd = dropout(softmax(scale * S + mask)) in bf16 (the A operand of O = Pd V); same row / mask / dropout conventions.
__global__ void __launch_bounds__(256) attn_softmax_fwd_kernel(const float* __restrict__ S, bf16* __restrict__ P, int H, int Tq,
                                                               int Tk, long long ld, float scale, int causal,
                                                               const int* __restrict__ key_mask, float p_drop,
                                                               const unsigned long long* __restrict__ seed_dev, uint32_t sid) {
  __shared__ float sh[32];
  const long long row = blockIdx.x;
  const int i = static_cast<int>(row % Tq);
  const int b = static_cast<int>(row / (static_cast<long long>(Tq) * H));
  const float* s = S + row * ld;
  bf16* p = P + row * ld;
  const int* km = key_mask ? key_mask + static_cast<long long>(b) * Tk : nullptr;
  const int lim = causal ? i + (Tk - Tq) : Tk - 1;
  const DropCfg dc = drop_cfg(p_drop, seed_dev, sid);
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < Tk; j += blockDim.x) {
    const bool ok = j <= lim && (km == nullptr || km[j] != 0);
    if (ok) mx = fmaxf(mx, s[j] * scale);
  }
  mx = block_max(mx, sh);
  float sum = 0.f;
  for (int j = threadIdx.x; j < Tk; j += blockDim.x) {
    const bool ok = j <= lim && (km == nullptr || km[j] != 0);
    sum += ok ? __expf(s[j] * scale - mx) : 0.f;
  }
  sum = block_sum(sum, sh);
  const float inv = sum > 0.f ? 1.f / sum : 0.f;
  const int n4 = (Tk + 3) >> 2;
  for (int j4 = threadIdx.x; j4 < n4; j4 += blockDim.x) {
    float m[4];
    drop_mult4(dc, static_cast<uint32_t>(row), static_cast<uint32_t>(j4), m);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = 4 * j4 + u;
      if (j >= Tk) break;
      const bool ok = j <= lim && (km == nullptr || km[j] != 0);
      p[j] = __float2bfloat16(ok ? __expf(s[j] * scale - mx) * inv * m[u] : 0.f);
    }
    // padding columns Tk .. ld-1 are never read (the consuming GEMM's K extent is Tk)
  }
}

// The dropout multipliers themselves (fp32, 0 or 1/(1-p)) for rows x cols of stream `sid`: test / debugging utility (the
// parity tests hand this mask to the autograd oracle).
__global__ void dropout_mask_kernel(float* __restrict__ out, long long ld, int rows, int cols, float p_drop,
                                    const unsigned long long* __restrict__ seed_dev, uint32_t sid) {
  const DropCfg dc = drop_cfg(p_drop, seed_dev, sid);
  const int n4 = (cols + 3) >> 2;
  const long long total = static_cast<long long>(rows) * n4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / n4), c4 = static_cast<int>(i % n4);
    float m[4];
    drop_mult4(dc, static_cast<uint32_t>(r), static_cast<uint32_t>(c4), m);
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (4 * c4 + u < cols) out[r * ld + 4 * c4 + u] = m[u];
  }
}

// ------------------------------------------------------------------------------------------------ cross-entropy backward
// Shifted CE of modeling.py:600-610: position t predicts labels[t+1].  dlogits[b,t,:] = (softmax(logits[b,t,:]) -
// onehot(labels[b,t+1])) * gscale / n_valid  when t < T-1 and the label is not -100, else 0.  In place is allowed.
__global__ void __launch_bounds__(512) ce_bwd_kernel(const bf16* __restrict__ logits, const long long* __restrict__ labels,
                                                     bf16* __restrict__ dlogits, int T, int V,
                                                     const int* __restrict__ n_valid, float gscale,
                                                     const float* __restrict__ gscale_dev) {
  __shared__ float sh[32];
  const long long row = blockIdx.x;  // b * T + t
  const int t = static_cast<int>(row % T);
  const bf16* x = logits + row * V;
  bf16* o = dlogits + row * V;
  long long lab = -100;
  if (t < T - 1) lab = labels[row + 1];
  if (lab < 0 || lab >= V) {
    for (int j = threadIdx.x; j < V; j += blockDim.x) o[j] = __float2bfloat16(0.f);
    return;
  }
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < V; j += blockDim.x) mx = fmaxf(mx, __bfloat162float(x[j]));
  mx = block_max(mx, sh);
  float sum = 0.f;
  for (int j = threadIdx.x; j < V; j += blockDim.x) sum += __expf(__bfloat162float(x[j]) - mx);
  sum = block_sum(sum, sh);
  const int nv = *n_valid;
  const float sc = gscale * (gscale_dev != nullptr ? *gscale_dev : 1.0f) / static_cast<float>(nv > 0 ? nv : 1);
  const float inv = 1.f / sum;
  for (int j = threadIdx.x; j < V; j += blockDim.x) {
    float pj = __expf(__bfloat162float(x[j]) - mx) * inv;
    if (j == lab) pj -= 1.f;
    o[j] = __float2bfloat16(pj * sc);
  }
}

// ------------------------------------------------------------------------------------------------ embedding gradient
// dtable[ids[i], :] += dx[i, :]  (bf16x2 atomics; rows with ids outside [0, vocab) are skipped)
__global__ void embed_scatter_add_kernel(const bf16* __restrict__ dx, long long ldx, const long long* __restrict__ ids,
                                         long long n, int dim, int vocab, bf16* __restrict__ dtable) {
  const int half_dim = dim >> 1;
  const long long total = n * half_dim;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / half_dim;
    const int c = static_cast<int>(i % half_dim);
    const long long id = ids[r];
    if (id < 0 || id >= vocab) continue;
    const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(dx + r * ldx + 2 * c);
    atomicAdd(reinterpret_cast<__nv_bfloat162*>(dtable + id * dim + 2 * c), v);
  }
}

// column sums of a bf16 (rows, cols) matrix into fp32 (bias gradients): out[c] += sum_r x[r, c]
__global__ void colsum_kernel(const bf16* __restrict__ x, long long ldx, int rows, int cols, float* __restrict__ out,
                              int rows_per_cta) {
  const int c = blockIdx.y * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const int r0 = blockIdx.x * rows_per_cta, r1 = min(rows, r0 + rows_per_cta);
  float acc = 0.f;
  for (int r = r0; r < r1; ++r) acc += __bfloat162float(x[static_cast<long long>(r) * ldx + c]);
  atomicAdd(&out[c], acc);
}

// ------------------------------------------------------------------------------------------------ AdamW
// Decoupled weight decay (Loshchilov & Hutter), fp32 master weights + moments, bf16 working copy:
//   m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;  w -= lr (m/bc1 / (sqrt(v/bc2) + eps) + wd w);  p = bf16(w)
// 8 elements per thread and iteration: one 128-bit gradient load, two 128-bit loads / stores per fp32 state tensor, one
// 128-bit parameter store (28 bytes of HBM traffic per parameter; the scalar kernel below reached 4.5 TB/s of it).
// kSched (mm_adamw_sched): lr, the gradient multiplier and the step come from the device optimizer state, and a skipped
// step returns before touching memory.
template <bool kSched>
__global__ void __launch_bounds__(256) adamw_vec8_kernel(bf16* __restrict__ p, const bf16* __restrict__ g, float* __restrict__ w,
                                                         float* __restrict__ m, float* __restrict__ v, long long n8, float lr,
                                                         float b1, float b2, float eps, float wd, float inv_bc1, float inv_bc2,
                                                         float gscale, const int* __restrict__ step_dev,
                                                         const mm_opt_state* __restrict__ st) {
  if constexpr (kSched) {
    if (!st->apply) return;
    lr = st->lr;
    gscale = st->clip_coef;
    step_dev = &st->step;
  }
  if (step_dev != nullptr) {
    const float t = static_cast<float>(*step_dev);
    inv_bc1 = 1.f / (1.f - powf(b1, t));
    inv_bc2 = 1.f / (1.f - powf(b2, t));
  }
  const float c1 = 1.f - b1, c2 = 1.f - b2;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint4 gu = __ldg(reinterpret_cast<const uint4*>(g) + i);
    float4 w0 = reinterpret_cast<const float4*>(w)[2 * i], w1 = reinterpret_cast<const float4*>(w)[2 * i + 1];
    float4 m0 = reinterpret_cast<const float4*>(m)[2 * i], m1 = reinterpret_cast<const float4*>(m)[2 * i + 1];
    float4 v0 = reinterpret_cast<const float4*>(v)[2 * i], v1 = reinterpret_cast<const float4*>(v)[2 * i + 1];
    float gf[8];
    unpack8f(gu, gf);
    float wf[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
    float mf[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
    float vf[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float gi = gf[j] * gscale;
      mf[j] = b1 * mf[j] + c1 * gi;
      vf[j] = b2 * vf[j] + c2 * gi * gi;
      wf[j] -= lr * (mf[j] * inv_bc1 / (sqrtf(vf[j] * inv_bc2) + eps) + wd * wf[j]);
    }
    reinterpret_cast<float4*>(m)[2 * i] = make_float4(mf[0], mf[1], mf[2], mf[3]);
    reinterpret_cast<float4*>(m)[2 * i + 1] = make_float4(mf[4], mf[5], mf[6], mf[7]);
    reinterpret_cast<float4*>(v)[2 * i] = make_float4(vf[0], vf[1], vf[2], vf[3]);
    reinterpret_cast<float4*>(v)[2 * i + 1] = make_float4(vf[4], vf[5], vf[6], vf[7]);
    reinterpret_cast<float4*>(w)[2 * i] = make_float4(wf[0], wf[1], wf[2], wf[3]);
    reinterpret_cast<float4*>(w)[2 * i + 1] = make_float4(wf[4], wf[5], wf[6], wf[7]);
    reinterpret_cast<uint4*>(p)[i] = pack8f(wf);
  }
}

template <bool kSched>
__global__ void adamw_kernel(bf16* __restrict__ p, const bf16* __restrict__ g, float* __restrict__ w, float* __restrict__ m,
                             float* __restrict__ v, long long n, float lr, float b1, float b2, float eps, float wd,
                             float inv_bc1, float inv_bc2, float gscale, const int* __restrict__ step_dev,
                             const mm_opt_state* __restrict__ st) {
  if constexpr (kSched) {
    if (!st->apply) return;
    lr = st->lr;
    gscale = st->clip_coef;
    step_dev = &st->step;
  }
  if (step_dev != nullptr) {  // step count read on the device: the launch can be replayed from a CUDA graph
    const float t = static_cast<float>(*step_dev);
    inv_bc1 = 1.f / (1.f - powf(b1, t));
    inv_bc2 = 1.f / (1.f - powf(b2, t));
  }
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float gi = __bfloat162float(g[i]) * gscale;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    float wi = w[i];
    wi -= lr * (mi * inv_bc1 / (sqrtf(vi * inv_bc2) + eps) + wd * wi);
    m[i] = mi;
    v[i] = vi;
    w[i] = wi;
    p[i] = __float2bfloat16(wi);
  }
}

// ------------------------------------------------------------------------------------------------ global gradient norm
// Sum of squares over a table of bf16 gradient tensors, then the optimizer's per-step scalars (clip coefficient, step,
// learning rate).  Work unit: a chunk of kNormChunk consecutive elements of one tensor; the chunks of all tensors are
// numbered in table order and chunk c belongs to CTA c % gridDim.x.  Each thread squares its kNormVecs 8-element runs of
// a chunk in fp32 and adds that run sum to its fp64 accumulator; CTA sums (fixed shuffle tree) go to partials[blockIdx.x]
// and the last CTA to arrive adds them in index order.  Nothing depends on timing: the result is bit-identical across
// runs, graph replays and data-parallel ranks.
constexpr int kNormThreads = 256, kNormVecs = 8;
constexpr long long kNormChunk = static_cast<long long>(kNormThreads) * 8 * kNormVecs;

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// fixed-order CTA sum of one double per thread (every thread gets the result)
__device__ __forceinline__ double block_sum_f64(double v, double* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum_f64(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  return warp_sum_f64(lane < (kNormThreads >> 5) ? sh[lane] : 0.0);
}

// transformers.optimization lambdas, in fp64 as the Python LambdaLR computes them
__device__ double sched_lambda(int schedule, long long s, long long warmup, long long total) {
  if (schedule == MM_SCHED_CONSTANT) return 1.0;
  if (s < warmup) return static_cast<double>(s) / static_cast<double>(warmup > 1 ? warmup : 1);
  if (schedule == MM_SCHED_CONSTANT_WITH_WARMUP) return 1.0;
  const long long span = total - warmup > 1 ? total - warmup : 1;
  if (schedule == MM_SCHED_LINEAR) return fmax(0.0, static_cast<double>(total - s) / static_cast<double>(span));
  const double progress = static_cast<double>(s - warmup) / static_cast<double>(span);
  return fmax(0.0, 0.5 * (1.0 + cospi(0.5 * 2.0 * progress)));  // cos(pi * 2 * num_cycles * progress)
}

__global__ void __launch_bounds__(kNormThreads) grad_norm_kernel(const long long* __restrict__ table, int n_tensors,
                                                                 double* __restrict__ partials, mm_opt_state* st,
                                                                 float max_norm, int skip_nonfinite, float base_lr,
                                                                 int schedule, int warmup, int total) {
  __shared__ double sh[32];
  __shared__ bool last;
  const int G = gridDim.x, tid = threadIdx.x;
  const long long b = blockIdx.x;
  double acc = 0.0;
  long long base = 0;  // index of the current tensor's first chunk
  for (int t = 0; t < n_tensors; ++t) {
    const bf16* x = reinterpret_cast<const bf16*>(table[2 * t]);
    const long long n = table[2 * t + 1];
    const long long nc = (n + kNormChunk - 1) / kNormChunk;
    const bool vec = (reinterpret_cast<uintptr_t>(x) & 15) == 0;
    for (long long c = base + ((b - base % G) % G + G) % G; c < base + nc; c += G) {
      const long long e0 = (c - base) * kNormChunk;
      const long long e1 = e0 + kNormChunk < n ? e0 + kNormChunk : n;
      float run = 0.f;
      if (vec && e1 - e0 == kNormChunk) {
        uint4 u[kNormVecs];
#pragma unroll
        for (int j = 0; j < kNormVecs; ++j)
          u[j] = __ldg(reinterpret_cast<const uint4*>(x + e0) + j * kNormThreads + tid);
#pragma unroll
        for (int j = 0; j < kNormVecs; ++j) {
          float f[8];
          unpack8f(u[j], f);
#pragma unroll
          for (int k = 0; k < 8; ++k) run = fmaf(f[k], f[k], run);
        }
      } else {  // the last chunk of a tensor, or an unaligned tensor: scalar loads
        for (long long i = e0 + tid; i < e1; i += kNormThreads) {
          const float f = __bfloat162float(x[i]);
          run = fmaf(f, f, run);
        }
      }
      acc += static_cast<double>(run);
    }
    base += nc;
  }
  acc = block_sum_f64(acc, sh);
  if (tid == 0) {
    partials[blockIdx.x] = acc;
    __threadfence();
    last = atomicAdd(&st->arrived, 1) == G - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  double tot = 0.0;
  for (int i = tid; i < G; i += kNormThreads) tot += __ldcg(partials + i);
  tot = block_sum_f64(tot, sh);
  if (tid != 0) return;
  st->arrived = 0;
  const float norm = static_cast<float>(sqrt(tot));
  const bool finite = isfinite(tot);
  // torch.nn.utils.clip_grad_norm_: clamp(max_norm / (norm + 1e-6), max=1) in the norm's fp32 (NaN propagates)
  float coef = 1.f;
  if (max_norm > 0.f) {
    coef = max_norm / (norm + 1e-6f);
    coef = coef > 1.f ? 1.f : coef;
  }
  st->grad_norm = norm;
  st->finite = finite ? 1 : 0;
  st->clip_coef = coef;
  if (finite || !skip_nonfinite) {
    const int s = st->step;  // optimizer step s + 1 runs at lambda(s)
    st->step = s + 1;
    st->lr = static_cast<float>(static_cast<double>(base_lr) * sched_lambda(schedule, s, warmup, total));
    st->apply = 1;
  } else {
    st->skipped += 1;
    st->apply = 0;
  }
}

// ------------------------------------------------------------------------------------------------ alignment softmax backward
// One CTA per query row r of the absorbed alignment attention.  Inputs: G[r, v] = dctx~[r] . table[v] (fp32), the
// un-normalised fp16 probabilities P' of the forward pass and 1 / l, the gradients of the two per-row probability sums
// (d p_sum_real, d p_extra) and the UN-dropped p_extra.  With P = P' / l over the V real keys (+ the bias_k key, column V,
// with weight p_extra; the zero key's value is 0 so its dP is 0) and m the dropout multipliers (ones when off):
//   dP_v = m_v (G_v + d p_sum_real),   D = sum_v P_v dP_v + p_extra m_V d p_extra,   dS_v = P_v (dP_v - D)
// Outputs: Pd = m . P and dS as bf16 (operands of the table-gradient GEMMs dT += Pd^T dctx~ + dS^T q~ and of dq~ = dS . table),
// dstats[0][r] = gscale * sum_v dS_v, dstats[1][r] = gscale * p_extra * (m_V d p_extra - D) — the gradients of row_bias and
// of the bias_k key's score (planar [2][R]).
__global__ void __launch_bounds__(512) align_softmax_bwd_kernel(const float* __restrict__ G, long long ldg,
                                                                const __half* __restrict__ Pp, long long ldp,
                                                                const float* __restrict__ inv_l,
                                                                const float* __restrict__ dpsr, const float* __restrict__ pe,
                                                                const float* __restrict__ dpe, float gscale,
                                                                bf16* __restrict__ P, bf16* __restrict__ dS, long long ldo,
                                                                float* __restrict__ dstats, int V, float p_drop,
                                                                const unsigned long long* __restrict__ seed_dev,
                                                                uint32_t sid) {
  __shared__ float sh[32];
  const long long r = blockIdx.x;
  const float* g = G + r * ldg;
  const __half* pp = Pp + r * ldp;
  bf16* po = P + r * ldo;
  bf16* dso = dS + r * ldo;
  const float il = inv_l[r], a = dpsr[r], pex = pe[r], dpex = dpe[r];
  const DropCfg dc = drop_cfg(p_drop, seed_dev, sid);
  const int n4 = (V + 3) >> 2;
  float acc = 0.f;
  for (int v4 = threadIdx.x; v4 < n4; v4 += blockDim.x) {
    float m[4];
    drop_mult4(dc, static_cast<uint32_t>(r), static_cast<uint32_t>(v4), m);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int v = 4 * v4 + u;
      if (v < V) acc += __half2float(pp[v]) * il * m[u] * (g[v] + a);
    }
  }
  const float me = drop_mult1(dc, static_cast<uint32_t>(r), static_cast<uint32_t>(V));
  const float D = block_sum(acc, sh) + pex * me * dpex;
  float srow = 0.f;
  for (int v4 = threadIdx.x; v4 < n4; v4 += blockDim.x) {
    float m[4];
    drop_mult4(dc, static_cast<uint32_t>(r), static_cast<uint32_t>(v4), m);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int v = 4 * v4 + u;
      if (v >= V) break;
      const float pv = __half2float(pp[v]) * il;
      const float d = pv * (m[u] * (g[v] + a) - D);
      po[v] = __float2bfloat16(pv * m[u]);
      dso[v] = __float2bfloat16(d);
      srow += d;
    }
  }
  srow = block_sum(srow, sh);
  if (threadIdx.x == 0) {  // planar [2][R]: each half is the per-row scale array of a row-scaled GEMM bias term
    dstats[r] = gscale * srow;
    dstats[gridDim.x + r] = gscale * pex * (me * dpex - D);
  }
}

// Training-mode dropout of the alignment probabilities (forward): from the fused kernel's un-normalised fp16 P' makes
// Pm = P' where kept, 0 where dropped (UNSCALED: P' may sit near the top of the fp16 range), the per-row scale
// rs = (1 / l) / (1 - p) of the following ctx~ = rs . (Pm . table) GEMM, and the dropped probability sums
// p_sum_real_d = rs * sum_v Pm_v,  p_extra_d = m_V * p_extra (column V = the bias_k key; the zero key has no effect).
__global__ void __launch_bounds__(512) align_dropout_fwd_kernel(const __half* __restrict__ Pp, __half* __restrict__ Pm,
                                                                long long ldp, const float* __restrict__ inv_l,
                                                                const float* __restrict__ pe, float* __restrict__ rs,
                                                                float* __restrict__ psum_d, float* __restrict__ pext_d,
                                                                int V, float p_drop,
                                                                const unsigned long long* __restrict__ seed_dev,
                                                                uint32_t sid) {
  __shared__ float sh[32];
  const long long r = blockIdx.x;
  const __half* pp = Pp + r * ldp;
  __half* po = Pm + r * ldp;
  const DropCfg dc = drop_cfg(p_drop, seed_dev, sid);
  const int n4 = (V + 3) >> 2;
  float acc = 0.f;
  for (int v4 = threadIdx.x; v4 < n4; v4 += blockDim.x) {
    float m[4];
    drop_mult4(dc, static_cast<uint32_t>(r), static_cast<uint32_t>(v4), m);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int v = 4 * v4 + u;
      if (v >= V) break;
      const __half h = pp[v];
      const bool keep = m[u] != 0.f;
      po[v] = keep ? h : __float2half_rn(0.f);
      if (keep) acc += __half2float(h);
    }
  }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) {
    const float s = inv_l[r] * dc.scale;
    rs[r] = s;
    psum_d[r] = s * acc;
    pext_d[r] = pe[r] * drop_mult1(dc, static_cast<uint32_t>(r), static_cast<uint32_t>(V));
  }
}

// out[h*hd + d] += sum_n w[h*Nq + n] * x[n, h*hd + d]   (x bf16 or fp16; bias gradients of the per-head bias terms)
__global__ void head_weighted_colsum_kernel(const void* __restrict__ x, long long ldx, int x_fp16,
                                            const float* __restrict__ w, long long w_stride, int Nq, int E, int hd,
                                            float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= E) return;
  const int h = c / hd;
  float acc = 0.f;
  for (int n = 0; n < Nq; ++n) {
    const float xv = x_fp16 ? __half2float(reinterpret_cast<const __half*>(x)[static_cast<long long>(n) * ldx + c])
                            : __bfloat162float(reinterpret_cast<const bf16*>(x)[static_cast<long long>(n) * ldx + c]);
    acc += w[(static_cast<long long>(h) * Nq + n) * w_stride] * xv;
  }
  atomicAdd(&out[c], acc);
}

__global__ void cast_f16_bf16_kernel(const __half* __restrict__ x, long long ldx, bf16* __restrict__ y, long long ldy,
                                     int rows, int cols) {
  const long long total = static_cast<long long>(rows) * cols;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / cols;
    const int c = static_cast<int>(i % cols);
    y[r * ldy + c] = __float2bfloat16(__half2float(x[r * ldx + c]));
  }
}

// Data gradient of a strided Conv1d over the token axis (col2im): dwin[(b*Lq + l), k*C + c] holds d(window l)[k, c];
// dfeats[b, t, c] = sum over the windows l that contain token t (l*ss <= t < l*ss + kk) of dwin[b*Lq + l, (t - l*ss)*C + c].
__global__ void window_gather_add_kernel(const bf16* __restrict__ dwin, int B, int N, int C, int Lq, int kk, int ss,
                                         bf16* __restrict__ dfeats) {
  const long long total = static_cast<long long>(B) * N * C;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const int t = static_cast<int>((i / C) % N);
    const int b = static_cast<int>(i / (static_cast<long long>(C) * N));
    int l_hi = t / ss;
    if (l_hi > Lq - 1) l_hi = Lq - 1;
    int l_lo = (t - kk + ss) / ss;  // ceil((t - kk + 1) / ss)
    if (t - kk + 1 <= 0) l_lo = 0;
    float acc = 0.f;
    for (int l = l_lo; l <= l_hi; ++l) {
      const int k = t - l * ss;
      if (k >= 0 && k < kk)
        acc += __bfloat162float(dwin[(static_cast<long long>(b) * Lq + l) * (static_cast<long long>(kk) * C) +
                                     static_cast<long long>(k) * C + c]);
    }
    dfeats[i] = __float2bfloat16(acc);
  }
}

static inline int grid_for(long long total, int block, int cap_mult = 16) {
  long long g = (total + block - 1) / block;
  const long long cap = static_cast<long long>(num_sms()) * cap_mult;
  return static_cast<int>(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace mm

using namespace mm;
#define AL16(p) ((reinterpret_cast<uintptr_t>(p) & 15) == 0)

extern "C" int32_t mm_rmsnorm_bwd_parts(int32_t rows) {
  int rpc = (rows + 4 * num_sms() - 1) / (4 * num_sms());
  if (rpc < 1) rpc = 1;
  return (rows + rpc - 1) / rpc;
}

extern "C" int32_t mm_rmsnorm_bwd(const void* dy, const void* x, const float* rstd, const void* g, const void* dres,
                                  void* dx, float* dg, float* dg_partials, int32_t rows, int32_t cols, void* stream) {
  MM_REQUIRE(dy && x && rstd && g && dx && rows > 0 && cols > 0 && cols % 8 == 0 && cols <= 256 * 8 * kNormMaxChunks,
             "mm_rmsnorm_bwd: bad arguments (cols %% 8 == 0, cols <= %d)", 256 * 8 * kNormMaxChunks);
  MM_REQUIRE(AL16(dy) && AL16(x) && AL16(g) && AL16(dx) && (dres == nullptr || AL16(dres)), "mm_rmsnorm_bwd: alignment");
  int rpc = (rows + 4 * num_sms() - 1) / (4 * num_sms());
  if (rpc < 1) rpc = 1;
  const int grid = (rows + rpc - 1) / rpc;
  MM_REQUIRE(dg_partials == nullptr || (dg != nullptr && AL16(dg_partials)), "mm_rmsnorm_bwd: dg_partials needs dg, 16-byte aligned");
#define MM_RB(NCH_) \
  rmsnorm_bwd_kernel<NCH_><<<grid, 256, 0, ST(stream)>>>((const bf16*)dy, (const bf16*)x, rstd, (const bf16*)g,           \
                                                         (const bf16*)dres, (bf16*)dx, dg, dg_partials, rows, cols, rpc)
  if (cols <= 256 * 8) MM_RB(1);
  else if (cols <= 256 * 8 * 2) MM_RB(2);
  else MM_RB(4);
#undef MM_RB
  if (dg_partials != nullptr) dg_reduce_kernel<<<(cols + 31) / 32, 256, 0, ST(stream)>>>(dg_partials, grid, cols, dg);
  return check_launch("mm_rmsnorm_bwd");
}

extern "C" int32_t mm_swiglu_fwd(const void* gate, const void* up, void* h, int64_t n, void* stream) {
  MM_REQUIRE(gate && up && h && n > 0 && n % 8 == 0 && AL16(gate) && AL16(up) && AL16(h), "mm_swiglu_fwd: bad arguments");
  swiglu_fwd_kernel<<<grid_for(n / 8, 256), 256, 0, ST(stream)>>>((const bf16*)gate, (const bf16*)up, (bf16*)h, n / 8);
  return check_launch("mm_swiglu_fwd");
}

extern "C" int32_t mm_swiglu_bwd(const void* dh, const void* gate, const void* up, void* dgate, void* dup, int64_t n,
                                 void* stream) {
  MM_REQUIRE(dh && gate && up && dgate && dup && n > 0 && n % 8 == 0, "mm_swiglu_bwd: bad arguments");
  MM_REQUIRE(AL16(dh) && AL16(gate) && AL16(up) && AL16(dgate) && AL16(dup), "mm_swiglu_bwd: alignment");
  swiglu_bwd_kernel<<<grid_for(n / 8, 256), 256, 0, ST(stream)>>>((const bf16*)dh, (const bf16*)gate, (const bf16*)up,
                                                                 (bf16*)dgate, (bf16*)dup, n / 8);
  return check_launch("mm_swiglu_bwd");
}

extern "C" int32_t mm_attn_softmax_bwd(const float* S, const float* dP, void* P, void* dS, int32_t B, int32_t H, int32_t Tq,
                                       int32_t Tk, int64_t ld, float scale, int32_t causal, const int32_t* key_mask,
                                       float p_drop, const uint64_t* seed_dev, uint32_t sid, void* stream) {
  MM_REQUIRE(S && dP && P && dS && B > 0 && H > 0 && Tq > 0 && Tk > 0 && ld >= Tk, "mm_attn_softmax_bwd: bad arguments");
  MM_REQUIRE(p_drop >= 0.f && p_drop < 1.f && (p_drop == 0.f || seed_dev != nullptr), "mm_attn_softmax_bwd: dropout arguments");
  const long long rows = static_cast<long long>(B) * H * Tq;
  MM_REQUIRE(rows < (1LL << 31), "mm_attn_softmax_bwd: too many rows");
  const unsigned wgrid = static_cast<unsigned>((rows + 7) / 8);
#define MM_SB(NV_) \
  attn_softmax_bwd_warp_kernel<NV_><<<wgrid, 256, 0, ST(stream)>>>(S, dP, (bf16*)P, (bf16*)dS, rows, H, Tq, Tk, ld, scale, \
                                                                   causal, key_mask, p_drop,                               \
                                                                   (const unsigned long long*)seed_dev, sid)
  const int need = (Tk + 31) / 32;  // columns per lane
  if (need <= 4) MM_SB(4);
  else if (need <= 8) MM_SB(8);
  else if (need <= 12) MM_SB(12);
  else if (need <= 16) MM_SB(16);
  else if (need <= 17) MM_SB(17);  // T = 528: the training bench's sequence length
  else if (need <= 20) MM_SB(20);
  else if (need <= 24) MM_SB(24);
  else if (need <= 32) MM_SB(32);
  else
    attn_softmax_bwd_kernel<<<static_cast<unsigned>(rows), 256, 0, ST(stream)>>>(S, dP, (bf16*)P, (bf16*)dS, H, Tq, Tk, ld,
                                                                                 scale, causal, key_mask, p_drop,
                                                                                 (const unsigned long long*)seed_dev, sid);
#undef MM_SB
  return check_launch("mm_attn_softmax_bwd");
}

extern "C" int32_t mm_attn_softmax_fwd(const float* S, void* P, int32_t B, int32_t H, int32_t Tq, int32_t Tk, int64_t ld,
                                       float scale, int32_t causal, const int32_t* key_mask, float p_drop,
                                       const uint64_t* seed_dev, uint32_t sid, void* stream) {
  MM_REQUIRE(S && P && B > 0 && H > 0 && Tq > 0 && Tk > 0 && ld >= Tk, "mm_attn_softmax_fwd: bad arguments");
  MM_REQUIRE(p_drop >= 0.f && p_drop < 1.f && (p_drop == 0.f || seed_dev != nullptr), "mm_attn_softmax_fwd: dropout arguments");
  const long long rows = static_cast<long long>(B) * H * Tq;
  MM_REQUIRE(rows < (1LL << 31), "mm_attn_softmax_fwd: too many rows");
  attn_softmax_fwd_kernel<<<static_cast<unsigned>(rows), 256, 0, ST(stream)>>>(S, (bf16*)P, H, Tq, Tk, ld, scale, causal,
                                                                               key_mask, p_drop,
                                                                               (const unsigned long long*)seed_dev, sid);
  return check_launch("mm_attn_softmax_fwd");
}

extern "C" int32_t mm_dropout_mask(float* out, int64_t ld, int32_t rows, int32_t cols, float p_drop, const uint64_t* seed_dev,
                                   uint32_t sid, void* stream) {
  MM_REQUIRE(out && rows > 0 && cols > 0 && ld >= cols && p_drop >= 0.f && p_drop < 1.f && seed_dev, "mm_dropout_mask: bad arguments");
  const long long total = static_cast<long long>(rows) * ((cols + 3) / 4);
  dropout_mask_kernel<<<grid_for(total, 256), 256, 0, ST(stream)>>>(out, ld, rows, cols, p_drop,
                                                                   (const unsigned long long*)seed_dev, sid);
  return check_launch("mm_dropout_mask");
}

extern "C" int32_t mm_align_dropout_fwd(const void* Pp, void* Pm, int64_t ldp, const float* inv_l, const float* pe, float* rs,
                                        float* psum_d, float* pext_d, int32_t R, int32_t V, float p_drop,
                                        const uint64_t* seed_dev, uint32_t sid, void* stream) {
  MM_REQUIRE(Pp && Pm && inv_l && pe && rs && psum_d && pext_d && R > 0 && V > 0 && ldp >= V, "mm_align_dropout_fwd: bad arguments");
  MM_REQUIRE(p_drop >= 0.f && p_drop < 1.f && (p_drop == 0.f || seed_dev != nullptr), "mm_align_dropout_fwd: dropout arguments");
  align_dropout_fwd_kernel<<<R, 512, 0, ST(stream)>>>((const __half*)Pp, (__half*)Pm, ldp, inv_l, pe, rs, psum_d, pext_d, V,
                                                      p_drop, (const unsigned long long*)seed_dev, sid);
  return check_launch("mm_align_dropout_fwd");
}

extern "C" int32_t mm_ce_bwd(const void* logits, const int64_t* labels, void* dlogits, int32_t B, int32_t T, int32_t V,
                             const int32_t* n_valid, float grad_scale, const float* grad_scale_dev, void* stream) {
  MM_REQUIRE(logits && labels && dlogits && n_valid && B > 0 && T > 0 && V > 0, "mm_ce_bwd: bad arguments");
  ce_bwd_kernel<<<B * T, 512, 0, ST(stream)>>>((const bf16*)logits, (const long long*)labels, (bf16*)dlogits, T, V, n_valid,
                                               grad_scale, grad_scale_dev);
  return check_launch("mm_ce_bwd");
}

extern "C" int32_t mm_embed_scatter_add(const void* dx, int64_t ldx, const int64_t* ids, int64_t n, int32_t dim,
                                        int32_t vocab, void* dtable, void* stream) {
  MM_REQUIRE(dx && ids && dtable && n > 0 && dim > 0 && dim % 2 == 0 && ldx % 2 == 0 && vocab > 0,
             "mm_embed_scatter_add: bad arguments");
  embed_scatter_add_kernel<<<grid_for(n * (dim / 2), 256), 256, 0, ST(stream)>>>((const bf16*)dx, ldx, (const long long*)ids, n,
                                                                                dim, vocab, (bf16*)dtable);
  return check_launch("mm_embed_scatter_add");
}

extern "C" int32_t mm_colsum(const void* x, int64_t ldx, int32_t rows, int32_t cols, float* out, void* stream) {
  MM_REQUIRE(x && out && rows > 0 && cols > 0, "mm_colsum: bad arguments");
  int rpc = (rows + 63) / 64;
  dim3 grid((rows + rpc - 1) / rpc, (cols + 255) / 256);
  colsum_kernel<<<grid, 256, 0, ST(stream)>>>((const bf16*)x, ldx, rows, cols, out, rpc);
  return check_launch("mm_colsum");
}

template <bool kSched>
static void launch_adamw(void* p, const void* g, float* master, float* m, float* v, long long n, float lr, float beta1,
                         float beta2, float eps, float weight_decay, float inv_bc1, float inv_bc2, float grad_scale,
                         const int32_t* step_dev, const mm_opt_state* st, void* stream) {
  const long long n8 = (AL16(p) && AL16(g) && AL16(master) && AL16(m) && AL16(v)) ? n / 8 : 0;
  if (n8 > 0)
    adamw_vec8_kernel<kSched><<<grid_for(n8, 256, 32), 256, 0, ST(stream)>>>((bf16*)p, (const bf16*)g, master, m, v, n8, lr,
                                                                             beta1, beta2, eps, weight_decay, inv_bc1, inv_bc2,
                                                                             grad_scale, step_dev, st);
  if (n - 8 * n8 > 0) {  // unaligned tensors / the last n % 8 elements
    const long long o = 8 * n8;
    adamw_kernel<kSched><<<grid_for(n - o, 256), 256, 0, ST(stream)>>>((bf16*)p + o, (const bf16*)g + o, master + o, m + o,
                                                                       v + o, n - o, lr, beta1, beta2, eps, weight_decay,
                                                                       inv_bc1, inv_bc2, grad_scale, step_dev, st);
  }
}

extern "C" int32_t mm_adamw(void* p, const void* g, float* master, float* m, float* v, int64_t n, float lr, float beta1,
                            float beta2, float eps, float weight_decay, int32_t step, const int32_t* step_dev,
                            float grad_scale, void* stream) {
  MM_REQUIRE(p && g && master && m && v && n > 0 && (step > 0 || step_dev != nullptr), "mm_adamw: bad arguments");
  if (step <= 0) step = 1;
  const float inv_bc1 = 1.f / (1.f - powf(beta1, static_cast<float>(step)));
  const float inv_bc2 = 1.f / (1.f - powf(beta2, static_cast<float>(step)));
  launch_adamw<false>(p, g, master, m, v, n, lr, beta1, beta2, eps, weight_decay, inv_bc1, inv_bc2, grad_scale, step_dev,
                      nullptr, stream);
  return check_launch("mm_adamw");
}

extern "C" int32_t mm_adamw_sched(void* p, const void* g, float* master, float* m, float* v, int64_t n, float beta1,
                                  float beta2, float eps, float weight_decay, const mm_opt_state* state, void* stream) {
  MM_REQUIRE(p && g && master && m && v && n > 0 && state, "mm_adamw_sched: bad arguments");
  launch_adamw<true>(p, g, master, m, v, n, 0.f, beta1, beta2, eps, weight_decay, 1.f, 1.f, 1.f, nullptr, state, stream);
  return check_launch("mm_adamw_sched");
}

extern "C" int32_t mm_grad_norm(const int64_t* table, int32_t n_tensors, double* partials, mm_opt_state* state,
                                float max_norm, int32_t skip_nonfinite, float base_lr, int32_t schedule, int32_t warmup_steps,
                                int32_t total_steps, void* stream) {
  MM_REQUIRE(state && partials && n_tensors >= 0 && (n_tensors == 0 || table), "mm_grad_norm: bad arguments");
  MM_REQUIRE(schedule >= MM_SCHED_CONSTANT && schedule <= MM_SCHED_COSINE && warmup_steps >= 0 && total_steps >= 0,
             "mm_grad_norm: bad schedule");
  // the grid is a constant (not a function of the device): the partition, hence every bit of the sum, is the same on
  // every rank.  Without tensors the launch is the finisher alone.
  const int grid = n_tensors > 0 ? MM_GRAD_NORM_PARTS : 1;
  grad_norm_kernel<<<grid, kNormThreads, 0, ST(stream)>>>((const long long*)table, n_tensors, partials, state, max_norm,
                                                          skip_nonfinite, base_lr, schedule, warmup_steps, total_steps);
  return check_launch("mm_grad_norm");
}

extern "C" int32_t mm_align_softmax_bwd(const float* G, int64_t ldg, const void* Pp, int64_t ldp, const float* inv_l,
                                        const float* dpsr, const float* pe, const float* dpe, float gscale, void* P,
                                        void* dS, int64_t ldo, float* dstats, int32_t R, int32_t V, float p_drop,
                                        const uint64_t* seed_dev, uint32_t sid, void* stream) {
  MM_REQUIRE(G && Pp && inv_l && dpsr && pe && dpe && P && dS && dstats && R > 0 && V > 0 && ldg >= V && ldp >= V && ldo >= V,
             "mm_align_softmax_bwd: bad arguments");
  MM_REQUIRE(p_drop >= 0.f && p_drop < 1.f && (p_drop == 0.f || seed_dev != nullptr), "mm_align_softmax_bwd: dropout arguments");
  align_softmax_bwd_kernel<<<R, 512, 0, ST(stream)>>>(G, ldg, (const __half*)Pp, ldp, inv_l, dpsr, pe, dpe, gscale, (bf16*)P,
                                                      (bf16*)dS, ldo, dstats, V, p_drop,
                                                      (const unsigned long long*)seed_dev, sid);
  return check_launch("mm_align_softmax_bwd");
}

extern "C" int32_t mm_head_weighted_colsum(const void* x, int64_t ldx, int32_t x_fp16, const float* w, int64_t w_stride,
                                           int32_t Nq, int32_t E, int32_t head_dim, float* out, void* stream) {
  MM_REQUIRE(x && w && out && Nq > 0 && E > 0 && head_dim > 0 && E % head_dim == 0 && w_stride > 0,
             "mm_head_weighted_colsum: bad arguments");
  head_weighted_colsum_kernel<<<(E + 255) / 256, 256, 0, ST(stream)>>>(x, ldx, x_fp16, w, w_stride, Nq, E, head_dim, out);
  return check_launch("mm_head_weighted_colsum");
}

extern "C" int32_t mm_cast_f16_bf16(const void* x, int64_t ldx, void* y, int64_t ldy, int32_t rows, int32_t cols,
                                    void* stream) {
  MM_REQUIRE(x && y && rows > 0 && cols > 0, "mm_cast_f16_bf16: bad arguments");
  cast_f16_bf16_kernel<<<grid_for(static_cast<long long>(rows) * cols, 256), 256, 0, ST(stream)>>>(
      (const __half*)x, ldx, (bf16*)y, ldy, rows, cols);
  return check_launch("mm_cast_f16_bf16");
}

extern "C" int32_t mm_window_gather_add(const void* dwin, int32_t B, int32_t N, int32_t C, int32_t Lq, int32_t kk, int32_t ss,
                                        void* dfeats, void* stream) {
  MM_REQUIRE(dwin && dfeats && B > 0 && N > 0 && C > 0 && Lq > 0 && kk > 0 && ss > 0, "mm_window_gather_add: bad arguments");
  window_gather_add_kernel<<<grid_for(static_cast<long long>(B) * N * C, 256), 256, 0, ST(stream)>>>(
      (const bf16*)dwin, B, N, C, Lq, kk, ss, (bf16*)dfeats);
  return check_launch("mm_window_gather_add");
}
