// td.cu - time-dependency + pooling kernels.
//   adapt arch  : Linear 384->64 + LayerNorm (reference nisqa/NISQA_lib.py:989-991),
//                 2x post-norm encoder layer with 1-head attention (lib:1025-1040),
//                 5 (or 1) PoolAttFF heads (lib:1171-1183, fan-out lib:260-268).
//   standard    : fc_out 768->20 (lib:832-834), BiLSTM (lib:925-943), PoolLastStepBi
//                 (lib:1107-1115).
// All of it is row-local fp32 work on [n_seg, 64] matrices (3.5 % of the FLOPs of a clip):
// one thread owns one time step (row); weights sit in shared memory as [k][out] so the
// inner loop is a warp-broadcast LDS.128 per 4 FMAs.  Clips are ragged: every kernel works
// on the valid rows only, so no key-padding mask exists (masked keys in the reference
// contribute exactly 0 after softmax).
#include <algorithm>

#include "common.cuh"

namespace nisqa {

constexpr int kRows = 128;       // rows (threads) per CTA in the row-thread kernels
constexpr int kXS = 65;          // padded row stride of the per-thread smem row

// acc[j] += sum_{k<kc} xrow[k] * ws[k*NCOL + j]
template <int NCOL>
__device__ __forceinline__ void rowgemm(float (&acc)[NCOL], const float* xrow, const float* ws, int kc) {
  static_assert(NCOL % 4 == 0, "NCOL");
#pragma unroll 4
  for (int k = 0; k < kc; ++k) {
    const float xv = xrow[k];
    const float4* w4 = reinterpret_cast<const float4*>(ws + k * NCOL);
#pragma unroll
    for (int q = 0; q < NCOL / 4; ++q) {
      const float4 w = w4[q];
      acc[q * 4 + 0] = fmaf(xv, w.x, acc[q * 4 + 0]);
      acc[q * 4 + 1] = fmaf(xv, w.y, acc[q * 4 + 1]);
      acc[q * 4 + 2] = fmaf(xv, w.z, acc[q * 4 + 2]);
      acc[q * 4 + 3] = fmaf(xv, w.w, acc[q * 4 + 3]);
    }
  }
}

// nn.LayerNorm(64): biased variance, eps 1e-5
__device__ __forceinline__ void layernorm64(float (&v)[64], const float* __restrict__ gamma,
                                            const float* __restrict__ beta) {
  float mean = 0.f;
#pragma unroll
  for (int j = 0; j < 64; ++j) mean += v[j];
  mean *= (1.0f / 64.0f);
  float var = 0.f;
#pragma unroll
  for (int j = 0; j < 64; ++j) { const float d = v[j] - mean; var = fmaf(d, d, var); }
  const float rstd = 1.0f / sqrtf(var * (1.0f / 64.0f) + 1e-5f);
#pragma unroll
  for (int j = 0; j < 64; ++j) v[j] = (v[j] - mean) * rstd * __ldg(gamma + j) + __ldg(beta + j);
}

__device__ __forceinline__ void stage_f4(float* dst, const float* __restrict__ src, int n_floats) {
  const float4* s = reinterpret_cast<const float4*>(src);
  for (int i = threadIdx.x; i < n_floats / 4; i += blockDim.x) reinterpret_cast<float4*>(dst)[i] = __ldg(s + i);
}

// ---------------------------------------------------------------------------------------
// out[row][0..NOUT) = (LN?)( in[row][0..K) @ WT[K][NOUT] + bias )   K % 64 == 0
template <int NOUT, bool LN>
__global__ void __launch_bounds__(kRows)
linear_rows_kernel(const float* __restrict__ in, int K, const float* __restrict__ WT,
                   const float* __restrict__ bias, const float* __restrict__ gamma,
                   const float* __restrict__ beta, float* __restrict__ out, int n_rows) {
  extern __shared__ __align__(16) float sm[];
  float* xs = sm;                       // [kRows][kXS]
  float* ws = sm + kRows * kXS;         // [64][NOUT]
  const int row0 = blockIdx.x * kRows, tid = threadIdx.x;
  float acc[NOUT];
#pragma unroll
  for (int j = 0; j < NOUT; ++j) acc[j] = __ldg(bias + j);
  for (int k0 = 0; k0 < K; k0 += 64) {
    __syncthreads();
    for (int i = tid; i < kRows * 64; i += kRows) {
      const int r = i >> 6, k = i & 63;
      xs[r * kXS + k] = (row0 + r < n_rows) ? __ldg(in + (size_t)(row0 + r) * K + k0 + k) : 0.f;
    }
    stage_f4(ws, WT + (size_t)k0 * NOUT, 64 * NOUT);
    __syncthreads();
    rowgemm<NOUT>(acc, xs + tid * kXS, ws, 64);
  }
  if (row0 + tid >= n_rows) return;
  if constexpr (LN) {
    static_assert(!LN || NOUT == 64, "LayerNorm width");
    layernorm64(acc, gamma, beta);
  }
  float* o = out + (size_t)(row0 + tid) * NOUT;
#pragma unroll
  for (int q = 0; q < NOUT / 4; ++q)
    reinterpret_cast<float4*>(o)[q] = make_float4(acc[q * 4], acc[q * 4 + 1], acc[q * 4 + 2], acc[q * 4 + 3]);
}

// ---------------------------------------------------------------------------------------
struct SaLayerParams {
  const float* WoT; const float* bo; const float* W1T; const float* b1; const float* W2T;
  const float* b2; const float* ln1_g; const float* ln1_b; const float* ln2_g; const float* ln2_b;
};
// PoolAttFF (lib:1156-1183): the logits w2_h . relu(W1_h x + b1_h) + b2_h come out of td_sa_kernel's fused tail
struct PoolHeadParams {      // device pointers, heads concatenated
  const float* W1T;   // [n_heads][64 k][128 j]
  const float* b1;    // [n_heads][128]
  const float* w2;    // [n_heads][128]
  const float* b2;    // [n_heads]
  const float* w3;    // [n_heads][64]
  const float* b3;    // [n_heads]
};

// softmax over the clip's time steps, weighted sum of x, Linear 64->1   (lib:1177-1181)
// grid = n_clips, block = 64 * n_heads; thread (h, d).  The softmax numerators are formed once per (head, step) into shared
// memory; the weighted sum keeps ONE accumulator per thread in step order (the result does not depend on the unrolling) with
// eight independent loads in flight.
__global__ void pool_final_kernel(const float* __restrict__ x, const float* __restrict__ logits,
                                  const ClipDesc* __restrict__ clips, PoolHeadParams P, int n_heads, int max_seg,
                                  float* __restrict__ scores) {
  __shared__ float red[5 * 64];
  extern __shared__ float pnum[];                       // [n_heads][max_seg] softmax numerators
  const ClipDesc cd = clips[blockIdx.x];
  const int S = cd.n_seg;
  const int h = threadIdx.x >> 6, d = threadIdx.x & 63;
  if (S <= 0) { if (d == 0) scores[blockIdx.x * n_heads + h] = __int_as_float(0x7fc00000); return; }
  const float* lg = logits + (size_t)cd.seg_off * n_heads + h;
  float* pn = pnum + (size_t)h * max_seg;
  float mx = -INFINITY;
  for (int t = d; t < S; t += 64) mx = fmaxf(mx, __ldg(lg + (size_t)t * n_heads));
  red[threadIdx.x] = mx;
  __syncthreads();
  for (int o = 32; o > 0; o >>= 1) { if (d < o) red[threadIdx.x] = fmaxf(red[threadIdx.x], red[threadIdx.x + o]); __syncthreads(); }
  mx = red[h * 64];
  __syncthreads();
  float sum = 0.f;
  for (int t = d; t < S; t += 64) { const float e = expf(__ldg(lg + (size_t)t * n_heads) - mx); pn[t] = e; sum += e; }
  red[threadIdx.x] = sum;
  __syncthreads();
  for (int o = 32; o > 0; o >>= 1) { if (d < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
  sum = red[h * 64];
  __syncthreads();
  const float* xb = x + (size_t)cd.seg_off * 64 + d;
  float acc = 0.f;
  int t = 0;
  for (; t + 8 <= S; t += 8) {
    float xv[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) xv[u] = __ldg(xb + (size_t)(t + u) * 64);
#pragma unroll
    for (int u = 0; u < 8; ++u) acc = fmaf(pn[t + u], xv[u], acc);
  }
  for (; t < S; ++t) acc = fmaf(pn[t], __ldg(xb + (size_t)t * 64), acc);
  acc = (acc / sum) * __ldg(P.w3 + h * 64 + d);
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 32; o > 0; o >>= 1) { if (d < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
  if (d == 0) scores[blockIdx.x * n_heads + h] = red[h * 64] + __ldg(P.b3 + h);
}

// ---------------------------------------------------------------------------------------
// The other pooling modules of the reference (user-trained checkpoints, SURVEY.md 8f.4), one CTA per clip, D threads
// (thread d owns feature d; D = 64 after self-attention, 256 after the BiLSTM):
//   mode 1 PoolAtt       (lib:1131-1154): att_t = a1 . x_t + a1b, softmax over the clip's steps, sum_t att_t x_t, Linear
//   mode 2 PoolAvg       (lib:1185-1204): mean over the clip's steps, Linear
//   mode 3 PoolMax       (lib:1206-1225): max over the clip's steps, Linear
//   mode 4 PoolLastStep  (lib:1117-1129): x at the last valid step, Linear
// One Linear(D -> 1) per head (NISQA_DIM: five heads with their own weights, lib:260-268).
struct PoolSimpleParams { const float* a1; const float* a1b; const float* w3; const float* b3; };

template <int D>
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int w = 0; w < D / 32; ++w) t += red[w];
  return t;
}
template <int D>
__device__ __forceinline__ float block_max(float v, float* red) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = -INFINITY;
#pragma unroll
  for (int w = 0; w < D / 32; ++w) t = fmaxf(t, red[w]);
  return t;
}

template <int D>
__global__ void __launch_bounds__(D)
pool_simple_kernel(const float* __restrict__ x /*[n_seg][D]*/, const ClipDesc* __restrict__ clips, int mode,
                   PoolSimpleParams P, int n_heads, float* __restrict__ scores) {
  extern __shared__ __align__(16) float slog[];          // mode 1: softmax numerators of the clip's steps
  __shared__ float red[D / 32];
  const ClipDesc cd = clips[blockIdx.x];
  const int S = cd.n_seg, d = threadIdx.x, lane = d & 31, warp = d >> 5;
  if (S <= 0) { if (d < n_heads) scores[blockIdx.x * n_heads + d] = __int_as_float(0x7fc00000); return; }
  const float* xb = x + (size_t)cd.seg_off * D;
  float pooled = 0.f;
  if (mode == 2) {
    for (int t = 0; t < S; ++t) pooled += __ldg(xb + (size_t)t * D + d);
    pooled = pooled / (float)S;
  } else if (mode == 3) {
    pooled = -INFINITY;
    for (int t = 0; t < S; ++t) pooled = fmaxf(pooled, __ldg(xb + (size_t)t * D + d));
  } else if (mode == 4) {
    pooled = __ldg(xb + (size_t)(S - 1) * D + d);
  }
  for (int h = 0; h < n_heads; ++h) {
    if (mode == 1) {
      __syncthreads();                                    // slog of the previous head consumed
      for (int t = warp; t < S; t += D / 32) {
        float a = 0.f;
        for (int k = lane; k < D; k += 32) a = fmaf(__ldg(xb + (size_t)t * D + k), __ldg(P.a1 + h * D + k), a);
        a = warp_sum(a);
        if (lane == 0) slog[t] = a + __ldg(P.a1b + h);
      }
      __syncthreads();
      float mx = -INFINITY;
      for (int t = d; t < S; t += D) mx = fmaxf(mx, slog[t]);
      mx = block_max<D>(mx, red);
      float sum = 0.f;
      for (int t = d; t < S; t += D) { const float e = expf(slog[t] - mx); slog[t] = e; sum += e; }
      sum = block_sum<D>(sum, red);                       // (its barriers also publish the numerators)
      float acc = 0.f;
      for (int t = 0; t < S; ++t) acc = fmaf(slog[t], __ldg(xb + (size_t)t * D + d), acc);
      pooled = acc / sum;
    }
    const float tot = block_sum<D>(pooled * __ldg(P.w3 + h * D + d), red);
    if (d == 0) scores[blockIdx.x * n_heads + h] = tot + __ldg(P.b3 + h);
  }
}

// ---------------------------------------------------------------------------------------
// BiLSTM(20 -> 128) + PoolLastStepBi
struct LstmParams {
  const float* w_ih;   // [2][512][20]
  const float* w_hh;   // [2][512][128]
  const float* b;      // [2][512]   (bias_ih + bias_hh)
  const float* w_pool; // [256]
};

// One CTA advances NB clips of one direction in lock step, so that the recurrent weights
// (512 x 128 fp32 = 256 KB: half in registers, half in shared memory) are fetched once per step for NB sequences
// instead of once per sequence - the step is FMA bound (2 x 148 x NB FMAs per thread) instead of LDS / barrier bound,
// and 256 clips x 2 directions fit on the chip in ONE wave (one CTA per sequence needs 3.5 waves of 987 serial
// steps).  256 threads: thread t owns hidden unit u = t >> 1 and the gate pair gp = t & 1 ((i, f) or
// (g, o), PyTorch row order i, f, g, o), i.e. two rows of W_hh / W_ih; the pair of lanes of a unit exchanges its four
// gate values with two shuffles per sequence and both update the (replicated) cell state.  Sequences of a group may
// have different lengths (clips are sorted by length on the host): a finished sequence keeps its state.
// `order` lists the clips of the pass by decreasing n_seg; group g = clips order[NB g .. NB g + NB).
template <int NB>
__global__ void __launch_bounds__(256, 1)
lstm_batched_kernel(const float* __restrict__ feats /*[n_seg][20]*/, const ClipDesc* __restrict__ clips,
                    const int* __restrict__ order, int n_clips, LstmParams P,
                    float* __restrict__ td_out /*[n_seg][256] or nullptr*/, float* __restrict__ partial /*[n_clips][2]*/) {
  extern __shared__ __align__(16) float sm[];
  float2* whs = reinterpret_cast<float2*>(sm);       // [64 k][256 t]: taps 64..127 of this thread's two rows
  float* hbuf = sm + 2 * 64 * 256;                   // [2][NB][128]
  float* xbuf = hbuf + 2 * NB * 128;                 // [2][NB][32]   (20 used)
  float* red = xbuf + 2 * NB * 32;                   // [NB][128]
  const int t = threadIdx.x, u = t >> 1, gp = t & 1;
  const int dir = blockIdx.x & 1, g0 = (blockIdx.x >> 1) * NB;
  int S[NB], clip[NB];
  const float* fb[NB];
  size_t seg_off[NB];
  int maxS = 0;
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    clip[b] = (g0 + b < n_clips) ? __ldg(order + g0 + b) : -1;
    S[b] = 0; fb[b] = feats; seg_off[b] = 0;
    if (clip[b] >= 0) {
      const ClipDesc cd = clips[clip[b]];
      S[b] = cd.n_seg; seg_off[b] = (size_t)cd.seg_off; fb[b] = feats + (size_t)cd.seg_off * 20;
    }
    maxS = max(maxS, S[b]);
  }
  const int rowA = (2 * gp) * 128 + u, rowB = rowA + 128;
  float wrA[64], wrB[64], wiA[20], wiB[20];
  {
    const float* ra = P.w_hh + ((size_t)dir * 512 + rowA) * 128;
    const float* rb = P.w_hh + ((size_t)dir * 512 + rowB) * 128;
#pragma unroll
    for (int k = 0; k < 64; ++k) { wrA[k] = __ldg(ra + k); wrB[k] = __ldg(rb + k); }
    for (int k = 0; k < 64; ++k) whs[k * 256 + t] = make_float2(__ldg(ra + 64 + k), __ldg(rb + 64 + k));
    const float* ia = P.w_ih + ((size_t)dir * 512 + rowA) * 20;
    const float* ib = P.w_ih + ((size_t)dir * 512 + rowB) * 20;
#pragma unroll
    for (int k = 0; k < 20; ++k) { wiA[k] = __ldg(ia + k); wiB[k] = __ldg(ib + k); }
  }
  const float biasA = __ldg(P.b + dir * 512 + rowA), biasB = __ldg(P.b + dir * 512 + rowB);
  for (int i = t; i < 2 * NB * 128; i += 256) hbuf[i] = 0.f;
  for (int i = t; i < 2 * NB * 32; i += 256) xbuf[i] = 0.f;
  float cst[NB], hl[NB];
#pragma unroll
  for (int b = 0; b < NB; ++b) { cst[b] = 0.f; hl[b] = 0.f; }
  __syncthreads();
  // x of step 0: thread t < NB * 32 loads element (b = t >> 5, k = t & 31)
  const int xb_ = t >> 5, xk_ = t & 31;
  if (t < NB * 32 && xk_ < 20) {
    int Sb = 0; const float* f = feats;
#pragma unroll
    for (int b = 0; b < NB; ++b) if (b == xb_) { Sb = S[b]; f = fb[b]; }
    if (Sb > 0) xbuf[xb_ * 32 + xk_] = __ldg(f + (size_t)(dir ? Sb - 1 : 0) * 20 + xk_);
  }
  __syncthreads();

  for (int step = 0; step < maxS; ++step) {
    const float* h = hbuf + (step & 1) * NB * 128;
    const float* xt = xbuf + (step & 1) * NB * 32;
    float xnext = 0.f;
    bool xload = false;
    if (t < NB * 32 && xk_ < 20) {
      int Sb = 0; const float* f = feats;
#pragma unroll
      for (int b = 0; b < NB; ++b) if (b == xb_) { Sb = S[b]; f = fb[b]; }
      if (step + 1 < Sb) { xnext = __ldg(f + (size_t)(dir ? Sb - 2 - step : step + 1) * 20 + xk_); xload = true; }
    }
    // every row keeps two partial sums (even / odd taps), whatever NB is: a clip's result must not depend on how many
    // clips share its CTA (alone == in a batch, bit for bit), and one 148-long dependent FMA chain per row would
    // leave the NB = 1 variant latency bound
    constexpr int PART = 2;
    float pA[NB][PART], pB[NB][PART];
#pragma unroll
    for (int b = 0; b < NB; ++b)
#pragma unroll
      for (int q = 0; q < PART; ++q) { pA[b][q] = q ? 0.f : biasA; pB[b][q] = q ? 0.f : biasB; }
#pragma unroll
    for (int k = 0; k < 20; k += 4) {
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        const float4 xv = *reinterpret_cast<const float4*>(xt + b * 32 + k);
        pA[b][0] = fmaf(wiA[k], xv.x, pA[b][0]); pA[b][1 % PART] = fmaf(wiA[k + 1], xv.y, pA[b][1 % PART]);
        pA[b][2 % PART] = fmaf(wiA[k + 2], xv.z, pA[b][2 % PART]); pA[b][3 % PART] = fmaf(wiA[k + 3], xv.w, pA[b][3 % PART]);
        pB[b][0] = fmaf(wiB[k], xv.x, pB[b][0]); pB[b][1 % PART] = fmaf(wiB[k + 1], xv.y, pB[b][1 % PART]);
        pB[b][2 % PART] = fmaf(wiB[k + 2], xv.z, pB[b][2 % PART]); pB[b][3 % PART] = fmaf(wiB[k + 3], xv.w, pB[b][3 % PART]);
      }
    }
#pragma unroll
    for (int k = 0; k < 64; k += 4) {
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        const float4 hv = *reinterpret_cast<const float4*>(h + b * 128 + k);
        pA[b][0] = fmaf(wrA[k], hv.x, pA[b][0]); pA[b][1 % PART] = fmaf(wrA[k + 1], hv.y, pA[b][1 % PART]);
        pA[b][2 % PART] = fmaf(wrA[k + 2], hv.z, pA[b][2 % PART]); pA[b][3 % PART] = fmaf(wrA[k + 3], hv.w, pA[b][3 % PART]);
        pB[b][0] = fmaf(wrB[k], hv.x, pB[b][0]); pB[b][1 % PART] = fmaf(wrB[k + 1], hv.y, pB[b][1 % PART]);
        pB[b][2 % PART] = fmaf(wrB[k + 2], hv.z, pB[b][2 % PART]); pB[b][3 % PART] = fmaf(wrB[k + 3], hv.w, pB[b][3 % PART]);
      }
    }
#pragma unroll 4
    for (int k = 0; k < 64; k += 4) {
      const float2 w0 = whs[(k) * 256 + t], w1 = whs[(k + 1) * 256 + t], w2 = whs[(k + 2) * 256 + t], w3 = whs[(k + 3) * 256 + t];
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        const float4 hv = *reinterpret_cast<const float4*>(h + b * 128 + 64 + k);
        pA[b][0] = fmaf(w0.x, hv.x, pA[b][0]); pA[b][1 % PART] = fmaf(w1.x, hv.y, pA[b][1 % PART]);
        pA[b][2 % PART] = fmaf(w2.x, hv.z, pA[b][2 % PART]); pA[b][3 % PART] = fmaf(w3.x, hv.w, pA[b][3 % PART]);
        pB[b][0] = fmaf(w0.y, hv.x, pB[b][0]); pB[b][1 % PART] = fmaf(w1.y, hv.y, pB[b][1 % PART]);
        pB[b][2 % PART] = fmaf(w2.y, hv.z, pB[b][2 % PART]); pB[b][3 % PART] = fmaf(w3.y, hv.w, pB[b][3 % PART]);
      }
    }
    float aA[NB], aB[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      if (PART == 4) { aA[b] = (pA[b][0] + pA[b][1 % PART]) + (pA[b][2 % PART] + pA[b][3 % PART]); aB[b] = (pB[b][0] + pB[b][1 % PART]) + (pB[b][2 % PART] + pB[b][3 % PART]); }
      else if (PART == 2) { aA[b] = pA[b][0] + pA[b][1 % PART]; aB[b] = pB[b][0] + pB[b][1 % PART]; }
      else { aA[b] = pA[b][0]; aB[b] = pB[b][0]; }
    }
    float* hn = hbuf + ((step + 1) & 1) * NB * 128;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      // gp == 0: (aA, aB) = pre-activations of (i, f); gp == 1: of (g, o)
      const float actA = gp ? tanhf(aA[b]) : 1.0f / (1.0f + expf(-aA[b]));
      const float actB = 1.0f / (1.0f + expf(-aB[b]));
      const float pA = __shfl_xor_sync(0xffffffffu, actA, 1), pB = __shfl_xor_sync(0xffffffffu, actB, 1);
      const float ig = gp ? pA : actA, fg = gp ? pB : actB, gg = gp ? actA : pA, og = gp ? actB : pB;
      if (step < S[b]) {                       // warp-uniform: S[b] is the same for every thread
        cst[b] = fmaf(fg, cst[b], ig * gg);
        hl[b] = og * tanhf(cst[b]);
        if (gp == 0) {
          hn[b * 128 + u] = hl[b];
          if (td_out) td_out[(seg_off[b] + (size_t)(dir ? S[b] - 1 - step : step)) * 256 + dir * 128 + u] = hl[b];
        }
      } else if (gp == 0) {
        hn[b * 128 + u] = hl[b];               // finished sequence: state carried along unchanged
      }
    }
    if (xload) xbuf[((step + 1) & 1) * NB * 32 + xb_ * 32 + xk_] = xnext;
    __syncthreads();
  }
  // PoolLastStepBi: this direction's final hidden state . w_pool half (lib:1107-1115)
  if (gp == 0) {
    const float w = P.w_pool ? __ldg(P.w_pool + dir * 128 + u) : 0.f;      // (other pooling modes read td_out instead)
#pragma unroll
    for (int b = 0; b < NB; ++b) red[b * 128 + u] = hl[b] * w;
  }
  __syncthreads();
  if (t < 32 * NB) {
    const int b = t >> 5, lane = t & 31;
    float v = red[b * 128 + lane] + red[b * 128 + lane + 32] + red[b * 128 + lane + 64] + red[b * 128 + lane + 96];
    v = warp_sum(v);
    int cb = -1;
#pragma unroll
    for (int bb = 0; bb < NB; ++bb) if (bb == b) cb = clip[bb];
    if (lane == 0 && cb >= 0) partial[cb * 2 + dir] = v;      // clips without segments: 0 (lastbi_final writes NaN for them)
  }
}

__global__ void lastbi_final_kernel(const float* __restrict__ partial, const ClipDesc* __restrict__ clips,
                                    float bias, float* __restrict__ scores, int n_clips) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_clips) return;
  scores[c] = (clips[c].n_seg > 0) ? (partial[2 * c] + partial[2 * c + 1]) + bias
                                   : __int_as_float(0x7fc00000);
}

// ------------------------------------------------------------------ host launchers
constexpr int kRowSmem20 = (kRows * kXS + 64 * 20) * 4;

void launch_fc20(cudaStream_t st, const float* feats, const float* WT, const float* b, float* out, int n_rows) {
  linear_rows_kernel<20, false><<<(n_rows + kRows - 1) / kRows, kRows, kRowSmem20, st>>>(feats, 768, WT, b, nullptr, nullptr, out, n_rows);
}
void launch_pool_final(cudaStream_t st, const float* x, const float* logits, const ClipDesc* clips, int n_clips,
                       const PoolHeadParams& P, int n_heads, int max_seg, float* scores) {
  const int smem = n_heads * std::max(max_seg, 1) * 4;          // <= 5 x 1300 x 4 bytes at ms_max_segments = 1300
  if (smem > 40 * 1024) cudaFuncSetAttribute(pool_final_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  pool_final_kernel<<<n_clips, 64 * n_heads, smem, st>>>(x, logits, clips, P, n_heads, std::max(max_seg, 1), scores);
}
void launch_pool_simple(cudaStream_t st, const float* x, int D, const ClipDesc* clips, int n_clips, int mode,
                        const PoolSimpleParams& P, int n_heads, int max_seg, float* scores) {
  const int smem = (mode == 1 ? max_seg : 0) * 4 + 16;
  if (D == 64) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(pool_simple_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    pool_simple_kernel<64><<<n_clips, 64, smem, st>>>(x, clips, mode, P, n_heads, scores);
  } else {
    if (smem > 48 * 1024) cudaFuncSetAttribute(pool_simple_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    pool_simple_kernel<256><<<n_clips, 256, smem, st>>>(x, clips, mode, P, n_heads, scores);
  }
}

template <int NB> constexpr int lstm_batched_smem() { return (2 * 64 * 256 + 2 * NB * 128 + 2 * NB * 32 + NB * 128) * 4; }

// `order`: device array of the pass's clip indices sorted by decreasing n_seg (host-built, run_pass); the batch
// width follows the number of sequences per SM: 148 SMs x NB sequences per direction pair of CTAs in one wave
void launch_lstm_batched(cudaStream_t st, const float* feats20, const ClipDesc* clips, const int* order, int n_clips,
                         const LstmParams& P, float* td_out, float* partial, float pool_bias, float* scores) {
  static unsigned long long cfg = 0;
  if (first_launch_on_device(cfg)) {
    cudaFuncSetAttribute(lstm_batched_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lstm_batched_smem<1>());
    cudaFuncSetAttribute(lstm_batched_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lstm_batched_smem<2>());
    cudaFuncSetAttribute(lstm_batched_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, lstm_batched_smem<4>());
  }
  const int seqs = 2 * n_clips;
  if (seqs <= 148)
    lstm_batched_kernel<1><<<2 * n_clips, 256, lstm_batched_smem<1>(), st>>>(feats20, clips, order, n_clips, P, td_out, partial);
  else if (seqs <= 2 * 148)
    lstm_batched_kernel<2><<<2 * ((n_clips + 1) / 2), 256, lstm_batched_smem<2>(), st>>>(feats20, clips, order, n_clips, P, td_out, partial);
  else
    lstm_batched_kernel<4><<<2 * ((n_clips + 3) / 4), 256, lstm_batched_smem<4>(), st>>>(feats20, clips, order, n_clips, P, td_out, partial);
  if (scores) lastbi_final_kernel<<<(n_clips + 127) / 128, 128, 0, st>>>(partial, clips, pool_bias, scores, n_clips);
}

}  // namespace nisqa
