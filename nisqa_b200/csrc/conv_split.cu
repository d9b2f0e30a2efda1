// conv_split.cu - conv3..conv6 of the AdaptCNN / StandardCNN (reference nisqa/NISQA_lib.py:696-706,
// 820-830) as implicit GEMMs on the 5th-generation tensor cores (tcgen05 + TMEM), with the activations
// travelling BETWEEN the layers already in the form the tensor core consumes.
//
// Arithmetic: an error-compensated two-term FP16 split, so that the result stays within fp32 rounding
// noise of the reference (plain TF32 / BF16 operands move MOS by 2e-3 / 1.7e-2, SURVEY.md 0.8):
//      a = a_hi + a_lo,  b = b_hi + b_lo      (fp16 parts: 11 + 11 significant bits)
//      a*b ~= a_hi*b_hi + a_hi*b_lo + a_lo*b_hi          (dropped a_lo*b_lo ~ 2^-22 |a b|)
// Issued as TWO MMAs per K-step: A_hi x [B_hi | B_lo] with N = 2*C_out (accumulator columns
// [0,C) = hi*hi, [C,2C) = hi*lo) and A_lo x B_hi with N = C_out into columns [C,2C) as well; the
// epilogue adds the two column halves.  Every A element is thus fetched from shared memory twice per
// tap instead of three times.  Products are exact in the tensor core and accumulate in fp32 (TMEM).
// The weights are pre-scaled by 2^S on the host (S chosen per layer so that max|w| 2^S <= 1024) to
// keep b_lo out of the fp16 subnormal range; the epilogue multiplies by 2^-S (exact).  Compared with
// 3xTF32 this halves shared memory, weight traffic and MMA time (kind::f16 has K = 16).
//
// GEMM view:  D[pos, co] = sum_{tap, ci} X[pos + off(tap), ci] * W[tap][co][ci]
//   M = flattened padded positions of G segments, N = C_out, K = 9 * C_in.  The 9 taps are the SAME
//   activation tile addressed through row-shifted descriptors, so im2col is never materialised.
//
// The activations are two fp16 planes (hi, lo) laid out in HBM as the exact shared-memory image of the
// implicit-GEMM A tile:
//
//   plane row g(seg, hh, ww) = kSplitLead + seg * BLK + hh * P + ww,   P = W + 1, BLK = (H + 1) * P
//     hh = 0 / ww = 0 are the shared zero row / zero column (never written: the planes are zeroed
//     when they are allocated), interior positions are hh = h + 1, ww = w + 1
//   row = CIN halves (32 / 64 / 128 bytes); the 16-byte chunk c of row g sits at chunk position
//     c ^ f(g), f = the hardware 32B / 64B / 128B swizzle of a tile whose row index is == g (mod 8)
//
// so that a CTA's whole activation tile (256 + 2 * HALO consecutive rows, two planes) arrives with
// TWO cp.async.bulk copies issued by one thread (placed at row offset g0 & 7 inside a 1024-byte
// aligned tile so that the absolute-address swizzle of the UMMA descriptors matches the image), and
// the producing layer's epilogue does the split once, right where the fp32 value exists.
#include <cuda_fp16.h>

#include <algorithm>

#include "common.cuh"
#include "tc_ptx.cuh"
#include "conv_split.cuh"

namespace nisqa {

// Persistent, warp-specialised kernel.  Measured on B200 (profiles/r02b_mma_probe_issuers.txt): one issuing thread
// retires a M=128 K=16 MMA every ~96 cycles whatever N is; two issuers (two CTAs, or two warps of one CTA) overlap
// until the pipe's own floor binds (N=128: 64 cycles = 8 KB of operands at 128 B/clk; N=64: 48 cycles, operand-fetch
// bound).  A CTA that runs one tile and exits leaves the tensor pipe idle during fill, epilogue and teardown (47 % of
// the time on conv4).  Here ONE CTA per SM stays resident and walks over its tiles with every phase overlapped:
//
//   warps 0..7   epilogue of tile i-1 (TMEM -> registers -> staging -> pool / split -> HBM)
//   warp  8      producer: activation tile of tile i+1 (two bulk copies) as soon as its buffer is free
//   warp  9      producer: weights, tap by tap through a ring (or ONCE, when all nine taps fit: conv3)
//   warps 10,11  MMA issuers of tile i, one per M-tile (two issuers reach the pipe's rate, one does not)
//
// Two activation buffers and two accumulator sets (2 x 4 C_out TMEM columns) alternate; the epilogue stages its
// tile in the activation buffer it has just finished with, so a buffer returns to the producer when the tile's
// output has left it.
//
// -DNISQA_TC_TIMING: each layer L (3..6) accumulates per-CTA cycle counters in its own block of g_pipe_timing
// (tools/pipe_timing.py).
#ifdef NISQA_TC_TIMING
__device__ long long g_pipe_timing[4 * 256 * 16];   // [layer - 3][CTA][slot]
#define PIPE_NOW() clock64()
#define PIPE_ADD(slot, t0) do { if (blockIdx.x < 256) g_pipe_timing[((L - 3) * 256 + blockIdx.x) * 16 + (slot)] += clock64() - (t0); } while (0)
#define PIPE_COUNT(slot, n) do { if (blockIdx.x < 256) g_pipe_timing[((L - 3) * 256 + blockIdx.x) * 16 + (slot)] += (n); } while (0)
#else
#define PIPE_NOW() 0ll
#define PIPE_ADD(slot, t0) do { (void)(t0); } while (0)
#define PIPE_COUNT(slot, n) do { } while (0)
#endif

template <class C>
struct PipeCfg {
  static constexpr int NT = 12 * 32;
  static constexpr int STG_BYTES = (C::POOL != SP_POOL_NONE) ? C::G * C::H * C::W * C::STG_STRIDE * 4
                                                             : (C::OUT_SPLIT ? 2 : 1) * C::IMG_BYTES;
  static constexpr int BUF_RAW = (2 * C::A_BYTES > STG_BYTES) ? 2 * C::A_BYTES : STG_BYTES;
  static constexpr int BUF_BYTES = (BUF_RAW + 1023) & ~1023;
  static constexpr int AB_BYTES = 2 * BUF_BYTES;                       // two activation buffers (also the staging tiles)
  static constexpr bool RESIDENT = AB_BYTES + 9 * C::B_STAGE <= 196 * 1024;     // all nine taps stay in shared memory
  static constexpr int NSW = RESIDENT ? 9 : ((AB_BYTES + 4 * C::B_STAGE <= 216 * 1024) ? 4 : 3);
  static constexpr int OFF_B = AB_BYTES;
  static constexpr int OFF_BAR = OFF_B + NSW * C::B_STAGE;
  static constexpr int N_BAR = 2 + 2 + 2 * NSW + 2 + 2 + 2;
  static constexpr int SMEM_BYTES = OFF_BAR + 8 * N_BAR + 32 + 1024;
  static constexpr int COLS_TILE = 4 * C::COUT;                        // 2 M-tiles x [hi*hi+lo*hi | hi*lo]
  static constexpr int TMEM_ALLOC = 2 * COLS_TILE;                     // 512 (C_out 64) / 256 (C_out 32): powers of two
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
  static_assert(TMEM_ALLOC == 256 || TMEM_ALLOC == 512, "TMEM allocation");
};

template <class C, int L>
__global__ void __launch_bounds__(PipeCfg<C>::NT, 1)
conv_pipe_kernel(const unsigned char* __restrict__ in_hi, const unsigned char* __restrict__ in_lo,
                 const __half* __restrict__ wtc, const float* __restrict__ bias, float out_scale,
                 unsigned char* __restrict__ out_hi, unsigned char* __restrict__ out_lo,
                 float* __restrict__ out_f32, int n_seg, int n_tiles) {
  using Pc = PipeCfg<C>;
  constexpr int H = C::H, W = C::W, CIN = C::CIN, COUT = C::COUT, P = C::P, BLK = C::BLK, G = C::G;
  constexpr int HALO = C::HALO, ROWB = C::ROWB, NSW = Pc::NSW;
  constexpr int EPI_THREADS = 256;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t sbase = smem_u32(smem);
  const uint32_t b_base = sbase + Pc::OFF_B;
  const uint32_t bar0 = sbase + Pc::OFF_BAR;
  const uint32_t bar_a_full = bar0, bar_a_free = bar0 + 16, bar_b_full = bar0 + 32, bar_b_empty = bar_b_full + 8 * NSW;
  const uint32_t bar_acc_full = bar_b_empty + 8 * NSW, bar_acc_free = bar_acc_full + 16, bar_stage_ready = bar_acc_free + 16;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + Pc::OFF_BAR + 8 * Pc::N_BAR + 8);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), Pc::TMEM_ALLOC);
  if (tid == 256) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_a_full + 8 * i, 1); mbar_init(bar_a_free + 8 * i, 1);
      mbar_init(bar_acc_full + 8 * i, 2);          // both MMA issuers commit
      mbar_init(bar_acc_free + 8 * i, 8);          // one arrival per epilogue warp
      mbar_init(bar_stage_ready + 8 * i, 8);       // un-pooled layers: the staged output image is complete
    }
    for (int i = 0; i < NSW; ++i) { mbar_init(bar_b_full + 8 * i, 1); mbar_init(bar_b_empty + 8 * i, 2); }
    fence_barrier_init();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 8) {
    // ===== producer A: activation tile of every tile this CTA owns, two buffers ahead of the epilogue.  For the
    // un-pooled layers it also ships the staged output image of tile it-2 (bulk stores) out of the buffer it is
    // about to refill - the epilogue warps never wait for a store =====
    if (lane == 0) {
      constexpr uint32_t A_COPY = (uint32_t)C::AROWS * ROWB;
      auto store_tile = [&](int j) {
        const int b = j & 1;
        mbar_wait(bar_stage_ready + 8 * b, (j >> 1) & 1);          // all eight epilogue warps have staged tile j
        const int seg0 = (blockIdx.x + j * (int)gridDim.x) * G;
        const int nvalid = min(G, n_seg - seg0);
        const uint32_t sb = sbase + b * Pc::BUF_BYTES;
        if constexpr (C::OUT_SPLIT) {
          const size_t img0 = (size_t)(kSplitLead + seg0 * BLK) * C::OROWB;
          const uint32_t bytes = (uint32_t)nvalid * C::OBLK * C::OROWB;
          bulk_s2g(out_hi + img0, sb, bytes);
          bulk_s2g(out_lo + img0, sb + C::IMG_BYTES, bytes);
        } else {
          const uint32_t per_seg = C::HO * C::WO * COUT * 4;
          bulk_s2g(out_f32 + (size_t)seg0 * (per_seg / 4), sb, (uint32_t)nvalid * per_seg);
        }
        bulk_commit();
        bulk_wait_read0();                                         // the stores have read the buffer
      };
      int it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1, ph = (it >> 1) & 1;
        const long long tw = PIPE_NOW();
        if constexpr (C::POOL == SP_POOL_NONE) { if (it >= 2) store_tile(it - 2); }
        else mbar_wait(bar_a_free + 8 * buf, ph ^ 1);              // the pooling epilogue of tile it-2 has left the buffer
        PIPE_ADD(9, tw);
        const int g0 = kSplitLead + tile * G * BLK - HALO;
        const uint32_t sh = (uint32_t)(g0 & 7);
        const uint32_t a_hi = sbase + buf * Pc::BUF_BYTES, a_lo = a_hi + C::A_BYTES;
        mbar_expect_tx(bar_a_full + 8 * buf, 2 * A_COPY);
        bulk_g2s(a_hi + sh * ROWB, in_hi + (size_t)g0 * ROWB, A_COPY, bar_a_full + 8 * buf);
        bulk_g2s(a_lo + sh * ROWB, in_lo + (size_t)g0 * ROWB, A_COPY, bar_a_full + 8 * buf);
      }
      if constexpr (C::POOL == SP_POOL_NONE)
        for (int j = (it >= 2 ? it - 2 : 0); j < it; ++j) store_tile(j);
    }
  } else if (warp == 9) {
    // ===== producer W: the nine weight taps per tile through the ring (once, when they all stay resident) =====
    if (lane == 0) {
      int cnt = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (int t = 0; t < 9; ++t, ++cnt) {
          if (Pc::RESIDENT && cnt >= 9) continue;
          const int s = cnt % NSW;
          const long long tw = PIPE_NOW();
          if (!Pc::RESIDENT) mbar_wait(bar_b_empty + 8 * s, ((cnt / NSW) & 1) ^ 1);
          PIPE_ADD(11, tw);
          mbar_expect_tx(bar_b_full + 8 * s, C::B_STAGE);
          bulk_g2s(b_base + s * C::B_STAGE, wtc + (size_t)t * (C::B_STAGE / 2), C::B_STAGE, bar_b_full + 8 * s);
        }
      }
    }
  } else if (warp >= 10) {
    // ===== MMA issuers: warp 10 owns M-tile 0, warp 11 M-tile 1 =====
    if (lane == 0) {
      const int mt = warp - 10;
      int it = 0, cnt = 0;
      const long long t_all = PIPE_NOW();
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1, ph = (it >> 1) & 1;
        long long tw = PIPE_NOW();
        mbar_wait(bar_acc_free + 8 * buf, ph ^ 1);         // accumulators of tile it-2 drained
        if (mt == 0) PIPE_ADD(0, tw);
        tw = PIPE_NOW();
        mbar_wait(bar_a_full + 8 * buf, ph);
        if (mt == 0) PIPE_ADD(1, tw);
        tc_fence_after();
        const int g0 = kSplitLead + tile * G * BLK - HALO;
        const uint32_t sh = (uint32_t)(g0 & 7);
        const uint32_t a_hi = sbase + buf * Pc::BUF_BYTES, a_lo = a_hi + C::A_BYTES;
        const uint32_t d = tmem + buf * Pc::COLS_TILE + mt * (2 * COUT);
        for (int t = 0; t < 9; ++t, ++cnt) {
          const int s = Pc::RESIDENT ? t : cnt % NSW;
          tw = PIPE_NOW();
          if (!Pc::RESIDENT || it == 0) {                  // (an already completed barrier still costs ~150 cycles to ask)
            mbar_wait(bar_b_full + 8 * s, Pc::RESIDENT ? 0 : (cnt / NSW) & 1);
            tc_fence_after();
          }
          if (mt == 0) PIPE_ADD(2, tw);
          const int tapoff = (t / 3 - 1) * P + (t % 3 - 1);
          const uint32_t bst = b_base + s * C::B_STAGE;
          const uint32_t row = sh + (uint32_t)(HALO + mt * 128 + tapoff);
#pragma unroll
          for (int ks = 0; ks < CIN / 16; ++ks) {
            const uint64_t db = make_desc(bst + (uint32_t)(2 * ks) * (2 * COUT * 16), 2 * COUT * 16, 128);
            const uint32_t aoff = row * ROWB + (uint32_t)ks * 32;
            umma_f16(d, make_desc_swz(a_hi + aoff, 8 * ROWB, C::LAYOUT), db, C::IDESC_2N, (t | ks) != 0);   // [0,C) += hi*hi ; [C,2C) += hi*lo
            umma_f16(d + COUT, make_desc_swz(a_lo + aoff, 8 * ROWB, C::LAYOUT), db, C::IDESC_1N, 1);        // [C,2C) += lo*hi (small accumulator)
          }
          if (!Pc::RESIDENT) umma_commit(bar_b_empty + 8 * s);
        }
        umma_commit(bar_acc_full + 8 * buf);
      }
      if (mt == 0) { PIPE_ADD(4, t_all); PIPE_COUNT(15, it); }
    }
  } else {
    // ===== epilogue: warp w drains TMEM lanes 32 (w & 3) .. +31 of M-tile w >> 2 =====
    const int quarter = warp & 3, mt = warp >> 2;
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1, ph = (it >> 1) & 1;
      const int seg0 = tile * G;
      unsigned char* sbuf = smem + buf * Pc::BUF_BYTES;          // staging = the tile's own activation buffer
      float* stg = reinterpret_cast<float*>(sbuf);
      long long tw = PIPE_NOW();
      mbar_wait(bar_acc_full + 8 * buf, ph);                     // every MMA of the tile has retired
      if (tid == 0) PIPE_ADD(5, tw);
      tw = PIPE_NOW();
      tc_fence_after();
      {
        const int r = mt * 128 + quarter * 32 + lane;
        const int s = r / BLK, q = r - s * BLK;
        const int hh = q / P, ww = q - hh * P;
        const bool live = (s < G) && (seg0 + s < n_seg);
        bool valid = live && hh >= 1 && ww >= 1;
        if (C::CENTER) valid = valid && (ww == 2);
        const uint32_t trow = tmem + ((uint32_t)(quarter * 32) << 16) + buf * Pc::COLS_TILE + mt * (2 * COUT);
#pragma unroll 1
        for (int c16 = 0; c16 < COUT / 16; ++c16) {
          uint32_t ra[16], rb[16];
          tmem_ld16_nowait(trow + c16 * 16, ra);
          tmem_ld16_nowait(trow + COUT + c16 * 16, rb);
          tmem_ld_wait();
          float v[16];
          const float4* b4 = reinterpret_cast<const float4*>(bias + c16 * 16);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 bb = __ldg(b4 + j);
            v[4 * j + 0] = fmaxf(fmaf(__uint_as_float(ra[4 * j + 0]) + __uint_as_float(rb[4 * j + 0]), out_scale, bb.x), 0.f);
            v[4 * j + 1] = fmaxf(fmaf(__uint_as_float(ra[4 * j + 1]) + __uint_as_float(rb[4 * j + 1]), out_scale, bb.y), 0.f);
            v[4 * j + 2] = fmaxf(fmaf(__uint_as_float(ra[4 * j + 2]) + __uint_as_float(rb[4 * j + 2]), out_scale, bb.z), 0.f);
            v[4 * j + 3] = fmaxf(fmaf(__uint_as_float(ra[4 * j + 3]) + __uint_as_float(rb[4 * j + 3]), out_scale, bb.w), 0.f);
          }
          if constexpr (C::POOL != SP_POOL_NONE) {
            if (valid) {
              float4* dst = reinterpret_cast<float4*>(stg + ((s * H + (hh - 1)) * W + (ww - 1)) * C::STG_STRIDE + c16 * 16);
#pragma unroll
              for (int j = 0; j < 4; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
          } else if constexpr (C::OUT_SPLIT) {
            if (live) {
              const int g = kSplitLead + seg0 * BLK + r;
              const size_t img0 = (size_t)(kSplitLead + seg0 * BLK) * C::OROWB;
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                uint4 hi = make_uint4(0u, 0u, 0u, 0u), lo = hi;
                if (valid)
                  split8(make_float4(v[8 * j], v[8 * j + 1], v[8 * j + 2], v[8 * j + 3]),
                         make_float4(v[8 * j + 4], v[8 * j + 5], v[8 * j + 6], v[8 * j + 7]), hi, lo);
                const uint32_t o = (uint32_t)(split_off<C::OROWB>(g, c16 * 2 + j) - img0);
                *reinterpret_cast<uint4*>(sbuf + o) = hi;
                *reinterpret_cast<uint4*>(sbuf + C::IMG_BYTES + o) = lo;
              }
            }
          } else {
            if (valid) {
              const int w = C::CENTER ? 0 : ww - 1;
              float4* dst = reinterpret_cast<float4*>(stg + ((s * H + (hh - 1)) * C::WO + w) * COUT + c16 * 16);
#pragma unroll
              for (int j = 0; j < 4; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_free + 8 * buf);          // this warp's share of the accumulators is in shared memory
      if constexpr (C::POOL == SP_POOL_NONE) {
        fence_proxy_async();                                       // staged image -> visible to the producer's bulk stores
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_stage_ready + 8 * buf);
        if (tid == 0) PIPE_ADD(6, tw);
      } else {
        if (tid == 0) PIPE_ADD(6, tw);
        tw = PIPE_NOW();
        named_bar_sync(1, EPI_THREADS);                            // staging tile complete (epilogue warps only)
        constexpr int POW = C::POW, HO = H / 2, C8 = COUT / 8;
        for (int i2 = tid; i2 < G * HO * POW * C8; i2 += EPI_THREADS) {
          const int c8 = i2 % C8;
          int rest = i2 / C8;
          const int pw = rest % POW; rest /= POW;
          const int ph2 = rest % HO;
          const int s = rest / HO;
          if (seg0 + s >= n_seg) continue;
          int x0, x1;
          if (C::POOL == SP_POOL_ADAPT) { x0 = (pw * W) / POW; x1 = ((pw + 1) * W + POW - 1) / POW; }
          else { x0 = 2 * pw; x1 = 2 * pw + 2; }
          float4 ma = make_float4(0.f, 0.f, 0.f, 0.f), mb = ma;     // post-ReLU values are >= 0
          for (int hy = 2 * ph2; hy < 2 * ph2 + 2; ++hy)
            for (int x = x0; x < x1; ++x) {
              const float4* tp = reinterpret_cast<const float4*>(stg + ((s * H + hy) * W + x) * C::STG_STRIDE + c8 * 8);
              const float4 ta = tp[0], tb = tp[1];
              ma.x = fmaxf(ma.x, ta.x); ma.y = fmaxf(ma.y, ta.y); ma.z = fmaxf(ma.z, ta.z); ma.w = fmaxf(ma.w, ta.w);
              mb.x = fmaxf(mb.x, tb.x); mb.y = fmaxf(mb.y, tb.y); mb.z = fmaxf(mb.z, tb.z); mb.w = fmaxf(mb.w, tb.w);
            }
          uint4 hi, lo;
          split8(ma, mb, hi, lo);
          const int g = kSplitLead + (seg0 + s) * C::OBLK + (ph2 + 1) * C::OP + (pw + 1);
          const size_t o = split_off<C::OROWB>(g, c8);
          *reinterpret_cast<uint4*>(out_hi + o) = hi;
          *reinterpret_cast<uint4*>(out_lo + o) = lo;
        }
        named_bar_sync(2, EPI_THREADS);                            // every thread has read its part of the staging tile
        if (tid == 0) { mbar_arrive(bar_a_free + 8 * buf); PIPE_ADD(7, tw); }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, Pc::TMEM_ALLOC);
}

// planes -> fp32 channels-last [seg][H][W][C] (stage dumps for the parity tests; x_hi + x_lo == x to 2^-22)
template <int ROWB>
__global__ void unsplit_kernel(const unsigned char* __restrict__ hi, const unsigned char* __restrict__ lo,
                               float* __restrict__ out, long long n_items, int H, int W) {
  constexpr int C8 = ROWB / 16;
  const int P = W + 1, BLK = (H + 1) * P;
  for (long long it = (long long)blockIdx.x * blockDim.x + threadIdx.x; it < n_items; it += (long long)gridDim.x * blockDim.x) {
    const int c8 = (int)(it % C8);
    long long rest = it / C8;
    const int w = (int)(rest % W); rest /= W;
    const int h = (int)(rest % H);
    const int seg = (int)(rest / H);
    const int g = kSplitLead + seg * BLK + (h + 1) * P + (w + 1);
    const size_t o = split_off<ROWB>(g, c8);
    const uint4 a = *reinterpret_cast<const uint4*>(hi + o), b = *reinterpret_cast<const uint4*>(lo + o);
    const __half2* ah = reinterpret_cast<const __half2*>(&a);
    const __half2* bh = reinterpret_cast<const __half2*>(&b);
    float r[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 x = __half22float2(ah[i]), y = __half22float2(bh[i]);
      r[2 * i] = x.x + y.x; r[2 * i + 1] = x.y + y.y;
    }
    float4* dst = reinterpret_cast<float4*>(out + it * 8);
    dst[0] = make_float4(r[0], r[1], r[2], r[3]);
    dst[1] = make_float4(r[4], r[5], r[6], r[7]);
  }
}


template <class C, int L>
static void launch_pipe(cudaStream_t st, const unsigned char* in_hi, const unsigned char* in_lo, const __half* wtc,
                        const float* b, float scale, unsigned char* out_hi, unsigned char* out_lo, float* out_f32,
                        int n_seg) {
  using Pc = PipeCfg<C>;
  static unsigned long long configured = 0;
  static int n_sm = 0;
  if (first_launch_on_device(configured)) {
    cudaFuncSetAttribute(conv_pipe_kernel<C, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, Pc::SMEM_BYTES);
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  }
  const int n_tiles = (n_seg + C::G - 1) / C::G;
  const int grid = std::min(n_tiles, n_sm > 0 ? n_sm : 148);
  conv_pipe_kernel<C, L><<<grid, Pc::NT, Pc::SMEM_BYTES, st>>>(in_hi, in_lo, wtc, b, scale, out_hi, out_lo, out_f32, n_seg, n_tiles);
}

// Geometry of the plane pair that feeds conv layer `layer` (2..6): rows of the padded image per segment,
// bytes per row, and the bytes of one plane for n_seg segments (tile over-read included).
void split_geometry(int std_mode, int layer, int* H, int* W, int* C) {
  static const int ha[7] = {0, 0, 24, 12, 12, 6, 6}, ca[7] = {0, 0, 16, 32, 64, 64, 64};
  static const int wa[7] = {0, 0, 7, 5, 5, 3, 3}, ws[7] = {0, 0, 8, 4, 4, 2, 2};
  *H = ha[layer]; *C = ca[layer]; *W = std_mode ? ws[layer] : wa[layer];
}
size_t split_plane_bytes(int std_mode, int layer, int n_seg) {
  int H, W, C;
  split_geometry(std_mode, layer, &H, &W, &C);
  const size_t rows = (size_t)kSplitLead + (size_t)n_seg * (H + 1) * (W + 1) + 256 + 32;
  return (rows * (size_t)C * 2 + 1023) & ~(size_t)1023;
}

// conv layer 3..6 on planes; the last layer (6) writes the fp32 CNN features (adapt: [seg][6][64];
// standard: [seg][6][2][64])
void launch_conv_split(cudaStream_t st, int std_mode, int layer, const void* in_hi, const void* in_lo,
                       const void* wtc, const float* b, float out_scale, void* out_hi, void* out_lo,
                       float* out_f32, int n_seg) {
  const __half* w = reinterpret_cast<const __half*>(wtc);
  const unsigned char* ih = static_cast<const unsigned char*>(in_hi);
  const unsigned char* il = static_cast<const unsigned char*>(in_lo);
  unsigned char* oh = static_cast<unsigned char*>(out_hi);
  unsigned char* ol = static_cast<unsigned char*>(out_lo);
  if (!std_mode) {
    switch (layer) {
      case 3: launch_pipe<SpConv3A, 3>(st, ih, il, w, b, out_scale, oh, ol, out_f32, n_seg); break;
      case 4: launch_pipe<SpConv4A, 4>(st, ih, il, w, b, out_scale, oh, ol, out_f32, n_seg); break;
      case 5: launch_pipe<SpConv5A, 5>(st, ih, il, w, b, out_scale, oh, ol, out_f32, n_seg); break;
      default: launch_pipe<SpConv6A, 6>(st, ih, il, w, b, out_scale, oh, ol, out_f32, n_seg); break;
    }
  } else {
    switch (layer) {
      case 3: launch_pipe<SpConv3S, 3>(st, ih, il, w, b, out_scale, oh, ol, out_f32, n_seg); break;
      case 4: launch_pipe<SpConv4S, 4>(st, ih, il, w, b, out_scale, oh, ol, out_f32, n_seg); break;
      case 5: launch_pipe<SpConv5S, 5>(st, ih, il, w, b, out_scale, oh, ol, out_f32, n_seg); break;
      default: launch_pipe<SpConv6S, 6>(st, ih, il, w, b, out_scale, oh, ol, out_f32, n_seg); break;
    }
  }
}

void launch_unsplit(cudaStream_t st, int std_mode, int layer, const void* hi, const void* lo, float* out, int n_seg) {
  int H, W, C;
  split_geometry(std_mode, layer, &H, &W, &C);
  const long long items = (long long)n_seg * H * W * (C / 8);
  const unsigned char* h = static_cast<const unsigned char*>(hi);
  const unsigned char* l = static_cast<const unsigned char*>(lo);
  const int grid = (int)std::min<long long>((items + 255) / 256, 148 * 16);
  if (C == 16) unsplit_kernel<32><<<grid, 256, 0, st>>>(h, l, out, items, H, W);
  else if (C == 32) unsplit_kernel<64><<<grid, 256, 0, st>>>(h, l, out, items, H, W);
  else unsplit_kernel<128><<<grid, 256, 0, st>>>(h, l, out, items, H, W);
}

#ifdef NISQA_TC_TIMING
int pipe_timing_read(long long* host, int n, int reset) {
  int rc = (int)cudaMemcpyFromSymbol(host, g_pipe_timing, sizeof(long long) * n);
  if (reset) { static long long zero[4 * 256 * 16]; cudaMemcpyToSymbol(g_pipe_timing, zero, sizeof zero); }
  return rc;
}
#endif

}  // namespace nisqa
