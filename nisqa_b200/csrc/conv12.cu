// conv12.cu - conv1 + pool1 + conv2 + pool2 of the framewise CNN in ONE persistent kernel.
//
// Writing pool1 to HBM as fp16 plane pairs and reading it back for conv2 would cost 123 + 202 MB per 64-clip step
// (21 % of the CNN's DRAM traffic) and two launches whose CTAs spend most of their life filling / draining.  Here the
// pool1 tile of a segment never leaves the SM: producer warps compute conv1 + BN + ReLU + pool1 of segment i+1 straight into the shared-memory image of
// conv2's implicit-GEMM A operand (the plane layout of conv_split.cuh: padded rows of 16 halves, 32-byte swizzle,
// hi / lo split) while the tensor pipe runs conv2 of segment i and the epilogue warps pool / split / store segment
// i-1.  Reference: nisqa/NISQA_lib.py:688-695 (AdaptCNN) / 811-818 (StandardCNN).
//
//   warps 0..7    epilogue: TMEM -> bias / ReLU -> staging -> max-pool -> fp16 hi / lo planes of pool2 (conv3's input)
//   warps 8..15   producers: one thread per pooled cell (24 x 7 or 24 x 8; a warp owns three pooled rows), all 16 channels
//                 (NISQA_C12_GROUPS = 2 splits the channels over two groups of eight warps: measured, no gain)
//                 (conv1_cell.cuh, packed FFMA2).  Lanes run along the pooled columns: consecutive plane rows, so that
//                 the 16-byte stores into the swizzled A image are bank-conflict free
//   warp  16      loads conv2's weights (all nine taps stay resident: 18 KB) and stages every segment's 15 mel rows
//                 (192 bytes each, padded to a pitch of 52 floats: the producers' patch reads spread over the banks)
//                 into a four-slot shared-memory ring with bulk copies, several tiles ahead: the producers never wait
//                 for global memory
//   warps 17,18   MMA issuers, one per M-tile (two issuers reach the tensor pipe's rate, one does not)
//
// One tile = one segment (its padded 25 x 8 / 25 x 9 map is 200 / 225 of the 256 GEMM rows).  Three A buffers, two
// accumulator sets, two staging tiles.  conv2 uses the two-term fp16 split of conv_split.cu and the same MMA order per
// accumulator as conv_pipe_kernel; conv1 is conv1_cell, which conv1_pool1_kernel (conv1.cu) shares to dump pool1.
#include <algorithm>
#include <type_traits>

#include "conv1_cell.cuh"
#include "conv_split.cuh"

namespace nisqa {

#ifdef NISQA_TC_TIMING
__device__ long long g_c12_timing[256 * 16];        // per CTA: cycles accumulated per role / wait (tools/pipe_timing.py)
#define C12_NOW() clock64()
#define C12_ADD(slot, t0) do { if (blockIdx.x < 256) g_c12_timing[blockIdx.x * 16 + (slot)] += clock64() - (t0); } while (0)
#define C12_COUNT(slot, n) do { if (blockIdx.x < 256) g_c12_timing[blockIdx.x * 16 + (slot)] += (n); } while (0)
#else
#define C12_NOW() 0ll
#define C12_ADD(slot, t0) do { (void)(t0); } while (0)
#define C12_COUNT(slot, n) do { } while (0)
#endif

template <int MODE>
struct C12Cfg {
  using C = typename std::conditional<MODE == 0, SpConv2A, SpConv2S>::type;
  static constexpr int PW = C::W;                       // pooled width of conv1's output = conv2's input width
  static constexpr int NCELL = 24 * PW;                 // producer threads with work
#ifndef NISQA_C12_GROUPS
#define NISQA_C12_GROUPS 1      // producer warp groups: 2 = the 16 conv1 channels split over two groups of eight warps (measured: no gain, profiles/r02v_ab_kernels.txt)
#endif
  static constexpr int N_GROUPS = NISQA_C12_GROUPS;     // each group computes 16 / N_GROUPS channels of every cell
  static constexpr int N_PROD_WARPS = 8 * N_GROUPS;
  static constexpr int CPW = 3 * PW;                    // cells per producer warp: three pooled rows
  static_assert(CPW <= 32 && 8 * CPW == NCELL && (N_GROUPS == 1 || N_GROUPS == 2), "a warp owns three pooled rows");
  static constexpr int NT = (8 + N_PROD_WARPS + 1 + 2) * 32;
  static constexpr int W_PROD0 = 8, W_LOAD = 8 + N_PROD_WARPS, W_MMA0 = W_LOAD + 1;
  static constexpr int NA = 3;                          // A buffers (hi + lo tile each)
  static constexpr int BUF_BYTES = 2 * C::A_BYTES;
  static constexpr int STG_BYTES = (C::G * C::H * C::W * C::STG_STRIDE * 4 + 1023) & ~1023;
  static constexpr int OFF_STG = NA * BUF_BYTES;
  static constexpr int NSTG = 2;                        // staging tiles: a warp starts draining tile i+1 while others still pool tile i
  static constexpr int OFF_B = OFF_STG + NSTG * STG_BYTES;
  static constexpr int B_BYTES = 9 * C::B_STAGE;
  static constexpr int OFF_W1 = OFF_B + B_BYTES;        // conv1: [9][16] weights + 16 biases (fp32)
  static constexpr int NM = 4;                          // mel slots (one segment = kSegLen x kMels fp32 = 2880 bytes)
  static constexpr int MEL_BYTES = kSegLen * kMels * 4;
  static constexpr int MEL_PITCH = 52;                  // floats per staged mel row: 16-byte aligned rows, 2 * 52 = 8 banks (mod 32) per pooled column
  static constexpr int MEL_SLOT = (kSegLen * MEL_PITCH * 4 + 127) & ~127;
  static constexpr int OFF_MEL = OFF_W1 + 1024;
  static constexpr int OFF_BAR = OFF_MEL + NM * MEL_SLOT;
  static constexpr int N_BAR = 2 * NA + 2 + 2 + 1 + 2 * NM;
  static constexpr int SMEM_BYTES = OFF_BAR + 8 * N_BAR + 32 + 1024;
  static constexpr int COLS_TILE = 4 * C::COUT;         // 128
  static constexpr int TMEM_ALLOC = 2 * COLS_TILE;      // 256
  static_assert(C::G == 1, "one segment per tile");
  static_assert(C::A_BYTES % 1024 == 0 && TMEM_ALLOC == 256, "layout");
};

template <int MODE>
__global__ void __launch_bounds__(C12Cfg<MODE>::NT, 1)
conv12_kernel(const float* __restrict__ mel, const int* __restrict__ seg_frame0, const float* __restrict__ seg_thr,
              const float* __restrict__ w1 /*[9][16]*/, const float* __restrict__ b1 /*[16]*/,
              const __half* __restrict__ wtc /*conv2: [9][CIN/8][hi co | lo co][8] fp16*/,
              const float* __restrict__ bias, float out_scale,
              unsigned char* __restrict__ out_hi, unsigned char* __restrict__ out_lo, int n_seg) {
  using K = C12Cfg<MODE>;
  using C = typename K::C;
  constexpr int H = C::H, W = C::W, CIN = C::CIN, COUT = C::COUT, P = C::P, BLK = C::BLK;
  constexpr int HALO = C::HALO, ROWB = C::ROWB, NA = K::NA;
  constexpr int EPI_THREADS = 256;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t sbase = smem_u32(smem);
  const uint32_t b_base = sbase + K::OFF_B;
  float* ws = reinterpret_cast<float*>(smem + K::OFF_W1);
  const uint32_t bar0 = sbase + K::OFF_BAR;
  const uint32_t bar_a_full = bar0, bar_a_free = bar0 + 8 * NA;
  const uint32_t bar_acc_full = bar_a_free + 8 * NA, bar_acc_free = bar_acc_full + 16, bar_w = bar_acc_free + 16;
  const uint32_t bar_mel_full = bar_w + 8, bar_mel_free = bar_mel_full + 8 * K::NM;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + K::OFF_BAR + 8 * K::N_BAR + 8);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_tiles = n_seg;

  // the zero row / zero column / halo rows of every A buffer are never written again
  for (int i = tid; i < NA * K::BUF_BYTES / 16; i += K::NT) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0u, 0u, 0u, 0u);
  for (int i = tid; i < 9 * 16 + 16; i += K::NT) ws[i] = (i < 144) ? __ldg(w1 + i) : __ldg(b1 + i - 144);
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), K::TMEM_ALLOC);
  if (tid == 32) {
    for (int i = 0; i < NA; ++i) {
      mbar_init(bar_a_full + 8 * i, K::N_PROD_WARPS);        // one arrival per producer warp
      mbar_init(bar_a_free + 8 * i, 2);                      // both MMA issuers have retired their reads
    }
    for (int i = 0; i < 2; ++i) { mbar_init(bar_acc_full + 8 * i, 2); mbar_init(bar_acc_free + 8 * i, 8); }
    mbar_init(bar_w, 1);
    for (int i = 0; i < K::NM; ++i) { mbar_init(bar_mel_full + 8 * i, 1); mbar_init(bar_mel_free + 8 * i, K::N_PROD_WARPS); }
    fence_barrier_init();
  }
  fence_proxy_async();                 // the zero fill above is read by the tensor core (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp >= K::W_PROD0 && warp < K::W_LOAD) {
    // ===== producers: conv1 + pool1 of tile `it` into A buffer it % NA =====
    const int grp = (warp - K::W_PROD0) >> 3;                 // channel group: channels 8 grp .. 8 grp + 7 when N_GROUPS == 2
    const int cell = ((warp - K::W_PROD0) & 7) * K::CPW + lane;
    const bool has_cell = lane < K::CPW;
    const int ph = cell / K::PW, pw = cell - ph * K::PW;      // lanes run along the pooled columns: consecutive plane rows
    const uint32_t row = (uint32_t)(HALO + (ph + 1) * P + (pw + 1));   // plane row q of the cell sits at tile row HALO + q
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
      const int buf = it % NA, use = it / NA, ms = it % K::NM;
      constexpr int NCQ = 4 / K::N_GROUPS;
      float res[4 * NCQ];
      long long tw = C12_NOW();
      mbar_wait_relaxed(bar_mel_full + 8 * ms, (it / K::NM) & 1);     // the segment's 15 mel rows are in the ring
      if (tid == K::W_PROD0 * 32) C12_ADD(0, tw);
      tw = C12_NOW();
      const float* mslot = reinterpret_cast<const float*>(smem + K::OFF_MEL + ms * K::MEL_SLOT);
      const float thr = mslot[kMels];                         // the clip's top_db floor, left in row 0's padding by the load warp
      if (has_cell) conv1_cell<MODE, false, K::MEL_PITCH, NCQ>(mslot, 0, thr, ws, ph, pw, res, grp * NCQ);
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_mel_free + 8 * ms);      // (the patch sits in registers: the slot may be refilled)
      if (tid == K::W_PROD0 * 32) C12_ADD(1, tw);
      tw = C12_NOW();
      mbar_wait_relaxed(bar_a_free + 8 * buf, (use & 1) ^ 1);         // the MMAs of tile it - NA have read the buffer
      if (tid == K::W_PROD0 * 32) C12_ADD(2, tw);
      tw = C12_NOW();
      if (has_cell) {
        unsigned char* a_hi = smem + buf * K::BUF_BYTES;
        unsigned char* a_lo = a_hi + C::A_BYTES;
#pragma unroll
        for (int c_ = 0; c_ < NCQ / 2; ++c_) {
          const int c = K::N_GROUPS == 2 ? grp : c_;          // the 16-byte chunk (8 channels) of the plane row
          uint4 hi, lo;
          split8(make_float4(res[8 * c_], res[8 * c_ + 1], res[8 * c_ + 2], res[8 * c_ + 3]),
                 make_float4(res[8 * c_ + 4], res[8 * c_ + 5], res[8 * c_ + 6], res[8 * c_ + 7]), hi, lo);
          uint32_t o = row * 32u + (uint32_t)c * 16u;
          o ^= (o >> 3) & 16u;                                // Swizzle<1,4,3> of the absolute (1024-aligned) tile address
          *reinterpret_cast<uint4*>(a_hi + o) = hi;
          *reinterpret_cast<uint4*>(a_lo + o) = lo;
        }
      }
      fence_proxy_async();                                    // generic-proxy stores -> visible to tcgen05.mma
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_a_full + 8 * buf);
      if (tid == K::W_PROD0 * 32) { C12_ADD(3, tw); C12_COUNT(15, 1); }
    }
  } else if (warp == K::W_LOAD) {
    if (lane == 0) {
      mbar_expect_tx(bar_w, K::B_BYTES);
      for (int t = 0; t < 9; ++t)
        bulk_g2s(b_base + t * C::B_STAGE, wtc + (size_t)t * (C::B_STAGE / 2), C::B_STAGE, bar_w);
    }
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
      const int ms = it % K::NM;
      const int f0 = __ldg(seg_frame0 + tile);
      if (lane == 0) {
        const float thr = __ldg(seg_thr + tile);               // (a global-load latency the producers must not see)
        mbar_wait_relaxed(bar_mel_free + 8 * ms, ((it / K::NM) & 1) ^ 1);
        *reinterpret_cast<float*>(smem + K::OFF_MEL + ms * K::MEL_SLOT + kMels * 4) = thr;   // released by the arrive below
        mbar_expect_tx(bar_mel_full + 8 * ms, K::MEL_BYTES);
      }
      __syncwarp();                                            // slot free and the transaction count armed
      if (lane < kSegLen)                                      // lane t: mel row t of the segment (192 contiguous bytes)
        bulk_g2s(sbase + K::OFF_MEL + ms * K::MEL_SLOT + lane * (K::MEL_PITCH * 4), mel + (size_t)(f0 + lane) * kMels,
                 kMels * 4, bar_mel_full + 8 * ms);
    }
  } else if (warp >= K::W_MMA0) {
    // ===== MMA issuers =====
    if (lane == 0) {
      const int mt = warp - K::W_MMA0;
      mbar_wait(bar_w, 0);
      int it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int buf = it % NA, use = it / NA, ab = it & 1, aph = (it >> 1) & 1;
        long long tw = C12_NOW();
        mbar_wait(bar_acc_free + 8 * ab, aph ^ 1);            // accumulators of tile it-2 drained
        if (mt == 0) C12_ADD(4, tw);
        tw = C12_NOW();
        mbar_wait(bar_a_full + 8 * buf, use & 1);
        if (mt == 0) C12_ADD(5, tw);
        tw = C12_NOW();
        tc_fence_after();
        const uint32_t a_hi = sbase + buf * K::BUF_BYTES, a_lo = a_hi + C::A_BYTES;
        const uint32_t d = tmem + ab * K::COLS_TILE + mt * (2 * COUT);
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          const int tapoff = (t / 3 - 1) * P + (t % 3 - 1);
          const uint32_t bst = b_base + t * C::B_STAGE;
          const uint32_t rowm = (uint32_t)(HALO + mt * 128 + tapoff);
#pragma unroll
          for (int ks = 0; ks < CIN / 16; ++ks) {
            const uint64_t db = make_desc(bst + (uint32_t)(2 * ks) * (2 * COUT * 16), 2 * COUT * 16, 128);
            const uint32_t aoff = rowm * ROWB + (uint32_t)ks * 32;
            umma_f16(d, make_desc_swz(a_hi + aoff, 8 * ROWB, C::LAYOUT), db, C::IDESC_2N, (t | ks) != 0);   // [0,C) += hi*hi ; [C,2C) += hi*lo
            umma_f16(d + COUT, make_desc_swz(a_lo + aoff, 8 * ROWB, C::LAYOUT), db, C::IDESC_1N, 1);        // [C,2C) += lo*hi
          }
        }
        umma_commit(bar_a_free + 8 * buf);
        umma_commit(bar_acc_full + 8 * ab);
        if (mt == 0) C12_ADD(6, tw);
      }
    }
  } else {
    // ===== epilogue (conv2: bias, ReLU, max-pool, split, store) =====
    const int quarter = warp & 3, mt = warp >> 2;
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
      const int ab = it & 1, aph = (it >> 1) & 1;
      float* stg = reinterpret_cast<float*>(smem + K::OFF_STG + (it & 1) * K::STG_BYTES);
      long long tw = C12_NOW();
      mbar_wait_relaxed(bar_acc_full + 8 * ab, aph);
      if (tid == 0) C12_ADD(7, tw);
      tw = C12_NOW();
      tc_fence_after();
      {
        const int r = mt * 128 + quarter * 32 + lane;         // tile row == plane row q of the segment
        const int hh = r / P, ww = r - hh * P;
        const bool valid = r < BLK && hh >= 1 && ww >= 1;
        const uint32_t trow = tmem + ((uint32_t)(quarter * 32) << 16) + ab * K::COLS_TILE + mt * (2 * COUT);
#pragma unroll
        for (int c16 = 0; c16 < COUT / 16; ++c16) {
          uint32_t ra[16], rb[16];
          tmem_ld16_nowait(trow + c16 * 16, ra);
          tmem_ld16_nowait(trow + COUT + c16 * 16, rb);
          tmem_ld_wait();
          if (valid) {
            const float4* b4 = reinterpret_cast<const float4*>(bias + c16 * 16);
            float4* dst = reinterpret_cast<float4*>(stg + ((hh - 1) * W + (ww - 1)) * C::STG_STRIDE + c16 * 16);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 bb = __ldg(b4 + j);
              dst[j] = make_float4(
                  fmaxf(fmaf(__uint_as_float(ra[4 * j + 0]) + __uint_as_float(rb[4 * j + 0]), out_scale, bb.x), 0.f),
                  fmaxf(fmaf(__uint_as_float(ra[4 * j + 1]) + __uint_as_float(rb[4 * j + 1]), out_scale, bb.y), 0.f),
                  fmaxf(fmaf(__uint_as_float(ra[4 * j + 2]) + __uint_as_float(rb[4 * j + 2]), out_scale, bb.z), 0.f),
                  fmaxf(fmaf(__uint_as_float(ra[4 * j + 3]) + __uint_as_float(rb[4 * j + 3]), out_scale, bb.w), 0.f));
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_free + 8 * ab);
      if (tid == 0) C12_ADD(8, tw);
      tw = C12_NOW();
      named_bar_sync(1, EPI_THREADS);                         // staging tile complete
      constexpr int POW = C::POW, HO = H / 2, C8 = COUT / 8;
      for (int i2 = tid; i2 < HO * POW * C8; i2 += EPI_THREADS) {
        const int c8 = i2 % C8;
        int rest = i2 / C8;
        const int pw2 = rest % POW;
        const int ph2 = rest / POW;
        int x0, x1;
        if (C::POOL == SP_POOL_ADAPT) { x0 = (pw2 * W) / POW; x1 = ((pw2 + 1) * W + POW - 1) / POW; }
        else { x0 = 2 * pw2; x1 = 2 * pw2 + 2; }
        float4 ma = make_float4(0.f, 0.f, 0.f, 0.f), mb = ma;   // post-ReLU values are >= 0
        for (int hy = 2 * ph2; hy < 2 * ph2 + 2; ++hy)
          for (int x = x0; x < x1; ++x) {
            const float4* tp = reinterpret_cast<const float4*>(stg + (hy * W + x) * C::STG_STRIDE + c8 * 8);
            const float4 ta = tp[0], tb = tp[1];
            ma.x = fmaxf(ma.x, ta.x); ma.y = fmaxf(ma.y, ta.y); ma.z = fmaxf(ma.z, ta.z); ma.w = fmaxf(ma.w, ta.w);
            mb.x = fmaxf(mb.x, tb.x); mb.y = fmaxf(mb.y, tb.y); mb.z = fmaxf(mb.z, tb.z); mb.w = fmaxf(mb.w, tb.w);
          }
        uint4 hi, lo;
        split8(ma, mb, hi, lo);
        const int g = kSplitLead + tile * C::OBLK + (ph2 + 1) * C::OP + (pw2 + 1);
        const size_t o = split_off<C::OROWB>(g, c8);
        *reinterpret_cast<uint4*>(out_hi + o) = hi;
        *reinterpret_cast<uint4*>(out_lo + o) = lo;
      }
      // (no second barrier: tile it+1 is staged in the other tile, and the barrier of tile it+1 - passed by every
      // warp only after it finished pooling tile it - orders the reuse of this one for tile it+2)
      if (tid == 0) C12_ADD(9, tw);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, K::TMEM_ALLOC);
}

template <int MODE>
static void launch_c12(cudaStream_t st, const float* mel, const int* seg_frame0, const float* seg_thr, const float* w1,
                       const float* b1, const __half* wtc, const float* bias, float scale, unsigned char* out_hi,
                       unsigned char* out_lo, int n_seg) {
  using K = C12Cfg<MODE>;
  static unsigned long long configured = 0;
  static int n_sm = 0;
  if (first_launch_on_device(configured)) {
    cudaFuncSetAttribute(conv12_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, K::SMEM_BYTES);
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  }
  const int grid = std::min(n_seg, n_sm > 0 ? n_sm : 148);
  conv12_kernel<MODE><<<grid, K::NT, K::SMEM_BYTES, st>>>(mel, seg_frame0, seg_thr, w1, b1, wtc, bias, scale, out_hi, out_lo, n_seg);
}

#ifdef NISQA_TC_TIMING
int c12_timing_read(long long* host, int n, int reset) {
  int rc = (int)cudaMemcpyFromSymbol(host, g_c12_timing, sizeof(long long) * n);
  if (reset) { static long long zero[256 * 16]; cudaMemcpyToSymbol(g_c12_timing, zero, sizeof zero); }
  return rc;
}
#endif

// conv1 + pool1 + conv2 + pool2: mel segments -> the plane pair feeding conv3
void launch_conv12(cudaStream_t st, int std_mode, const float* mel, const int* seg_frame0, const float* seg_thr,
                   const float* w1, const float* b1, const void* wtc2, const float* bias2, float scale2,
                   void* out_hi, void* out_lo, int n_seg) {
  const __half* w = reinterpret_cast<const __half*>(wtc2);
  unsigned char* oh = static_cast<unsigned char*>(out_hi);
  unsigned char* ol = static_cast<unsigned char*>(out_lo);
  if (std_mode) launch_c12<1>(st, mel, seg_frame0, seg_thr, w1, b1, w, bias2, scale2, oh, ol, n_seg);
  else launch_c12<0>(st, mel, seg_frame0, seg_thr, w1, b1, w, bias2, scale2, oh, ol, n_seg);
}

}  // namespace nisqa
