// conv1_cell.cuh - conv1(1->16) + BN + ReLU fused with the first max-pool for ONE pooled cell of one segment (all 16
// channels), shared by the fused conv1 + conv2 kernel (conv12.cu) and conv1_pool1_kernel (conv1.cu), which writes pool1
// for the stage dump.
//   MODE 0 (adapt, reference lib:690-691): adaptive_max_pool2d 48x15 -> 24x7 : rows {2i,2i+1}, cols [2j,2j+3)
//   MODE 1 (standard, lib:813-814): MaxPool2d(2, stride 2, padding (0,1)) -> 24x8 : cols {2j-1,2j}
#pragma once
#include "common.cuh"
#include "f32x2.cuh"

#ifndef NISQA_C1_PK
#define NISQA_C1_PK 1        // conv1 FMAs as packed FFMA2 (bit-identical to the scalar form)
#endif

namespace nisqa {

// ws: [9][16] folded conv1 weights followed by the 16 biases (shared memory).  LDG: `mel` is global memory read through
// the read-only path; false: a shared-memory copy of the segment's 15 mel rows (f0 = 0), rows PITCH floats apart.
// NCQ channel quads starting at quad cq0 (NCQ = 4, cq0 = 0: all 16 channels; the fused kernel splits them over two warp groups).
template <int MODE, bool LDG = true, int PITCH = kMels, int NCQ = 4>
__device__ __forceinline__ void conv1_cell(const float* __restrict__ mel, int f0, float thr, const float* ws,
                                           int ph, int pw, float (&res)[4 * NCQ], int cq0 = 0) {
  constexpr int NWC = (MODE == 0) ? 3 : 2;       // window columns
  constexpr int PC = NWC + 2;                    // patch columns
  const int r0 = 2 * ph - 1;                     // first patch row (mel index)
  const int c0 = (MODE == 0) ? 2 * pw - 1 : 2 * pw - 2;   // first patch col (frame in segment)
  float patch[4][PC];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < PC; ++j) {
      const int r = r0 + i, t = c0 + j;
      float v = 0.f;                             // zero padding of the segment's own border
      if (r >= 0 && r < kMels && t >= 0 && t < kSegLen)
        v = fmaxf(LDG ? __ldg(mel + (size_t)(f0 + t) * PITCH + r) : mel[(f0 + t) * PITCH + r], thr);
      patch[i][j] = v;
    }

#if NISQA_C1_PK
  // 16 channels as 8 packed pairs (FFMA2: the same fp32 FMA per element and tap order as the scalar form, half the
  // instructions - the producer warps of conv12 are issue bound)
#pragma unroll
  for (int cq_ = 0; cq_ < NCQ; ++cq_) {
    const int cq = cq0 + cq_;
    f2 acc[2][NWC][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < NWC; ++j) { acc[i][j][0] = 0ull; acc[i][j][1] = 0ull; }
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const float4 w = *reinterpret_cast<const float4*>(ws + tap * 16 + cq * 4);
      const f2 w01 = pk(w.x, w.y), w23 = pk(w.z, w.w);
      const int ky = tap / 3, kx = tap % 3;
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < NWC; ++j) {
          const f2 a = bc(patch[i + ky][j + kx]);
          acc[i][j][0] = fma2(a, w01, acc[i][j][0]);
          acc[i][j][1] = fma2(a, w23, acc[i][j][1]);
        }
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < NWC; ++j) {
          const int col = c0 + 1 + j;            // conv output column of this window slot
          if (MODE == 0 || (col >= 0 && col < kSegLen)) {
            const float2 v = upk(acc[i][j][h]);
            m0 = fmaxf(m0, v.x); m1 = fmaxf(m1, v.y);
          }
        }
      res[cq_ * 4 + 2 * h] = fmaxf(m0 + ws[144 + cq * 4 + 2 * h], 0.f);           // bias + ReLU commute with max
      res[cq_ * 4 + 2 * h + 1] = fmaxf(m1 + ws[144 + cq * 4 + 2 * h + 1], 0.f);
    }
  }
}
#else
#pragma unroll
  for (int cq_ = 0; cq_ < NCQ; ++cq_) {
    const int cq = cq0 + cq_;
    float acc[2][NWC][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < NWC; ++j)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[i][j][c] = 0.f;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const float4 w = *reinterpret_cast<const float4*>(ws + tap * 16 + cq * 4);
      const int ky = tap / 3, kx = tap % 3;
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < NWC; ++j) {
          const float a = patch[i + ky][j + kx];
          acc[i][j][0] = fmaf(a, w.x, acc[i][j][0]);
          acc[i][j][1] = fmaf(a, w.y, acc[i][j][1]);
          acc[i][j][2] = fmaf(a, w.z, acc[i][j][2]);
          acc[i][j][3] = fmaf(a, w.w, acc[i][j][3]);
        }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float m = -INFINITY;
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < NWC; ++j) {
          const int col = c0 + 1 + j;            // conv output column of this window slot
          if (MODE == 0 || (col >= 0 && col < kSegLen)) m = fmaxf(m, acc[i][j][c]);
        }
      res[cq_ * 4 + c] = fmaxf(m + ws[144 + cq * 4 + c], 0.f);   // bias + ReLU commute with max
    }
  }
}
#endif

}  // namespace nisqa
