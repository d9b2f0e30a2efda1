// conv_split.cuh - geometry / layout of the fp16 plane pairs shared by the tcgen05 conv kernels (conv_split.cu:
// conv3..conv6; conv12.cu: conv1 + conv2 fused).  See conv_split.cu for the layout description.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace nisqa {

enum { SP_POOL_NONE = 0, SP_POOL_ADAPT = 1, SP_POOL_2X2 = 2 };


// byte offset of chunk c (8 halves) of plane row g, rows of ROWB bytes: Swizzle<log2(ROWB/16), 4, 3>
template <int ROWB>
__device__ __forceinline__ size_t split_off(int g, int c) {
  const size_t o = (size_t)g * ROWB + (size_t)c * 16;
  return o ^ ((o >> 3) & (size_t)(ROWB - 16));
}

template <int H_, int W_, int CIN_, int COUT_, int POOL_, int POW_, bool F32OUT_ = false, bool CENTER_ = false>
struct SpCfg {
  static constexpr int H = H_, W = W_, CIN = CIN_, COUT = COUT_, POOL = POOL_, POW = POW_;
  static constexpr bool CENTER = CENTER_;         // conv6 of the AdaptCNN: kernel (3,3), padding (1,0) on a
                                                  // 3-wide map == the padded conv evaluated at column 1 only
  static constexpr bool OUT_SPLIT = !F32OUT_;     // the last layer writes the CNN features as fp32 channels-last
  static constexpr int P = W + 1;                 // row pitch: W interior columns + 1 shared zero column
  static constexpr int BLK = (H + 1) * P;         // rows per segment: H interior rows + 1 shared zero row
  static constexpr int G = 256 / BLK;             // segments per CTA (2 M-tiles of 128 rows)
  static constexpr int HALO = P + 1;              // |row offset| of the farthest tap
  static constexpr int AROWS = 256 + 2 * HALO;    // rows of the tile (copied)
  static constexpr int ROWB = CIN * 2;            // bytes per row
  static constexpr uint32_t LAYOUT = (ROWB == 128) ? 2u : (ROWB == 64 ? 4u : 6u);
  static constexpr int A_BYTES = ((AROWS + 7) * ROWB + 1023) & ~1023;     // + placement shift (g0 & 7 rows)
  static constexpr int NCH = CIN / 8;             // 16-byte K chunks (8 halves)
  static constexpr int B_HALF = NCH * COUT * 16;  // per hi / lo
  static constexpr int B_STAGE = 2 * B_HALF;
  // output geometry (= the next layer's input geometry)
  static constexpr int HO = (POOL == SP_POOL_NONE) ? H : H / 2;
  static constexpr int WO = (POOL == SP_POOL_NONE) ? (CENTER ? 1 : W) : POW;
  static constexpr int OP = WO + 1, OBLK = (HO + 1) * OP, OROWB = COUT * 2;
  static constexpr int STG_STRIDE = COUT + 4;     // floats per staged row (conflict-free float4)
  // D=f32, A=B=f16, both K-major, M=128; N = 2*COUT ([b_hi|b_lo]) and N = COUT (b_hi only)
  static constexpr uint32_t IDESC_2N = (1u << 4) | ((uint32_t)((2 * COUT) >> 3) << 17) | ((128u >> 4) << 24);
  static constexpr uint32_t IDESC_1N = (1u << 4) | ((uint32_t)(COUT >> 3) << 17) | ((128u >> 4) << 24);
  // un-pooled layers stage their output in shared memory as the exact HBM image of the CTA's segments
  // (plane rows incl. the zero row / column, or the fp32 feature rows) and write it with bulk stores
  static constexpr int IMG_BYTES = OUT_SPLIT ? G * OBLK * OROWB : G * HO * WO * COUT * 4;
  static_assert(B_STAGE % 16 == 0 && CIN % 16 == 0 && COUT % 32 == 0, "shape");
  static_assert(ROWB == 32 || ROWB == 64 || ROWB == 128, "rows are 32 / 64 / 128 bytes (one swizzle atom)");
  static_assert(HALO <= kSplitLead, "kSplitLead");
  static_assert(!CENTER || F32OUT_, "the centre-column variant only exists as the last layer");
  static_assert(OUT_SPLIT || POOL == SP_POOL_NONE, "fp32 output is not pooled");
  static_assert(G >= 1, "tile");
};

// layers 2..6; std_mode selects the StandardCNN geometry (W 8/4/2, MaxPool2d(2)).  conv2 runs only inside conv12_kernel.
//                     H   W  CIN COUT POOL           POW F32OUT CENTER
using SpConv2A = SpCfg<24, 7, 16, 32, SP_POOL_ADAPT, 5>;
using SpConv3A = SpCfg<12, 5, 32, 64, SP_POOL_NONE, 0>;
using SpConv4A = SpCfg<12, 5, 64, 64, SP_POOL_ADAPT, 3>;
using SpConv5A = SpCfg<6, 3, 64, 64, SP_POOL_NONE, 0>;
using SpConv6A = SpCfg<6, 3, 64, 64, SP_POOL_NONE, 0, true, true>;
using SpConv2S = SpCfg<24, 8, 16, 32, SP_POOL_2X2, 4>;
using SpConv3S = SpCfg<12, 4, 32, 64, SP_POOL_NONE, 0>;
using SpConv4S = SpCfg<12, 4, 64, 64, SP_POOL_2X2, 2>;
using SpConv5S = SpCfg<6, 2, 64, 64, SP_POOL_NONE, 0>;
using SpConv6S = SpCfg<6, 2, 64, 64, SP_POOL_NONE, 0, true>;

}  // namespace nisqa
