// conv1.cu - conv1 + BN + ReLU + pool1 of the framewise CNN as a standalone kernel (reference
// nisqa/NISQA_lib.py:690-691 AdaptCNN, lib:813-814 StandardCNN; eval-mode BatchNorm folded into the
// conv weights on the host), and the NHWC -> NCHW conversion of the stage dumps.
//
// The product path computes pool1 inside conv12_kernel (conv12.cu) and never stores it.  This kernel
// only runs when nisqa_set_option("keep_pool1", 1) asks for pool1 to be kept for the stage dump: it
// writes the same values, in the plane layout of conv_split.cu, into a plane pair that nothing else reads.
#include "common.cuh"
#include "tc_ptx.cuh"
#include "conv1_cell.cuh"

namespace nisqa {

// ----------------------------------------------------------------------------------------
// conv1 + BN + ReLU + pool1
//   MODE 0 (adapt, lib:690-691): adaptive_max_pool2d 48x15 -> 24x7 : rows {2i,2i+1}, cols [2j,2j+3)
//   MODE 1 (standard, lib:813-814): MaxPool2d(2, stride 2, padding (0,1)) -> 24x8 : cols {2j-1,2j}
// thread = one pooled cell of one segment, all 16 channels.  The output goes out as two fp16 planes
// (conv_split.cu: padded rows of 16 halves = 32 bytes, 32-byte swizzle).
template <int MODE>
__global__ void __launch_bounds__(256)
conv1_pool1_kernel(const float* __restrict__ mel, const int* __restrict__ seg_frame0,
                   const float* __restrict__ seg_thr, const float* __restrict__ w1 /*[9][16]*/,
                   const float* __restrict__ b1 /*[16]*/, unsigned char* __restrict__ out_hi,
                   unsigned char* __restrict__ out_lo, int n_seg) {
  constexpr int PW = (MODE == 0) ? 7 : 8;
  __shared__ __align__(16) float ws[9 * 16 + 16];
  for (int i = threadIdx.x; i < 9 * 16 + 16; i += blockDim.x)
    ws[i] = (i < 144) ? __ldg(w1 + i) : __ldg(b1 + i - 144);
  __syncthreads();

  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int seg = (int)(gid / (24 * PW));
  if (seg >= n_seg) return;
  const int cell = (int)(gid - (long long)seg * (24 * PW));
  const int ph = cell % 24, pw = cell / 24;      // lanes run along mel rows: coalesced reads
  const int f0 = __ldg(seg_frame0 + seg);
  const float thr = __ldg(seg_thr + seg);

  float res[16];
  conv1_cell<MODE>(mel, f0, thr, ws, ph, pw, res);
  const int g = kSplitLead + seg * (25 * (PW + 1)) + (ph + 1) * (PW + 1) + (pw + 1);
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    uint4 hi, lo;
    split8(make_float4(res[8 * c], res[8 * c + 1], res[8 * c + 2], res[8 * c + 3]),
           make_float4(res[8 * c + 4], res[8 * c + 5], res[8 * c + 6], res[8 * c + 7]), hi, lo);
    size_t o = (size_t)g * 32 + (size_t)c * 16;
    o ^= (o >> 3) & 16;                          // Swizzle<1,4,3>
    *reinterpret_cast<uint4*>(out_hi + o) = hi;
    *reinterpret_cast<uint4*>(out_lo + o) = lo;
  }
}

// NHWC [n][HW][C] -> NCHW [n][C][HW] (stage dumps only; matches the reference tensor layout)
__global__ void nhwc_to_nchw_kernel(const float* __restrict__ in, float* __restrict__ out,
                                    long long n, int hw, int ch) {
  const long long total = n * hw * ch;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int p = (int)(i % hw);
    const int c = (int)((i / hw) % ch);
    const long long s = i / ((long long)hw * ch);
    out[i] = in[(s * hw + p) * ch + c];
  }
}

void launch_conv1(cudaStream_t st, int std_mode, const float* mel, const int* seg_frame0,
                  const float* seg_thr, const float* w1, const float* b1, void* out_hi, void* out_lo,
                  int n_seg) {
  const int cells = std_mode ? 24 * 8 : 24 * 7;
  const long long total = (long long)n_seg * cells;
  const int grid = (int)((total + 255) / 256);
  unsigned char* oh = static_cast<unsigned char*>(out_hi);
  unsigned char* ol = static_cast<unsigned char*>(out_lo);
  if (std_mode) conv1_pool1_kernel<1><<<grid, 256, 0, st>>>(mel, seg_frame0, seg_thr, w1, b1, oh, ol, n_seg);
  else conv1_pool1_kernel<0><<<grid, 256, 0, st>>>(mel, seg_frame0, seg_thr, w1, b1, oh, ol, n_seg);
}

void launch_nhwc_to_nchw(cudaStream_t st, const float* in, float* out, long long n, int hw, int ch) {
  nhwc_to_nchw_kernel<<<1024, 256, 0, st>>>(in, out, n, hw, ch);
}

}  // namespace nisqa
