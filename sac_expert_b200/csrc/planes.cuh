// Weight-plane image layout shared by the optimiser kernels (elem.cuh::k_adam) and the warp-specialised fused MLP
// kernels (mlp_ws.cuh).  Image of a [K x 256] matrix W[i][j] (fp16 hi plane + fp16 lo plane, lo = rn16(w - hi)):
//     [t = i>>5][plane hi|lo][s = j>>6][r = i&31][64 j]      16-byte chunks XOR (r & 7)   (SWIZZLE_128B atoms)
// One net = the W0 stages (32 input rows each, zero-padded to a multiple of 32) followed by the 8 W1 stages.
// Nets with more than one output (the actor) append a W2 section: W2^T [N2 = 16 * ceil(nout / 16) rows n][256 j]
// (rows n >= nout are zero) as  [s = j>>6][plane hi|lo][n][64 j], 16-byte chunks XOR (n & 7), N2 * 1024 bytes.  The
// forward pass (h2 W2, contraction over j) reads atom s as a K-major SWIZZLE_128B B operand with N = N2; the backward
// pass (dOut W2^T, contraction over n) reads the same bytes as an MN-major B operand with N = 256.  The section
// holds W2 * WS_W2_SCALE: output-layer weights are small (1e-3 .. 1e-1), and unscaled their lo plane would fall into
// the fp16 subnormals and keep only ~1e-5 of the weight instead of ~2^-22; the forward pass removes the power of two
// exactly.  Weights of magnitude >= 65504 / WS_W2_SCALE (about 256) would saturate.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cstdint>

namespace saceo {

constexpr int WS_STAGE = 32768;

constexpr float WS_W2_SCALE = 256.f;
// rows N2 of the W2 section (0: single-output nets have none)
__host__ __device__ inline int ws_w2_rows(int nout) { return nout > 1 ? (nout + 15) / 16 * 16 : 0; }
// bytes of the plane image of one net with K0 inputs and nout outputs: W0 stages, the 8 W1 stages, the W2 section
__host__ __device__ inline long long ws_image_bytes(int K0, int nout) {
  return (long long)((K0 + 31) / 32 + 8) * WS_STAGE + (long long)ws_w2_rows(nout) * 1024;
}
// byte offset inside the W2 section (hi plane; lo plane = + N2 * 128) of the 16-byte chunk holding W2[8*c8 .. 8*c8+7][n]
__host__ __device__ inline int ws_w2_off(int N2, int n, int c8) {
  return (c8 >> 3) * (N2 * 256) + n * 128 + (((c8 & 7) ^ (n & 7)) << 4);
}
// byte offset (hi plane; lo plane = +16384) of the 16-byte chunk holding W[row][8*c8 .. 8*c8+7]; row counts from the
// first W0 row, the W1 rows follow at row index 32 * n0
__host__ __device__ inline long long ws_image_off(int row, int c8) {
  const int t = row >> 5, r = row & 31, s = c8 >> 3, c = c8 & 7;
  return (long long)t * WS_STAGE + s * 4096 + r * 128 + ((c ^ (r & 7)) << 4);
}

// used by k_adam: the 4 consecutive parameters at flat index e (multiple of 4) of a net with K0 inputs and nout outputs
// -> image bytes
__device__ __forceinline__ void ws_planes_store4(uint8_t* __restrict__ img, int K0, int nout, long long e, const float (&x)[4]) {
  const long long oW1 = (long long)K0 * 256 + 256, oW2 = oW1 + 65536 + 256;
  int row, col;
  if (e < (long long)K0 * 256) { row = (int)(e >> 8); col = (int)(e & 255); }
  else if (e >= oW1 && e < oW1 + 65536) { const int e2 = (int)(e - oW1); row = ((K0 + 31) / 32) * 32 + (e2 >> 8); col = e2 & 255; }
  else if (nout > 1 && e >= oW2 && e < oW2 + 256LL * nout) {
    // W2[j][n] at oW2 + j * nout + n: a group of four straddles two rows j when nout % 4 != 0, so each element is
    // placed on its own (b2 and whatever follows are not part of the image)
    const int N2 = ws_w2_rows(nout);
    uint8_t* w2 = img + ((K0 + 31) / 32 + 8) * (long long)WS_STAGE;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long e2 = e + k - oW2;
      if (e2 < 0 || e2 >= 256LL * nout) continue;
      const int j = (int)(e2 / nout), n = (int)(e2 - (long long)j * nout);
      uint32_t h, l;      // the conversion of split8<true> (k_planes_build), element in the low half
      const float xs = x[k] * WS_W2_SCALE;
      asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(0.f), "f"(xs));
      const float hf = __half2float(__ushort_as_half((unsigned short)h));
      asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(l) : "f"(0.f), "f"(xs - hf));
      uint8_t* dst = w2 + ws_w2_off(N2, n, j >> 3) + (j & 7) * 2;
      *reinterpret_cast<uint16_t*>(dst) = (uint16_t)h;
      *reinterpret_cast<uint16_t*>(dst + N2 * 128) = (uint16_t)l;
    }
    return;
  }
  else return;
  uint32_t h0, h1, l0, l1;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h0) : "f"(x[1]), "f"(x[0]));
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h1) : "f"(x[3]), "f"(x[2]));
  const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&h0)), f1 = __half22float2(*reinterpret_cast<const __half2*>(&h1));
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(l0) : "f"(x[1] - f0.y), "f"(x[0] - f0.x));
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(l1) : "f"(x[3] - f1.y), "f"(x[2] - f1.x));
  uint8_t* dst = img + ws_image_off(row, col >> 3) + (col & 7) * 2;
  *reinterpret_cast<uint2*>(dst) = make_uint2(h0, h1);
  *reinterpret_cast<uint2*>(dst + 16384) = make_uint2(l0, l1);
}


}  // namespace saceo
