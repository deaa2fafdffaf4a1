// Warp-specialised fused forward / backward chains of the 2x256 MLPs (actor, twin critics, twin targets), round 2.
//
// What changed against the round-1 kernels (tc_gemm.cuh::k_mlp_fwd_tc / k_mlp_bwd_tc, kept as the fallback engine):
//   * WEIGHT PLANES.  The fp32 -> fp16 hi/lo operand split of W0 and W1 is no longer done by every CTA for every
//     128-row tile of every pass (the convert -> fence -> barrier chain that bounded the W1 loop, 7.05 us against
//     3.25 us of pure streaming).  The optimiser owns it: k_adam (and its Polyak line) emits the split planes of
//     every parameter it updates, pre-swizzled, into a library-owned image; k_planes_build creates the image from
//     the fp32 tables after a bind or an external write (saceo_weights_changed).
//   * TMA.  A producer warp streams 32 KB stages of that image with cp.async.bulk (UBLKCP) + mbarrier expect_tx
//     through a 4-deep shared-memory ring; nobody touches the bytes between HBM/L2 and the tensor core.
//   * ONE IMAGE, BOTH DIRECTIONS.  Image of a [K x 256] matrix W[i][j]:  [t = i>>5][plane hi|lo][s = j>>6][r = i&31][64 j]
//     (fp16, 16-byte chunks XOR (r & 7)).  The forward pass (X W, contraction over i) reads a stage t as an MN-MAJOR
//     SWIZZLE_128B B operand (LBO 4096 = next 64-wide j atom, SBO 1024 = next 8 i rows; probed on hardware,
//     tools/umma_probe.cu); the backward pass (dY W^T, contraction over j) reads 4 KB pieces (t, s) of the SAME image
//     as the K-MAJOR B operand the round-1 loader produced.
//   * WARP ROLES.  warps 0-7: operand conversion of the activation tile + epilogues (TMEM -> registers -> TMEM / HBM);
//     warp 8: TMA producer; warp 9: TMEM allocation + the single MMA-issuing thread.  Everything is mbarrier-paced;
//     the accumulator of layer l lives in one half of TMEM, the fp16 hi/lo A operand of layer l+1 is written IN PLACE
//     over it (32 fp32 columns -> 16 hi + 16 lo columns), the next accumulator goes to the other half, so the MMAs of
//     layer l+1 start on the first 64-wide k group while the epilogue still converts the rest.
//   * OUTPUT LAYER OF THE ACTOR ON THE TENSOR CORE.  Nets with more than one output append W2^T to their plane image
//     (planes.cuh); epilogue 1 writes h2 as fp16 hi/lo in place over its accumulator, exactly as epilogue 0 does for
//     h1, and the MMA thread forms out = h2 W2 (N = 16 ceil(nout / 16), 48 MMAs with A in TMEM) into the dead layer-0
//     half.  Nothing is converted or reduced across warps on the way: one TMEM read per row, plus b2.  The backward
//     kernel reads the same W2 bytes as an MN-major B operand for its first step dOut W2^T (K = 16 ceil(k_out / 16)),
//     with the dOut rows as a scaled fp16 hi/lo A operand in TMEM.
//   * SKINNY LAYERS ON CUDA CORES, EXACT FP32.  The critics' single-output layer and first backward step (an outer
//     product) and the action-column input gradient (N = A) are dot products against a few weight rows:
//     they are formed inside the epilogues from the row each thread already holds (weights broadcast from shared
//     memory).
//   * Backward operands: tcgen05 kind::f16 rejects mixed A/B formats (bf16 x fp16 traps, tools/umma_probe.cu), so the
//     gradient tile uses fp16 hi/lo planes too, with a per-row power-of-two scale (chosen from a bound on the row's
//     magnitude, removed exactly in the next epilogue): 22 significant bits relative to the row maximum.
#pragma once
#include "tc_gemm.cuh"
#include "planes.cuh"

namespace saceo {

constexpr int WS_NEW = 16;                    // conversion / epilogue warps: 4 TMEM lane quarters x 4 column groups of 64
constexpr int WS_NEPI = WS_NEW * 32, WS_NT = WS_NEPI + 64;    // + TMA producer warp + MMA / TMEM-allocator warp
constexpr int WS_NST = 3, WS_RING = WS_NST * WS_STAGE;
constexpr int WS_AUX = 49152;                 // [0, WS_RED): X planes (fwd layer 0) | fp32 skinny weights (bwd); [WS_RED, ..): reductions / column sums
constexpr int WS_PATCH1 = 32 * 32 * 4;        // warp-private 32 x 32 float transposition patch, 16-byte chunks XOR (row & 7)
constexpr int WS_PATCH = WS_NEW * WS_PATCH1;
constexpr int WS_MAIN = WS_RING + WS_AUX + WS_PATCH;
constexpr int WS_BYTES = WS_MAIN + 1024 + 256;
constexpr int WS_RED = 40960;                 // offset inside AUX of the 8 KB reduction / column-sum scratch
constexpr int WS_MAXOUT = 36;                 // skinny dims (n_out, k_out) supported: fp32 [256][<=36] fits below WS_RED
enum { WB_FULL = 0, WB_EMPTY = WS_NST, WB_XFULL = 2 * WS_NST, WB_XEMPTY, WB_D0, WB_D1, WB_AP /* 4 */, WB_D2 = WB_AP + 4 };

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 512;" ::: "memory"); }   // the 16 epilogue warps only
// MN-major SWIZZLE_128B descriptor of a weight-plane stage: LBO = next 64-wide n atom (4096 in the W0 / W1 stages),
// SBO = 1024 (next 8 k rows)
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t saddr, uint32_t lbo = 4096) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
constexpr uint32_t WS_IDESC_FWD = (1u << 4) | (1u << 16) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);  // fp16, B MN-major, N 256
constexpr uint32_t WS_IDESC_BWD = (1u << 4) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);              // fp16, K-major, N 128

// ------------------------------------------------------------------------------------------
// plane image maintenance
// ------------------------------------------------------------------------------------------
// Builds the images of `nets` nets from their fp32 tables.  grid: (ceil(items/256), nets), item = one 16-byte chunk.
__global__ void k_planes_build(const float* __restrict__ theta, long long stride, uint8_t* __restrict__ img, int K0, int nout) {
  const int n0 = (K0 + 31) / 32, N2 = ws_w2_rows(nout), rows = n0 * 32 + 256 + N2;
  const int item = blockIdx.x * blockDim.x + threadIdx.x;
  if (item >= rows * 32) return;
  const int row = item >> 5, c8 = item & 31;
  const float* th = theta + (long long)blockIdx.y * stride;
  uint8_t* net_img = img + (long long)blockIdx.y * ws_image_bytes(K0, nout);
  float x[8];
  if (row >= n0 * 32 + 256) {       // W2 section: row n of W2^T = column n of W2 [256][nout] (zero for n >= nout)
    const int n = row - n0 * 32 - 256;
    const long long o = (long long)K0 * 256 + 256 + 65536 + 256 + (long long)(c8 * 8) * nout + n;
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = n < nout ? th[o + (long long)j * nout] * WS_W2_SCALE : 0.f;
    uint4 hi, lo;
    split8<true>(x, hi, lo);
    uint8_t* dst = net_img + (long long)(n0 + 8) * WS_STAGE + ws_w2_off(N2, n, c8);
    *reinterpret_cast<uint4*>(dst) = hi;
    *reinterpret_cast<uint4*>(dst + N2 * 128) = lo;
    return;
  }
  if (row < n0 * 32) {
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = row < K0 ? th[(long long)row * 256 + c8 * 8 + j] : 0.f;
  } else {
    const long long o = (long long)K0 * 256 + 256 + (long long)(row - n0 * 32) * 256 + c8 * 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = th[o + j];
  }
  uint4 hi, lo;
  split8<true>(x, hi, lo);
  uint8_t* dst = net_img + ws_image_off(row, c8);
  *reinterpret_cast<uint4*>(dst) = hi;
  *reinterpret_cast<uint4*>(dst + 16384) = lo;
}

// ------------------------------------------------------------------------------------------
// shared pieces of the epilogues
// ------------------------------------------------------------------------------------------
// warp-private patch addressing: row r (0..31), float column c (0..31): chunk (c>>2) XOR (r&7); conflict-free for the
// lane-per-row float4 accesses, the 8-lanes-per-row float4 accesses and the lane-per-column scalar reads alike
__device__ __forceinline__ uint32_t ws_pa(uint32_t patch, int r, int c) {
  return patch + (uint32_t)(r * 128 + ((((c >> 2) ^ (r & 7)) << 4) | ((c & 3) << 2)));
}
// v (this lane's row, 32 columns) -> global tile rows through the warp-private patch (whole 128-byte segments per request)
// cs != 0: the column sums of the valid rows of the tile go to cs[q][col + c] (floats) - summed from the values each lane
// handles anyway (8 rows x 4 columns), finished with two shuffle steps in a fixed order
__device__ __forceinline__ void ws_store_rows(uint32_t patch, const uint32_t (&v)[32], float* __restrict__ G, int rbase,
                                              int rows, int col, int lane, uint32_t cs = 0, int q = 0) {
#pragma unroll
  for (int j = 0; j < 8; ++j) sts128(ws_pa(patch, lane, 4 * j), make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
  __syncwarp();
  const int lr = lane >> 3, lc = (lane & 7) * 4;
  float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int rr = 0; rr < 32; rr += 4) {
    const int r = rr + lr, grow = rbase + r;
    if (grow < rows) {
      const float4 t4 = lds128(ws_pa(patch, r, lc));
      if (G) *reinterpret_cast<float4*>(G + (long long)grow * FW_H + col + lc) = t4;
      sum.x += t4.x; sum.y += t4.y; sum.z += t4.z; sum.w += t4.w;
    }
  }
  if (cs) {
#pragma unroll
    for (int o = 8; o <= 16; o <<= 1) {
      sum.x += __shfl_xor_sync(0xffffffffu, sum.x, o); sum.y += __shfl_xor_sync(0xffffffffu, sum.y, o);
      sum.z += __shfl_xor_sync(0xffffffffu, sum.z, o); sum.w += __shfl_xor_sync(0xffffffffu, sum.w, o);
    }
    if (lane < 8) sts128f(cs + (uint32_t)(q * FW_H + col + lc) * 4, sum.x, sum.y, sum.z, sum.w);
  }
}
// column sums of the tile left in the patch by ws_store_rows (valid rows only) -> cs[q][col + lane]
__device__ __forceinline__ void ws_colsum(uint32_t patch, uint32_t cs, int q, int rbase, int rows, int col, int lane) {
  const int nvalid = rows - rbase;
  float s = 0.f;
#pragma unroll 8
  for (int r = 0; r < 32; ++r) { const float t = lds32(ws_pa(patch, r, lane)); s += r < nvalid ? t : 0.f; }
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(cs + (uint32_t)(q * FW_H + col + lane) * 4), "f"(s) : "memory");
}
// saved activations [32 rows x 32 cols] of this warp, two-phase: the global loads are issued early (before a barrier
// wait / during the previous chunk's math), the transposition through the patch happens when the values are needed
__device__ __forceinline__ void ws_rows_issue(const float* __restrict__ Hs, int rbase, int rows, int col, int lane, float4 (&t)[8]) {
  const int lr = lane >> 3, lc = (lane & 7) * 4;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int grow = rbase + 4 * i + lr;
    t[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (grow < rows) t[i] = __ldg(reinterpret_cast<const float4*>(Hs + (long long)grow * FW_H + col + lc));
  }
}
// L2 prefetch of the same tiles (one 128-byte line per lane): the backward kernel asks for the saved activations early
// WITHOUT holding 32 registers for them across the epilogue math (the 96-register cap of an 18-warp CTA made that
// prefetch buffer spill: 1.6 M local loads + 1.5 M local stores per launch at 17 % L1 hit rate, profiles/r2_step_ncu_full_summary.txt)
__device__ __forceinline__ void ws_rows_prefetch(const float* __restrict__ Hs, int rbase, int rows, int col, int lane) {
  if (rbase + lane < rows) asm volatile("prefetch.global.L2 [%0];" ::"l"(Hs + (long long)(rbase + lane) * FW_H + col));
}
__device__ __forceinline__ void ws_planes_prefetch(const uint8_t* __restrict__ img, int rbase, int rows, int col, int lane) {
  if (rbase + lane < rows) {
    const uint8_t* p = img + ws_image_off(rbase + lane, (col >> 6) << 3);     // the 128-byte row segment holding these 32 columns
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p + 16384));
  }
}
__device__ __forceinline__ void ws_rows_commit(uint32_t patch, int lane, const float4 (&t)[8], float (&aux)[32]) {
  const int lr = lane >> 3, lc = (lane & 7) * 4;
#pragma unroll
  for (int i = 0; i < 8; ++i)
    sts128(ws_pa(patch, 4 * i + lr, lc), make_uint4(__float_as_uint(t[i].x), __float_as_uint(t[i].y), __float_as_uint(t[i].z), __float_as_uint(t[i].w)));
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 t4 = lds128(ws_pa(patch, lane, 4 * j));
    aux[4 * j] = t4.x; aux[4 * j + 1] = t4.y; aux[4 * j + 2] = t4.z; aux[4 * j + 3] = t4.w;
  }
  __syncwarp();
}
__device__ __forceinline__ void ws_load_rows(uint32_t patch, const float* __restrict__ Hs, int rbase, int rows, int col, int lane,
                                             float (&aux)[32]) {
  const int lr = lane >> 3, lc = (lane & 7) * 4;
#pragma unroll
  for (int rr = 0; rr < 32; rr += 4) {
    const int r = rr + lr, grow = rbase + r;
    float4 t4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (grow < rows) t4 = __ldg(reinterpret_cast<const float4*>(Hs + (long long)grow * FW_H + col + lc));
    sts128(ws_pa(patch, r, lc), make_uint4(__float_as_uint(t4.x), __float_as_uint(t4.y), __float_as_uint(t4.z), __float_as_uint(t4.w)));
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 t4 = lds128(ws_pa(patch, lane, 4 * j));
    aux[4 * j] = t4.x; aux[4 * j + 1] = t4.y; aux[4 * j + 2] = t4.z; aux[4 * j + 3] = t4.w;
  }
  __syncwarp();
}
// Activation plane images (bf16 hi / lo, layout ws_image_off(row, 16-byte chunk)): the [32 rows x 32 cols] tile of a warp
// goes through the warp's transposition patch, so that every request touches whole 64-byte row segments (4 lanes per
// row, 8 rows per request) instead of 32 different lines.  k_dw_planes reads the images as MN-major operands.
//   store: the patch holds the fp32 tile (written lane-per-row, __syncwarp done)
__device__ __forceinline__ void ws_store_planes_p(uint32_t patch, uint8_t* __restrict__ img, int rbase, int rows, int col, int lane) {
  const int lr = lane >> 2, c8 = lane & 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = 8 * i + lr, grow = rbase + r;
    if (grow < rows) {
      const float4 a = lds128(ws_pa(patch, r, 8 * c8)), b = lds128(ws_pa(patch, r, 8 * c8 + 4));
      const float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
      uint4 hi, lo;
      split8<false>(x, hi, lo);
      uint8_t* dst = img + ws_image_off(grow, (col >> 3) + c8);
      *reinterpret_cast<uint4*>(dst) = hi;
      *reinterpret_cast<uint4*>(dst + 16384) = lo;
    }
  }
}
//   store + column sums in ONE pass over the patch (the gradient tiles whose fp32 form is not kept): v -> patch -> planes,
//   the column sums of the valid rows to cs[q][col + c] from the 4 rows x 8 columns each lane converts anyway, finished
//   with three shuffle steps in a fixed order
__device__ __forceinline__ void ws_store_planes_cs(uint32_t patch, const uint32_t (&v)[32], uint8_t* __restrict__ img, int rbase, int rows,
                                                   int col, int lane, uint32_t cs, int q) {
#pragma unroll
  for (int j = 0; j < 8; ++j) sts128(ws_pa(patch, lane, 4 * j), make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
  __syncwarp();
  const int lr = lane >> 2, c8 = lane & 3;
  float s[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = 8 * i + lr, grow = rbase + r;
    if (grow < rows) {
      const float4 a = lds128(ws_pa(patch, r, 8 * c8)), b = lds128(ws_pa(patch, r, 8 * c8 + 4));
      const float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
      uint4 hi, lo;
      split8<false>(x, hi, lo);
      uint8_t* dst = img + ws_image_off(grow, (col >> 3) + c8);
      *reinterpret_cast<uint4*>(dst) = hi;
      *reinterpret_cast<uint4*>(dst + 16384) = lo;
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += x[j];
    }
  }
  if (cs) {
#pragma unroll
    for (int o = 4; o <= 16; o <<= 1)
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
    if (lane < 4) {
      sts128f(cs + (uint32_t)(q * FW_H + col + 8 * c8) * 4, s[0], s[1], s[2], s[3]);
      sts128f(cs + (uint32_t)(q * FW_H + col + 8 * c8 + 4) * 4, s[4], s[5], s[6], s[7]);
    }
  }
}
//   load, two-phase: request the tile early (8 x 16 bytes per lane), decode it into the patch (fp32) when needed
__device__ __forceinline__ void ws_planes_issue(const uint8_t* __restrict__ img, int rbase, int rows, int col, int lane, float4 (&t)[8]) {
  const int lr = lane >> 2, c8 = lane & 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int grow = rbase + 8 * i + lr;
    t[2 * i] = make_float4(0.f, 0.f, 0.f, 0.f); t[2 * i + 1] = t[2 * i];
    if (grow < rows) {
      const uint8_t* src = img + ws_image_off(grow, (col >> 3) + c8);
      t[2 * i] = __ldg(reinterpret_cast<const float4*>(src));
      t[2 * i + 1] = __ldg(reinterpret_cast<const float4*>(src + 16384));
    }
  }
}
__device__ __forceinline__ void ws_planes_commit_p(uint32_t patch, int lane, const float4 (&t)[8]) {
  const int lr = lane >> 2, c8 = lane & 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t hw[4] = {__float_as_uint(t[2 * i].x), __float_as_uint(t[2 * i].y), __float_as_uint(t[2 * i].z), __float_as_uint(t[2 * i].w)};
    const uint32_t lw[4] = {__float_as_uint(t[2 * i + 1].x), __float_as_uint(t[2 * i + 1].y), __float_as_uint(t[2 * i + 1].z), __float_as_uint(t[2 * i + 1].w)};
    float h[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      h[2 * j] = __uint_as_float(hw[j] << 16) + __uint_as_float(lw[j] << 16);
      h[2 * j + 1] = __uint_as_float(hw[j] & 0xFFFF0000u) + __uint_as_float(lw[j] & 0xFFFF0000u);
    }
    sts128f(ws_pa(patch, 8 * i + lr, 8 * c8), h[0], h[1], h[2], h[3]);
    sts128f(ws_pa(patch, 8 * i + lr, 8 * c8 + 4), h[4], h[5], h[6], h[7]);
  }
  __syncwarp();
}
// tcgen05.ld without the wait: two chunks are requested back to back, then waited for once
__device__ __forceinline__ void tmem_ld32_nw(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
               "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
               "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                 "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                 "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                 "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
               : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// one row of a skinny fp32 weight block W[j][0..n) (row-major, n floats per row) -> registers, zero-padded to NR
template <int NR>
__device__ __forceinline__ void ws_load_wrow(const float* __restrict__ W, int j, int n, float (&w)[NR]) {
  const float* r = W + (long long)j * n;
  if ((n & 3) == 0) {
#pragma unroll
    for (int c4 = 0; c4 < NR / 4; ++c4) {
      float4 t4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c4 * 4 < n) t4 = __ldg(reinterpret_cast<const float4*>(r) + c4);
      w[4 * c4] = t4.x; w[4 * c4 + 1] = t4.y; w[4 * c4 + 2] = t4.z; w[4 * c4 + 3] = t4.w;
    }
  } else {
#pragma unroll
    for (int c = 0; c < NR; ++c) w[c] = c < n ? __ldg(r + c) : 0.f;
  }
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
// 32 fp32 values x scale -> fp16 hi/lo A-operand columns [c0, c0+16) hi, [c0+16, c0+32) lo, 16 values at a time (registers)
__device__ __forceinline__ void ws_split_store(uint32_t taddr, const uint32_t (&v)[32], float scale) {
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float x0 = __uint_as_float(v[16 * h + 2 * j]) * scale, x1 = __uint_as_float(v[16 * h + 2 * j + 1]) * scale;
      asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi[j]) : "f"(x1), "f"(x0));
      const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi[j]));
      asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo[j]) : "f"(x1 - hf.y), "f"(x0 - hf.x));
    }
    tmem_st8(taddr + 8 * h, hi);
    tmem_st8(taddr + 16 + 8 * h, lo);
  }
}
// v *= s * act'(h) with h = this lane's row of the saved activations parked in the patch by ws_rows_commit_p
template <int ACT>
__device__ __forceinline__ void ws_mul_dact_p(uint32_t (&v)[32], uint32_t patch, int lane, float s) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 h = lds128(ws_pa(patch, lane, 4 * j));
    v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) * s * dact_from_out(ACT, h.x));
    v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) * s * dact_from_out(ACT, h.y));
    v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) * s * dact_from_out(ACT, h.z));
    v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) * s * dact_from_out(ACT, h.w));
  }
  __syncwarp();
}
__device__ __forceinline__ void ws_mul_dact_p_rt(int act, uint32_t (&v)[32], uint32_t patch, int lane, float s) {
  if (act == ACT_RELU) ws_mul_dact_p<ACT_RELU>(v, patch, lane, s);
  else if (act == ACT_TANH) ws_mul_dact_p<ACT_TANH>(v, patch, lane, s);
  else ws_mul_dact_p<ACT_ELU>(v, patch, lane, s);
}
// the patch half of ws_rows_commit: rows in flight -> patch (row-wise), nothing kept in registers
__device__ __forceinline__ void ws_rows_commit_p(uint32_t patch, int lane, const float4 (&t)[8]) {
  const int lr = lane >> 3, lc = (lane & 7) * 4;
#pragma unroll
  for (int i = 0; i < 8; ++i)
    sts128(ws_pa(patch, 4 * i + lr, lc), make_uint4(__float_as_uint(t[i].x), __float_as_uint(t[i].y), __float_as_uint(t[i].z), __float_as_uint(t[i].w)));
  __syncwarp();
}
// fp32 x scale -> fp16 hi/lo pairs (A-operand columns)
__device__ __forceinline__ void ws_split_f16(const uint32_t (&v)[32], float scale, uint32_t (&hi)[16], uint32_t (&lo)[16]) {
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float x0 = __uint_as_float(v[2 * j]) * scale, x1 = __uint_as_float(v[2 * j + 1]) * scale;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi[j]) : "f"(x1), "f"(x0));
    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi[j]));
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo[j]) : "f"(x1 - hf.y), "f"(x0 - hf.x));
  }
}
// bias: shared-memory address of the 32 bias values of this chunk (staged once per CTA: a global load here would sit
// on the critical path of every chunk)
template <int ACT>
__device__ __forceinline__ void ws_bias_act(uint32_t (&v)[32], uint32_t bias) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 b = lds128(bias + j * 16);
    v[4 * j] = __float_as_uint(apply_act(ACT, __uint_as_float(v[4 * j]) + b.x));
    v[4 * j + 1] = __float_as_uint(apply_act(ACT, __uint_as_float(v[4 * j + 1]) + b.y));
    v[4 * j + 2] = __float_as_uint(apply_act(ACT, __uint_as_float(v[4 * j + 2]) + b.z));
    v[4 * j + 3] = __float_as_uint(apply_act(ACT, __uint_as_float(v[4 * j + 3]) + b.w));
  }
}
__device__ __forceinline__ void ws_bias_act_rt(int act, uint32_t (&v)[32], uint32_t bias) {
  if (act == ACT_RELU) ws_bias_act<ACT_RELU>(v, bias);
  else if (act == ACT_TANH) ws_bias_act<ACT_TANH>(v, bias);
  else ws_bias_act<ACT_ELU>(v, bias);
}
template <int ACT>
__device__ __forceinline__ void ws_mul_dact(uint32_t (&v)[32], const float (&aux)[32], float s) {
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) * s * dact_from_out(ACT, aux[j]));
}
__device__ __forceinline__ void ws_mul_dact_rt(int act, uint32_t (&v)[32], const float (&aux)[32], float s) {
  if (act == ACT_RELU) ws_mul_dact<ACT_RELU>(v, aux, s);
  else if (act == ACT_TANH) ws_mul_dact<ACT_TANH>(v, aux, s);
  else ws_mul_dact<ACT_ELU>(v, aux, s);
}
// power of two 2^k with  bound * 2^k  in [512, 1024)  (1 for a zero / non-finite bound): the fp16 hi/lo planes then hold
// every element of the row with 22 significant bits relative to that bound and cannot saturate
__device__ __forceinline__ float ws_row_scale(float bound) {
  if (!(bound > 0.f) || !(bound < 3.0e38f)) return 1.f;
  int e;
  frexpf(bound, &e);                 // bound = m 2^e, m in [0.5, 1)
  e = 10 - e;
  e = e > 120 ? 120 : (e < -120 ? -120 : e);
  return ldexpf(1.f, e);
}

// ==========================================================================================
// forward:  h1 = act0(X W0 + b0);  h2 = act1(h1 W1 + b1);  out = h2 W2 + b2        (nn_utils.py:101-136)
// grid (row tiles, agents * nnet), 576 threads.  Multi-output nets (the actor) form the output layer on the tensor core
// from the W2 section of the plane image (N = N2 = 16 ceil(nout / 16)); single-output nets (the critics) on CUDA cores.
// Epilogue warp w: TMEM lane quarter q = w & 3 (rows 32q..32q+31 of the tile), column group cg = w >> 2 (columns
// 64cg..64cg+63 = the k group cg of the next layer).
// ==========================================================================================
struct FwdW {
  const float* X; int ldx; long long sXa, sXn;
  const float* theta; long long sTa, sTn;
  const uint8_t* planes; long long sPa, sPn;      // plane images (bytes): per agent / per net strides
  float* H1; float* H2; long long sHa, sHn;       // optional saved activations [rows, 256]
  uint8_t* H1p; long long sQa, sQn;               // optional bf16 hi/lo plane image of h1 (operand of k_dw_planes), bytes
  float* Out; int ldo; long long sOa, sOn;
  int rows, K0, nout, nnet, act0, act1;
  unsigned long long* dbg;                         // optional per-CTA phase stamps (16 per CTA, globaltimer ns)
};
#define WS_STAMP(i) do { if (f.dbg && lane == 0) f.dbg[(size_t)(blockIdx.y * gridDim.x + blockIdx.x) * 16 + (i)] = gtime(); } while (0)

__global__ void __launch_bounds__(WS_NT, 1) k_mlp_fwd_ws(FwdW f) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t ring = sb, aux = sb + WS_RING, patch_base = aux + WS_AUX, bars = sb + WS_MAIN, tslot = bars + 8 * 16;
  auto bar = [&](int i) { return bars + 8u * (uint32_t)i; };
  const int z = blockIdx.y, agent = z / f.nnet, net = z - agent * f.nnet;
  const int row0 = blockIdx.x * TC_BM;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = (f.K0 + 31) >> 5, nk64 = (f.K0 + 63) >> 6;
  const int N2 = ws_w2_rows(f.nout);            // 0: single output, formed on CUDA cores
  const uint32_t idesc_out = (1u << 4) | ((uint32_t)(N2 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);   // fp16, K-major, N = N2

  if (threadIdx.x == 0) {
    for (int s = 0; s < 2 * WS_NST; ++s) mbar_init(bar(s), 1);
    mbar_init(bar(WB_XFULL), WS_NEW); mbar_init(bar(WB_XEMPTY), 1);
    mbar_init(bar(WB_D0), 1); mbar_init(bar(WB_D1), 1); mbar_init(bar(WB_D2), 1);
    for (int g = 0; g < 4; ++g) mbar_init(bar(WB_AP + g), 8);     // 4 lane quarters x the 2 warps converting the group's two chunks
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == WS_NEW + 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tslot), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = lds_u32(tslot);
  const uint32_t tP = tmem, tQ = tmem + 256;

  if (warp == WS_NEW) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      const uint8_t* img = f.planes + agent * f.sPa + net * f.sPn;
      // W0 stages, W1 stages, then (multi-output nets) the W2 section as two items of two 64-wide j atoms each
      const int total = n0 + 8 + (N2 ? 2 : 0);
      const uint32_t w2_item = (uint32_t)N2 * 512;
      auto item_src = [&](int it) { return it < n0 + 8 ? img + (long long)it * WS_STAGE : img + (long long)(n0 + 8) * WS_STAGE + (it - n0 - 8) * w2_item; };
      for (int it = 0; it < total; ++it) {
        const int s = it % WS_NST;
        const uint32_t bytes = it < n0 + 8 ? (uint32_t)WS_STAGE : w2_item;
        mbar_wait(bar(WB_EMPTY + s), (uint32_t)(((it / WS_NST) & 1) ^ 1));
        mbar_expect_tx(bar(WB_FULL + s), bytes);
        bulk_g2s(ring + s * WS_STAGE, item_src(it), bytes, bar(WB_FULL + s));
        if (it == WS_NST - 1)      // ring primed: pull the rest of the image into L2 so that the refills are L2 hits
          for (int j = WS_NST; j < total; ++j) bulk_prefetch_l2(item_src(j), j < n0 + 8 ? (uint32_t)WS_STAGE : w2_item);
      }
      WS_STAMP(11);
    }
  } else if (warp == WS_NEW + 1) {
    // ------------------------------ MMA issuer ------------------------------
    if (lane == 0) {
      int it = 0;
      for (int sl = 0; sl < nk64; ++sl) {          // layer 0: D0 (tP) = X . W0, A = X planes in AUX (K-major), B = W0 stages
        mbar_wait(bar(WB_XFULL), (uint32_t)(sl & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        for (int hh = 0; hh < 2 && sl * 2 + hh < n0; ++hh, ++it) {
          const int s = it % WS_NST;
          mbar_wait(bar(WB_FULL + s), (uint32_t)((it / WS_NST) & 1));
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t st = ring + s * WS_STAGE;
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {
            const uint32_t ka = (uint32_t)(hh * 2 + kk) * 32, kb = (uint32_t)kk * 2048;
            umma_f16(tP, umma_desc(aux + ka), umma_desc_mn(st + kb), WS_IDESC_FWD, (it | kk) ? 1u : 0u);
            umma_f16(tP, umma_desc(aux + ka), umma_desc_mn(st + 16384 + kb), WS_IDESC_FWD, 1u);
            umma_f16(tP, umma_desc(aux + 16384 + ka), umma_desc_mn(st + kb), WS_IDESC_FWD, 1u);
          }
          umma_commit(bar(WB_EMPTY + s));
        }
        umma_commit(bar(WB_XEMPTY));
      }
      umma_commit(bar(WB_D0));
      WS_STAMP(8);
      for (int g = 0; g < 4; ++g) {                // layer 1: D1 (tQ) = h1 . W1, A = h1 hi/lo written in place over D0
        mbar_wait(bar(WB_AP + g), 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (g == 3) WS_STAMP(9);
        for (int tt = 0; tt < 2; ++tt, ++it) {
          const int t = 2 * g + tt, s = it % WS_NST;
          mbar_wait(bar(WB_FULL + s), (uint32_t)((it / WS_NST) & 1));
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t st = ring + s * WS_STAGE;
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {
            const uint32_t ta_hi = tP + 32 * t + 8 * kk, ta_lo = ta_hi + 16, kb = (uint32_t)kk * 2048;
            umma_f16_ts(tQ, ta_hi, umma_desc_mn(st + kb), WS_IDESC_FWD, (t | kk) ? 1u : 0u);
            umma_f16_ts(tQ, ta_hi, umma_desc_mn(st + 16384 + kb), WS_IDESC_FWD, 1u);
            umma_f16_ts(tQ, ta_lo, umma_desc_mn(st + kb), WS_IDESC_FWD, 1u);
          }
          umma_commit(bar(WB_EMPTY + s));
        }
      }
      umma_commit(bar(WB_D1));
      WS_STAMP(10);
      if (N2) {                                    // output layer: D2 (tP[0, N2)) = h2 . W2, A = h2 hi/lo written in place over D1
        for (int w = 0; w < 2; ++w, ++it) {        // ring item w holds the W2 atoms (k groups) 2w, 2w+1
          const int s = it % WS_NST;
          mbar_wait(bar(WB_FULL + s), (uint32_t)((it / WS_NST) & 1));
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          for (int gg = 0; gg < 2; ++gg) {
            const int g = 2 * w + gg;
            mbar_wait(bar(WB_AP + g), 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t bh = ring + s * WS_STAGE + (uint32_t)(gg * N2 * 256), bl = bh + (uint32_t)N2 * 128;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              const uint32_t ta_hi = tQ + 64 * g + 32 * (kk >> 1) + 8 * (kk & 1), ta_lo = ta_hi + 16, kb = (uint32_t)kk * 32;
              umma_f16_ts(tP, ta_hi, umma_desc(bh + kb), idesc_out, (g | kk) ? 1u : 0u);
              umma_f16_ts(tP, ta_hi, umma_desc(bl + kb), idesc_out, 1u);
              umma_f16_ts(tP, ta_lo, umma_desc(bh + kb), idesc_out, 1u);
            }
          }
          umma_commit(bar(WB_EMPTY + s));
        }
        umma_commit(bar(WB_D2));
      }
    }
  } else {
    // ------------------------------ conversion + epilogue warps ------------------------------
    const int q = warp & 3, cg = warp >> 2;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const uint32_t patch = patch_base + (uint32_t)warp * WS_PATCH1;
    const int rbase = row0 + q * 32, grow = rbase + lane;
    const float* __restrict__ X = f.X + agent * f.sXa + net * f.sXn;
    const float* __restrict__ th = f.theta + agent * f.sTa + net * f.sTn;
    const long long ob0 = (long long)f.K0 * FW_H, oW1 = ob0 + FW_H, ob1 = oW1 + (long long)FW_H * FW_H,
                    oW2 = ob1 + FW_H, ob2 = oW2 + (long long)FW_H * f.nout;
    float* H1 = f.H1 ? f.H1 + agent * f.sHa + net * f.sHn : nullptr;
    float* H2 = f.H2 ? f.H2 + agent * f.sHa + net * f.sHn : nullptr;
    float* Out = f.Out + agent * f.sOa + net * f.sOn;
    if (warp == 0) WS_STAMP(0);
    // per-CTA constants -> shared memory: b0 | b1 | w2 (single-output nets) | b2
    const uint32_t cb0 = aux + WS_RED + 2048, cb1 = cb0 + 1024, cw2 = cb1 + 1024, cb2 = cw2 + 1024;
    if (threadIdx.x < FW_H) {
      const int t = threadIdx.x;
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(cb0 + t * 4), "f"(__ldg(th + ob0 + t)) : "memory");
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(cb1 + t * 4), "f"(__ldg(th + ob1 + t)) : "memory");
      if (f.nout == 1) asm volatile("st.shared.f32 [%0], %1;" ::"r"(cw2 + t * 4), "f"(__ldg(th + oW2 + t)) : "memory");
      if (t < f.nout) asm volatile("st.shared.f32 [%0], %1;" ::"r"(cb2 + t * 4), "f"(__ldg(th + ob2 + t)) : "memory");
    }
    {   // input tile -> fp16 hi/lo K-major planes (A operand of layer 0), one 64-wide k slab at a time
      Slab<TC_BM, WS_NEPI> sx;
      sx.init(X, f.ldx, 1, row0, f.rows);
      for (int sl = 0; sl < nk64; ++sl) {
        sx.ld(sl * 64, f.K0);
        if (sl > 0) mbar_wait(bar(WB_XEMPTY), (uint32_t)((sl - 1) & 1));
        sx.template st<true>(aux, aux + 16384);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(WB_XFULL));
      }
    }
    epi_bar();                                        // constants visible
    if (warp == 0) WS_STAMP(1);
    // ---- epilogue 0: h1 = act0(D0 + b0) -> fp16 hi/lo in place (A operand of layer 1) [+ saved h1]
    mbar_wait(bar(WB_D0), 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (warp == 0) WS_STAMP(2);
    // chunk order by k group: in step c the 16 warps convert k groups 2c and 2c+1 (warp pair cg>>1 takes one group, cg&1 its
    // 32-column half), so the layer-1 MMAs of groups 0 / 1 - and the W1 stages behind them - start after HALF of this
    // epilogue instead of at its end (the W1 stream through the 3-deep ring was two TMA round trips behind the last group)
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
      const int kg = 2 * c + (cg >> 1), col = kg * 64 + (cg & 1) * 32;
      uint32_t v[32];
      tmem_ld32(tP + lane_addr + (uint32_t)col, v);
      ws_bias_act_rt(f.act0, v, cb0 + col * 4);
      ws_split_store(tP + lane_addr + (uint32_t)col, v, 1.f);
      {
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(WB_AP + kg));      // the layer-1 MMAs of this 64-wide k group may start
      }
      if (f.H1p) {          // h1 leaves as a bf16 hi/lo plane image only (operand of k_dw_planes, read back by the backward chain)
#pragma unroll
        for (int j = 0; j < 8; ++j) sts128(ws_pa(patch, lane, 4 * j), make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
        __syncwarp();
        ws_store_planes_p(patch, f.H1p + agent * f.sQa + net * f.sQn, rbase, f.rows, col, lane);
        __syncwarp();
      } else if (H1) { ws_store_rows(patch, v, H1, rbase, f.rows, col, lane); __syncwarp(); }
    }
    if (warp == 0) WS_STAMP(3);
    if (warp == 0) WS_STAMP(4);
    mbar_wait(bar(WB_D1), 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (warp == 0) WS_STAMP(5);
    if (N2) {
      // ---- epilogue 1: h2 = act1(D1 + b1) -> fp16 hi/lo in place (A operand of the output layer) [+ saved h2], k groups in
      //      the order of epilogue 0, so that the output-layer MMAs of groups 0 / 1 start after half of it
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        const int kg = 2 * c + (cg >> 1), col = kg * 64 + (cg & 1) * 32;
        uint32_t v[32];
        tmem_ld32(tQ + lane_addr + (uint32_t)col, v);
        ws_bias_act_rt(f.act1, v, cb1 + col * 4);
        ws_split_store(tQ + lane_addr + (uint32_t)col, v, 1.f);
        {
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive(bar(WB_AP + kg));      // second phase of the k-group barrier: output-layer MMAs of group kg
        }
        if (H2) { ws_store_rows(patch, v, H2, rbase, f.rows, col, lane); __syncwarp(); }
      }
      if (warp == 0) WS_STAMP(6);
      // ---- out = D2 / WS_W2_SCALE + b2: column group 0 reads its rows' N2 accumulator columns
      if (cg == 0) {
        mbar_wait(bar(WB_D2), 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        for (int r0 = 0; r0 < N2; r0 += 32) {
          uint32_t v[32];
          tmem_ld32(tP + lane_addr + (uint32_t)r0, v);
          if (grow < f.rows) {
#pragma unroll
            for (int cc = 0; cc < 32; ++cc)
              if (r0 + cc < f.nout) Out[(long long)grow * f.ldo + r0 + cc] = __uint_as_float(v[cc]) * (1.f / WS_W2_SCALE) + lds32(cb2 + (uint32_t)(r0 + cc) * 4);
          }
        }
      }
    } else {
      // ---- epilogue 1: h2 = act1(D1 + b1) [+ saved h2]; out = h2 . w2 + b2 on CUDA cores (exact fp32), fixed-order sum of
      //      the four column groups
      float qacc = 0.f;
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        const int col = cg * 64 + c * 32;
        uint32_t v[32];
        tmem_ld32(tQ + lane_addr + (uint32_t)col, v);
        ws_bias_act_rt(f.act1, v, cb1 + col * 4);
        if (H2) { ws_store_rows(patch, v, H2, rbase, f.rows, col, lane); __syncwarp(); }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 t4 = lds128(cw2 + (uint32_t)(col + 4 * j) * 4);
          qacc = fmaf(__uint_as_float(v[4 * j]), t4.x, qacc); qacc = fmaf(__uint_as_float(v[4 * j + 1]), t4.y, qacc);
          qacc = fmaf(__uint_as_float(v[4 * j + 2]), t4.z, qacc); qacc = fmaf(__uint_as_float(v[4 * j + 3]), t4.w, qacc);
        }
      }
      if (warp == 0) WS_STAMP(6);
      const uint32_t red = aux + WS_RED;             // [3 groups][128 rows] scratch
      if (cg > 0) asm volatile("st.shared.f32 [%0], %1;" ::"r"(red + (uint32_t)((cg - 1) * TC_BM + q * 32 + lane) * 4), "f"(qacc) : "memory");
      epi_bar();
      if (cg == 0 && grow < f.rows) {
        const uint32_t r = red + (uint32_t)(q * 32 + lane) * 4;
        Out[(long long)grow * f.ldo] = ((qacc + lds32(r)) + (lds32(r + TC_BM * 4) + lds32(r + 2 * TC_BM * 4))) + lds32(cb2);
      }
    }
    if (warp == 0) WS_STAMP(7);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == WS_NEW + 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512) : "memory");
  }
}

// ==========================================================================================
// backward chain (weights fixed):
//     dH2 = (dOut W2[:, :kout]^T) * act1'(H2);   dH1 = (dH2 W1^T) * act0'(H1);   dXa = dH1 W0[S:S+A, :]^T
// grid (row tiles, agents * nnet), 576 threads.  NG = ceil(kout / 16), NA = ceil(a_cols / 16) (0: no dXa).
// ==========================================================================================
struct BwdW {
  const float* dOut; int ldd; long long sDa, sDn; int kout;
  const float* theta; long long sTa, sTn; int K0, nout;
  const uint8_t* planes; long long sPa, sPn;
  const float* H1; const float* H2; long long sHa, sHn;
  float* dH2; float* dH1;
  uint8_t* dH2p; long long sQa, sQn;               // optional bf16 hi/lo plane image of dH2 (replaces the fp32 dH2), bytes
  uint8_t* dH1p;                                   // optional plane image of dH1 (operand of k_dw0_planes; same strides)
  const uint8_t* H1p;                              // optional: h1 as a bf16 hi/lo plane image (then H1 is not read), strides sQa / sQn
  float* dXa; int s_cols, a_cols; long long sXa, sXn;
  int rows, nnet, act0, act1;
  float* dbpart;
  unsigned long long* dbg;
};

// MODE specialises the saved-activation / gradient-output forms at compile time (fewer live pointers and no dead
// alternative paths under the 96-register cap): 0 = decided at run time; 1 = the training form (h1 read from its plane
// image, dH2 and dH1 leave as plane images only); 2 = input gradient only (h1 from its plane image, nothing saved)
template <int NG, int NA, int MODE>
__global__ void __launch_bounds__(WS_NT, 1) k_mlp_bwd_ws(BwdW f) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t ring = sb, aux = sb + WS_RING, patch_base = aux + WS_AUX, bars = sb + WS_MAIN, tslot = bars + 8 * 16;
  const uint32_t cs2 = aux + WS_RED, cs1 = cs2 + 4096;
  auto bar = [&](int i) { return bars + 8u * (uint32_t)i; };
  const int z = blockIdx.y, agent = z / f.nnet, net = z - agent * f.nnet;
  const int row0 = blockIdx.x * TC_BM;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = (f.K0 + 31) >> 5;

  if (threadIdx.x == 0) {
    for (int s = 0; s < 2 * WS_NST; ++s) mbar_init(bar(s), 1);
    mbar_init(bar(WB_D0), 1); mbar_init(bar(WB_D1), 1);                 // accumulator halves 0 / 1
    for (int g = 0; g < 4; ++g) mbar_init(bar(WB_AP + g), 8);     // 4 lane quarters x the 2 warps converting the group's two chunks
    mbar_init(bar(WB_XFULL), 4); mbar_init(bar(WB_XEMPTY), 1);    // NG > 0: dOut operand written (4 lane quarters) / dOut W2^T formed
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(aux + WS_RED - 256), "r"(0u) : "memory");     // max |W2| accumulator
  }
  if (warp == WS_NEW + 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tslot), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = lds_u32(tslot);
  const uint32_t tP = tmem, tQ = tmem + 256;

  if (warp == WS_NEW) {
    // TMA producer: stage (h, s) = rows i in [128h, 128h+128) of the 64-wide j slab s, K-major: 4 KB pieces (t, plane, s)
    if (lane == 0) {
      const uint8_t* w1 = f.planes + agent * f.sPa + net * f.sPn + (long long)n0 * WS_STAGE;
      if (NG > 0) {   // multi-output nets: first the W2 section (planes.cuh), ring item 0 = its hi plane, item 1 = its lo plane,
                      // each compacted to [s][n][64 j] (the 64-wide j atoms N2 * 128 bytes apart)
        const int N2 = ws_w2_rows(f.nout);
        const uint8_t* w2 = w1 + 8LL * WS_STAGE;
        for (int pl = 0; pl < 2; ++pl) {
          mbar_expect_tx(bar(WB_FULL + pl), (uint32_t)N2 * 512);
          for (int sj = 0; sj < 4; ++sj)
            bulk_g2s(ring + pl * WS_STAGE + sj * N2 * 128, w2 + (sj * 2 + pl) * N2 * 128, (uint32_t)N2 * 128, bar(WB_FULL + pl));
        }
      }
      for (int i = 0; i < 8; ++i) {
        const int it = i + (NG > 0 ? 2 : 0), h = i >> 2, sj = i & 3, s = it % WS_NST;
        mbar_wait(bar(WB_EMPTY + s), (uint32_t)(((it / WS_NST) & 1) ^ 1));
        mbar_expect_tx(bar(WB_FULL + s), WS_STAGE);
        for (int pl = 0; pl < 2; ++pl)
          for (int tt = 0; tt < 4; ++tt)
            bulk_g2s(ring + s * WS_STAGE + pl * 16384 + tt * 4096,
                     w1 + (long long)(4 * h + tt) * WS_STAGE + pl * 16384 + sj * 4096, 4096, bar(WB_FULL + s));
        if (it == WS_NST - 1)
          for (int t = 0; t < 8; ++t) bulk_prefetch_l2(w1 + (long long)t * WS_STAGE, WS_STAGE);
      }
    }
  } else if (warp == WS_NEW + 1) {
    if (lane == 0) {
      if (NG > 0) {     // D0 (tP) = dOut' . W2^T: A = the scaled dOut rows as fp16 hi/lo in tQ, B = the W2 planes read MN-major
        const uint32_t lbo = (uint32_t)ws_w2_rows(f.nout) * 128;
        mbar_wait(bar(WB_XFULL), 0);
        mbar_wait(bar(WB_FULL + 0), 0);
        mbar_wait(bar(WB_FULL + 1), 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
        for (int ks = 0; ks < NG; ++ks) {
          const uint32_t ta_hi = tQ + 16 * ks, ta_lo = ta_hi + 8, kb = (uint32_t)ks * 2048;
          umma_f16_ts(tP, ta_hi, umma_desc_mn(ring + kb, lbo), WS_IDESC_FWD, ks ? 1u : 0u);
          umma_f16_ts(tP, ta_hi, umma_desc_mn(ring + WS_STAGE + kb, lbo), WS_IDESC_FWD, 1u);
          umma_f16_ts(tP, ta_lo, umma_desc_mn(ring + kb, lbo), WS_IDESC_FWD, 1u);
        }
        umma_commit(bar(WB_EMPTY + 0));
        umma_commit(bar(WB_EMPTY + 1));
        umma_commit(bar(WB_XEMPTY));
      }
      for (int i = 0; i < 8; ++i) {             // D1[:, 128h..] (tQ) = dH2' . W1^T, contraction over the j slab sj
        const int it = i + (NG > 0 ? 2 : 0), h = i >> 2, sj = i & 3, s = it % WS_NST;
        if (h == 0) {
          mbar_wait(bar(WB_AP + sj), 0);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        mbar_wait(bar(WB_FULL + s), (uint32_t)((it / WS_NST) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t st = ring + s * WS_STAGE;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const int ks = sj * 4 + kk;
          const uint32_t ta_hi = tP + 32 * (ks >> 1) + 8 * (ks & 1), ta_lo = ta_hi + 16, kb = (uint32_t)kk * 32;
          umma_f16_ts(tQ + 128 * h, ta_hi, umma_desc(st + kb), WS_IDESC_BWD, (sj | kk) ? 1u : 0u);
          umma_f16_ts(tQ + 128 * h, ta_hi, umma_desc(st + 16384 + kb), WS_IDESC_BWD, 1u);
          umma_f16_ts(tQ + 128 * h, ta_lo, umma_desc(st + kb), WS_IDESC_BWD, 1u);
        }
        umma_commit(bar(WB_EMPTY + s));
        if (sj == 3) { umma_commit(bar(h ? WB_D1 : WB_D0)); WS_STAMP(8 + h); }
      }
    }
  } else {
    const int q = warp & 3, cg = warp >> 2;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const uint32_t patch = patch_base + (uint32_t)warp * WS_PATCH1;
    const int rbase = row0 + q * 32, grow = rbase + lane;
    const bool rvalid = grow < f.rows;
    const float* __restrict__ dOut = f.dOut + agent * f.sDa + net * f.sDn;
    const float* __restrict__ th = f.theta + agent * f.sTa + net * f.sTn;
    const long long ob0 = (long long)f.K0 * FW_H, oW1 = ob0 + FW_H, ob1 = oW1 + (long long)FW_H * FW_H, oW2 = ob1 + FW_H;
    const float* H1 = f.H1 + agent * f.sHa + net * f.sHn;
    const float* H2 = f.H2 + agent * f.sHa + net * f.sHn;
    float* dH1 = (MODE == 0 && f.dH1) ? f.dH1 + agent * f.sHa + net * f.sHn : nullptr;
    float* dH2 = (MODE == 0 && f.dH2) ? f.dH2 + agent * f.sHa + net * f.sHn : nullptr;
    const bool pH1 = MODE != 0 || f.H1p != nullptr;
    const bool pdH2 = MODE == 1 || (MODE == 0 && f.dH2p != nullptr), pdH1 = MODE == 1 || (MODE == 0 && f.dH1p != nullptr);
    const bool want_cs = f.dbpart && (dH2 || pdH2) && (dH1 || pdH1);
    const uint32_t wmax_s = aux + WS_RED - 256;            // max |W2[:, :kout]| (int bit pattern)

    if (warp == 0) WS_STAMP(0);
    // chunk order of epilogue 0 by k group (as in the forward kernel): step c converts the j slabs 2c and 2c+1
    const int col0_0 = (cg >> 1) * 64 + (cg & 1) * 32, col0_1 = (2 + (cg >> 1)) * 64 + (cg & 1) * 32;
    ws_rows_prefetch(H2, rbase, f.rows, col0_0, lane);      // saved activations of both chunks -> L2 while W2 is staged
    ws_rows_prefetch(H2, rbase, f.rows, col0_1, lane);
    const float* __restrict__ drow = dOut + (long long)grow * f.ldd;
    // max |W2[:, :kout]| bounds every row of dOut . W2^T (row scale of the dH2 operand)
    float d0 = 0.f, bound = 0.f, inv_d = 1.f;
    if (NG == 0) {       // single output (critics): the first step is an outer product with w2 staged as fp32 in AUX
      d0 = rvalid ? __ldg(drow) : 0.f;
      bound = fabsf(d0);
      if (threadIdx.x < FW_H) {
        float wr[4];
        ws_load_wrow<4>(th + oW2, threadIdx.x, f.nout, wr);          // hidden unit j = threadIdx.x
        float m = fabsf(wr[0]);
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(aux + threadIdx.x * 4), "f"(wr[0]) : "memory");
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) atomicMax(reinterpret_cast<int*>(smem_raw + (wmax_s - smem_u32(smem_raw))), __float_as_int(m));
      }
    } else {
      // multi-output nets (actor): dOut . W2^T on the tensor core.  The dOut row goes in as fp16 hi/lo scaled by a power of
      // two that puts its largest element in [512, 1024); the accumulator then holds dH2 * dscale * WS_W2_SCALE
      float dmax = 0.f;
      for (int cc = 0; cc < f.kout; ++cc) {
        const float x = rvalid ? fabsf(__ldg(drow + cc)) : 0.f;
        bound += x; dmax = fmaxf(dmax, x);
      }
      const float dscale = ws_row_scale(dmax);
      inv_d = (1.f / dscale) * (1.f / WS_W2_SCALE);
      if (cg == 0) {     // one warp per lane quarter writes the A operand: K = 16 NG columns, [8 hi | 8 lo] per 16-wide k step
#pragma unroll
        for (int ks = 0; ks < NG; ++ks) {
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int c0 = 16 * ks + 2 * j;
            const float x0 = (rvalid && c0 < f.kout) ? __ldg(drow + c0) * dscale : 0.f;
            const float x1 = (rvalid && c0 + 1 < f.kout) ? __ldg(drow + c0 + 1) * dscale : 0.f;
            asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi[j]) : "f"(x1), "f"(x0));
            const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi[j]));
            asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo[j]) : "f"(x1 - hf.y), "f"(x0 - hf.x));
          }
          tmem_st8(tQ + lane_addr + 16 * ks, hi);
          tmem_st8(tQ + lane_addr + 16 * ks + 8, lo);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(WB_XFULL));
      }
      if (threadIdx.x < FW_H) {
        float m = 0.f;
        const float* wr = th + oW2 + (long long)threadIdx.x * f.nout;
        for (int cc = 0; cc < f.kout; ++cc) m = fmaxf(m, fabsf(__ldg(wr + cc)));
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) atomicMax(reinterpret_cast<int*>(smem_raw + (wmax_s - smem_u32(smem_raw))), __float_as_int(m));
      }
    }
    epi_bar();
    // this row's scale: |dH2[row, j]| <= sum_c |dOut[row, c]| * max |W2|
    bound *= __int_as_float((int)lds_u32(wmax_s));
    const float scale = ws_row_scale(bound), inv_scale = 1.f / scale;
    if (warp == 0) WS_STAMP(1);

    // ---- epilogue 0: dH2 = (dOut . W2^T) * act1'(H2) -> scaled fp16 hi/lo A operand in place (tP) [+ saved dH2, column sums]
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
      const int col = c ? col0_1 : col0_0, kg = 2 * c + (cg >> 1);
      {
        float4 hq[8];
        ws_rows_issue(H2, rbase, f.rows, col, lane, hq);
        ws_rows_commit_p(patch, lane, hq);
      }
      if (c == 1) {        // the H1 tiles of epilogue 1 -> L2 during the MMAs
        if (!pH1) { ws_rows_prefetch(H1, rbase, f.rows, cg * 64, lane); ws_rows_prefetch(H1, rbase, f.rows, cg * 64 + 32, lane); }
        else ws_planes_prefetch(f.H1p + agent * f.sQa + net * f.sQn, rbase, f.rows, cg * 64, lane);
      }
      uint32_t v[32];
      if (NG == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 t4 = lds128(aux + (uint32_t)(col + 4 * j) * 4);
          v[4 * j] = __float_as_uint(d0 * t4.x); v[4 * j + 1] = __float_as_uint(d0 * t4.y);
          v[4 * j + 2] = __float_as_uint(d0 * t4.z); v[4 * j + 3] = __float_as_uint(d0 * t4.w);
        }
      } else {
        if (c == 0) {
          mbar_wait(bar(WB_XEMPTY), 0);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        tmem_ld32(tP + lane_addr + (uint32_t)col, v);
      }
      ws_mul_dact_p_rt(f.act1, v, patch, lane, inv_d);
      ws_split_store(tP + lane_addr + (uint32_t)col, v, scale);
      {
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(WB_AP + kg));
      }
      if (pdH2 && !dH2) {
        ws_store_planes_cs(patch, v, f.dH2p + agent * f.sQa + net * f.sQn, rbase, f.rows, col, lane, want_cs ? cs2 : 0u, q);
        __syncwarp();
      } else if (dH2 || pdH2) {
        ws_store_rows(patch, v, dH2, rbase, f.rows, col, lane, want_cs ? cs2 : 0u, q);
        if (pdH2) ws_store_planes_p(patch, f.dH2p + agent * f.sQa + net * f.sQn, rbase, f.rows, col, lane);
        __syncwarp();
      }
    }
    if (warp == 0) WS_STAMP(2);
    // ---- action rows of W0, transposed: W0aT[j][ap] fp32 (the W2 stage is dead once every warp has left epilogue 0)
    const int ap = (f.a_cols + 3) & ~3;
    if (NA > 0) {
      epi_bar();
      if (threadIdx.x < FW_H) {
        const int j = threadIdx.x;
        for (int a = 0; a < ap; ++a) {
          const float w = a < f.a_cols ? __ldg(th + (long long)(f.s_cols + a) * FW_H + j) : 0.f;
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(aux + (uint32_t)(j * ap + a) * 4), "f"(w) : "memory");
        }
      }
      epi_bar();
    }
    // ---- epilogue 1: dH1 = (D1 / scale) * act0'(H1) [+ saved dH1, column sums]; dXa = dH1 . W0a^T on CUDA cores
    if (warp == 0) WS_STAMP(3);
    mbar_wait(bar(cg >= 2 ? WB_D1 : WB_D0), 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (warp == 0) WS_STAMP(4);
    if (warp == 8) WS_STAMP(12);
    float xa[NA > 0 ? NA * 16 : 1];
#pragma unroll
    for (int i = 0; i < (NA > 0 ? NA * 16 : 1); ++i) xa[i] = 0.f;
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
      const int col = cg * 64 + c * 32;
      uint32_t v[32];
      tmem_ld32_nw(tQ + lane_addr + (uint32_t)col, v);
      {
        float4 hq[8];
        if (pH1) {        // h1 from its plane image, decoded into the patch
          ws_planes_issue(f.H1p + agent * f.sQa + net * f.sQn, rbase, f.rows, col, lane, hq);
          ws_planes_commit_p(patch, lane, hq);
        } else {
          ws_rows_issue(H1, rbase, f.rows, col, lane, hq);
          ws_rows_commit_p(patch, lane, hq);
        }
      }
      tmem_ld_wait();
      ws_mul_dact_p_rt(f.act0, v, patch, lane, inv_scale);
      if (pdH1 && !dH1) {
        ws_store_planes_cs(patch, v, f.dH1p + agent * f.sQa + net * f.sQn, rbase, f.rows, col, lane, want_cs ? cs1 : 0u, q);
        __syncwarp();
      } else if (dH1 || pdH1) {
        ws_store_rows(patch, v, dH1, rbase, f.rows, col, lane, want_cs ? cs1 : 0u, q);
        if (pdH1) ws_store_planes_p(patch, f.dH1p + agent * f.sQa + net * f.sQn, rbase, f.rows, col, lane);
        __syncwarp();
      }
      if (NA > 0) {
#pragma unroll
        for (int jj = 0; jj < 32; ++jj) {
          const float g = __uint_as_float(v[jj]);
          const uint32_t wrow = aux + (uint32_t)((col + jj) * ap) * 4;
#pragma unroll
          for (int g4 = 0; g4 < (NA > 0 ? NA * 4 : 1); ++g4) {
            if (g4 * 4 < ap) {
              const float4 w = lds128(wrow + g4 * 16);
              xa[4 * g4] = fmaf(g, w.x, xa[4 * g4]); xa[4 * g4 + 1] = fmaf(g, w.y, xa[4 * g4 + 1]);
              xa[4 * g4 + 2] = fmaf(g, w.z, xa[4 * g4 + 2]); xa[4 * g4 + 3] = fmaf(g, w.w, xa[4 * g4 + 3]);
            }
          }
        }
      }
    }
    if (warp == 0) WS_STAMP(5);
    if (warp == 8) WS_STAMP(13);
    if (NA > 0) {      // fixed-order sum of the four column groups -> dXa[row, :a_cols]
      if (cg > 0) {
#pragma unroll
        for (int cc = 0; cc < (NA > 0 ? NA * 16 : 1); ++cc)
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(patch + (uint32_t)(lane * 32 + ((cc + lane) & 31)) * 4), "f"(xa[cc]) : "memory");
      }
      epi_bar();
      if (cg == 0 && rvalid) {
        float* o = f.dXa + agent * f.sXa + net * f.sXn + (long long)grow * f.a_cols;
#pragma unroll
        for (int cc = 0; cc < (NA > 0 ? NA * 16 : 1); ++cc) {
          if (cc < f.a_cols) {
            const uint32_t po = (uint32_t)(lane * 32 + ((cc + lane) & 31)) * 4;
            const float p1 = lds32(patch_base + (uint32_t)(warp + 4) * WS_PATCH1 + po), p2 = lds32(patch_base + (uint32_t)(warp + 8) * WS_PATCH1 + po),
                        p3 = lds32(patch_base + (uint32_t)(warp + 12) * WS_PATCH1 + po);
            o[cc] = (xa[cc] + p1) + (p2 + p3);
          }
        }
      }
    }
    if (want_cs) {     // fixed-order sum of the four row quarters -> per-tile bias-gradient partials
      epi_bar();
      if (threadIdx.x < FW_H) {
        const int t = threadIdx.x;
#pragma unroll
        for (int which = 0; which < 2; ++which) {
          const uint32_t b = (which ? cs1 : cs2) + (uint32_t)t * 4;
          const float s = ((lds32(b) + lds32(b + FW_H * 4)) + lds32(b + 2 * FW_H * 4)) + lds32(b + 3 * FW_H * 4);
          f.dbpart[(((long long)z * gridDim.x + blockIdx.x) * 2 + which) * FW_H + t] = s;
        }
      }
    }
    if (warp == 0) WS_STAMP(7);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == WS_NEW + 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512) : "memory");
  }
}

// ==========================================================================================
// Weight gradient of the hidden-to-hidden layer from the activation plane images:
//     dW1[i, j] = sum_b h1[b, i] * dH2[b, j]          (one CTA per (agent, net): the whole 256 x 256 block)
// Both operands arrive by TMA as bf16 hi/lo planes written by the fused forward (h1) and backward (dH2) kernels -
// MN-major SWIZZLE_128B operands with the batch row as the contraction index, 32 rows (64 KB: A + B) per stage - so
// the kernel converts nothing: producer warp, MMA thread (two 128-row accumulator blocks = all 512 TMEM columns,
// 3 MMAs per product), 16 epilogue warps that write the fp32 gradient block through the transposition patches.
// Replaces the cp.async + in-kernel-conversion GEMM for this shape (85 + 170 us per step at 256 agents -> see DESIGN).
// ==========================================================================================
struct DwP {
  const uint8_t* Ap; long long sAa, sAn;      // h1 planes  [rows(pad 32) x 256]
  const uint8_t* Bp; long long sBa, sBn;      // dH2 planes
  float* G; long long sGa, sGn;               // gradient block W1 of the flat layout (pitch 256)
  int rows, nnet;
};
constexpr int DW_STAGE = 2 * WS_STAGE, DW_NST = 3;
constexpr int DW_MAIN = DW_NST * DW_STAGE;                       // 192 KB; the epilogue patches overlay the ring
constexpr int DW_BYTES = DW_MAIN + 1024 + 256;
constexpr uint32_t DW_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

__global__ void __launch_bounds__(WS_NT, 1) k_dw_planes(DwP f) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t ring = sb, bars = sb + DW_MAIN, tslot = bars + 8 * 16;
  auto bar = [&](int i) { return bars + 8u * (uint32_t)i; };          // [0..3) full, [3..6) empty, [6] done
  const int z = blockIdx.x, agent = z / f.nnet, net = z - agent * f.nnet;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nst = (f.rows + 31) >> 5;
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2 * DW_NST + 1; ++s) mbar_init(bar(s), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == WS_NEW + 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tslot), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = lds_u32(tslot);
  if (warp == WS_NEW) {
    if (lane == 0) {
      const uint8_t* A = f.Ap + agent * f.sAa + net * f.sAn;
      const uint8_t* B = f.Bp + agent * f.sBa + net * f.sBn;
      for (int it = 0; it < nst; ++it) {
        const int s = it % DW_NST;
        mbar_wait(bar(DW_NST + s), (uint32_t)(((it / DW_NST) & 1) ^ 1));
        mbar_expect_tx(bar(s), DW_STAGE);
        bulk_g2s(ring + s * DW_STAGE, A + (long long)it * WS_STAGE, WS_STAGE, bar(s));
        bulk_g2s(ring + s * DW_STAGE + WS_STAGE, B + (long long)it * WS_STAGE, WS_STAGE, bar(s));
      }
    }
  } else if (warp == WS_NEW + 1) {
    if (lane == 0) {
      for (int it = 0; it < nst; ++it) {
        const int s = it % DW_NST;
        mbar_wait(bar(s), (uint32_t)((it / DW_NST) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sa = ring + s * DW_STAGE, sbb = sa + WS_STAGE;
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
          const uint32_t ko = (uint32_t)kk * 2048;
#pragma unroll
          for (int mb = 0; mb < 2; ++mb) {          // accumulator block mb: gradient rows i in [128 mb, 128 mb + 128)
            const uint32_t a_hi = sa + mb * 8192 + ko, a_lo = a_hi + 16384, b_hi = sbb + ko, b_lo = b_hi + 16384;
            const uint32_t d = tmem + 256 * mb, acc = (it | kk) ? 1u : 0u;
            umma_f16(d, umma_desc_mn(a_hi), umma_desc_mn(b_hi), DW_IDESC, acc);
            umma_f16(d, umma_desc_mn(a_hi), umma_desc_mn(b_lo), DW_IDESC, 1u);
            umma_f16(d, umma_desc_mn(a_lo), umma_desc_mn(b_hi), DW_IDESC, 1u);
          }
        }
        umma_commit(bar(DW_NST + s));
      }
      umma_commit(bar(2 * DW_NST));
    }
  } else {
    const int q = warp & 3, cg = warp >> 2;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const uint32_t patch = ring + (uint32_t)warp * WS_PATCH1;         // the operand ring is dead once the last MMA has retired
    float* G = f.G + agent * f.sGa + net * f.sGn;
    mbar_wait(bar(2 * DW_NST), 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
    for (int mb = 0; mb < 2; ++mb) {
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        const int col = cg * 64 + c * 32;
        uint32_t v[32];
        tmem_ld32(tmem + lane_addr + (uint32_t)(256 * mb + col), v);
        ws_store_rows(patch, v, G, mb * 128 + q * 32, 256, col, lane);
        __syncwarp();
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == WS_NEW + 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512) : "memory");
  }
}

// ==========================================================================================
// Weight gradient of the first layer from the dH1 plane image:
//     dW0[i, j] = sum_b X[b, i] * dH1[b, j]           (one CTA per (agent, net), in <= 64 inputs)
// B = dH1 planes by TMA exactly like k_dw_planes; A = the input rows X (fp32, a few dozen columns), converted ONCE by the
// epilogue warps into bf16 hi/lo MN-major stages in shared memory (8 KB per 32 batch rows: [plane][32 rows][64 inputs])
// while the first dH1 stages are in flight.  One 128-row accumulator of which rows [0, in) are the gradient block (the M
// atom stride of the shared descriptor form makes rows 64.. a by-product of the neighbouring plane; never read).
// Replaces the cp.async + in-kernel-conversion GEMM for this shape (82 + 47 us per step at 256 agents).
// ==========================================================================================
struct Dw0P {
  const float* X; int ldx; long long sXa, sXn;     // input rows [rows x in] (row stride ldx floats, 16-byte aligned)
  const uint8_t* Bp; long long sBa, sBn;           // dH1 planes
  float* G; long long sGa, sGn;                    // gradient block W0 of the flat layout (pitch 256)
  int rows, in, nnet;
};
constexpr int DW0_NST = 3, DW0_RING = DW0_NST * WS_STAGE, DW0_XST = 8192, DW0_MAXST = 14;
constexpr int DW0_BYTES = DW0_RING + DW0_MAXST * DW0_XST + 4096 + 1024 + 256;

__global__ void __launch_bounds__(WS_NT, 1) k_dw0_planes(Dw0P f) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t ring = sb, xs = sb + DW0_RING, bars = xs + DW0_MAXST * DW0_XST + 4096, tslot = bars + 8 * 16;
  auto bar = [&](int i) { return bars + 8u * (uint32_t)i; };          // [0..3) full, [3..6) empty, [6] done, [7] X stages ready
  const int z = blockIdx.x, agent = z / f.nnet, net = z - agent * f.nnet;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nst = (f.rows + 31) >> 5;
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2 * DW0_NST + 2; ++s) mbar_init(bar(s), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == WS_NEW + 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tslot), "n"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = lds_u32(tslot);
  if (warp == WS_NEW) {
    if (lane == 0) {
      const uint8_t* B = f.Bp + agent * f.sBa + net * f.sBn;
      for (int it = 0; it < nst; ++it) {
        const int s = it % DW0_NST;
        mbar_wait(bar(DW0_NST + s), (uint32_t)(((it / DW0_NST) & 1) ^ 1));
        mbar_expect_tx(bar(s), WS_STAGE);
        bulk_g2s(ring + s * WS_STAGE, B + (long long)it * WS_STAGE, WS_STAGE, bar(s));
      }
    }
  } else if (warp < WS_NEW) {
    // X -> bf16 hi/lo MN-major stages: item = (batch row, 8-input chunk); zeros beyond rows / in
    const float* X = f.X + agent * f.sXa + net * f.sXn;
    for (int it = threadIdx.x; it < nst * 32 * 8; it += WS_NEPI) {
      const int b = it >> 3, c8 = it & 7, t = b >> 5, r = b & 31;
      float x8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) x8[j] = 0.f;
      if (b < f.rows && 8 * c8 < f.in) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(X + (long long)b * f.ldx + 8 * c8));
        const float4 c = 8 * c8 + 4 < f.in ? __ldg(reinterpret_cast<const float4*>(X + (long long)b * f.ldx + 8 * c8 + 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float v8[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) x8[j] = 8 * c8 + j < f.in ? v8[j] : 0.f;
      }
      uint4 hi, lo;
      split8<false>(x8, hi, lo);
      const uint32_t dst = xs + (uint32_t)t * DW0_XST + (uint32_t)r * 128 + (uint32_t)((c8 ^ (r & 7)) << 4);
      sts128(dst, hi); sts128(dst + 4096, lo);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    epi_bar();                                       // the 16 conversion warps only (the producer is busy with its ring)
    if (threadIdx.x == 0) mbar_arrive(bar(2 * DW0_NST + 1));          // the X stages are complete and visible to the tensor core
  }
  if (warp == WS_NEW + 1) {
    if (lane == 0) {
      mbar_wait(bar(2 * DW0_NST + 1), 0);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      for (int it = 0; it < nst; ++it) {
        const int s = it % DW0_NST;
        mbar_wait(bar(s), (uint32_t)((it / DW0_NST) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sa = xs + (uint32_t)it * DW0_XST, sbb = ring + s * WS_STAGE;
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
          const uint32_t ko = (uint32_t)kk * 2048;
          const uint32_t a_hi = sa + ko, a_lo = a_hi + 4096, b_hi = sbb + ko, b_lo = b_hi + 16384, acc = (it | kk) ? 1u : 0u;
          umma_f16(tmem, umma_desc_mn(a_hi), umma_desc_mn(b_hi), DW_IDESC, acc);
          umma_f16(tmem, umma_desc_mn(a_hi), umma_desc_mn(b_lo), DW_IDESC, 1u);
          umma_f16(tmem, umma_desc_mn(a_lo), umma_desc_mn(b_hi), DW_IDESC, 1u);
        }
        umma_commit(bar(DW0_NST + s));
      }
      umma_commit(bar(2 * DW0_NST));
    }
  } else if (warp < WS_NEW) {
    const int q = warp & 3, cg = warp >> 2;
    if (q * 32 < f.in) {                              // lane quarters beyond the input width hold nothing
      const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
      const uint32_t patch = ring + (uint32_t)warp * WS_PATCH1;       // the operand ring is dead once the last MMA has retired
      float* G = f.G + agent * f.sGa + net * f.sGn;
      mbar_wait(bar(2 * DW0_NST), 0);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        const int col = cg * 64 + c * 32;
        uint32_t v[32];
        tmem_ld32(tmem + lane_addr + (uint32_t)col, v);
        ws_store_rows(patch, v, G, q * 32, f.in, col, lane);
        __syncwarp();
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == WS_NEW + 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(256) : "memory");
  }
}
static inline bool dw0_planes_eligible(int in, int rows, int ldx, const float* X, long long sXa, long long sXn) {
  return in >= 1 && in <= 64 && ((rows + 31) >> 5) <= DW0_MAXST && (ldx % 4) == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0 &&
         (sXa % 4) == 0 && (sXn % 4) == 0;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static inline cudaError_t mlp_ws_init() {
  static bool done_dev[64] = {};
  int dev_ = 0; cudaGetDevice(&dev_);
  bool& done = done_dev[dev_ & 63];
  if (done) return cudaSuccess;
  cudaError_t e;
#define WS_ATTR(K) e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, WS_BYTES); if (e) return e;
  WS_ATTR(k_mlp_fwd_ws)
  WS_ATTR((k_mlp_bwd_ws<0, 0, 0>)) WS_ATTR((k_mlp_bwd_ws<0, 1, 0>)) WS_ATTR((k_mlp_bwd_ws<0, 2, 0>))
  WS_ATTR((k_mlp_bwd_ws<1, 0, 0>)) WS_ATTR((k_mlp_bwd_ws<2, 0, 0>)) WS_ATTR((k_mlp_bwd_ws<3, 0, 0>))
  WS_ATTR((k_mlp_bwd_ws<0, 0, 1>)) WS_ATTR((k_mlp_bwd_ws<1, 0, 1>)) WS_ATTR((k_mlp_bwd_ws<0, 1, 2>))
#undef WS_ATTR
  e = cudaFuncSetAttribute(k_dw_planes, cudaFuncAttributeMaxDynamicSharedMemorySize, DW_BYTES); if (e) return e;
  e = cudaFuncSetAttribute(k_dw0_planes, cudaFuncAttributeMaxDynamicSharedMemorySize, DW0_BYTES); if (e) return e;
  done = true;
  return cudaSuccess;
}
static inline bool mlp_fwd_ws_eligible(int h1, int h2, int nout, int K0, const float* theta, long long sTa, long long sTn) {
  return h1 == FW_H && h2 == FW_H && nout >= 1 && nout <= WS_MAXOUT && K0 >= 1 &&
         ((reinterpret_cast<uintptr_t>(theta) & 15) == 0) && ((sTa & 3) == 0) && ((sTn & 3) == 0);
}
static inline cudaError_t mlp_fwd_ws_launch(const FwdW& f, int nagents, cudaStream_t st) {
  dim3 grid((f.rows + TC_BM - 1) / TC_BM, nagents * f.nnet);
  k_mlp_fwd_ws<<<grid, WS_NT, WS_BYTES, st>>>(f);
  return cudaPeekAtLastError();
}
// the backward variants that exist: single-output nets (critics) with 0 / 1 / 2 action groups, multi-output nets
// (actor, kout = nout) without an input gradient
static inline bool mlp_bwd_ws_eligible(int h1, int h2, int kout, int nout, bool want_dxa, int a_cols, const float* theta, long long sTa,
                                       long long sTn) {
  if (!(h1 == FW_H && h2 == FW_H && kout >= 1 && kout <= WS_MAXOUT && kout <= nout)) return false;
  if (want_dxa && (kout != 1 || a_cols < 1 || a_cols > 32)) return false;
  return ((reinterpret_cast<uintptr_t>(theta) & 15) == 0) && ((sTa & 3) == 0) && ((sTn & 3) == 0);
}
static inline cudaError_t mlp_bwd_ws_launch(const BwdW& f, int nagents, cudaStream_t st) {
  dim3 grid((f.rows + TC_BM - 1) / TC_BM, nagents * f.nnet);
  const int ng = f.kout == 1 ? 0 : (f.kout + 15) / 16, na = f.dXa ? (f.a_cols + 15) / 16 : 0;
  // the shapes of the SAC / SAC-EO step get compile-time specialised forms (MODE 1 / 2)
  const bool m1 = f.H1p && f.dH2p && f.dH1p && !f.dH2 && !f.dH1, m2 = f.H1p && !f.dH2p && !f.dH1p && !f.dH2 && !f.dH1;
  if (ng == 0 && na == 0 && m1) k_mlp_bwd_ws<0, 0, 1><<<grid, WS_NT, WS_BYTES, st>>>(f);
  else if (ng == 1 && na == 0 && m1) k_mlp_bwd_ws<1, 0, 1><<<grid, WS_NT, WS_BYTES, st>>>(f);
  else if (ng == 0 && na == 1 && m2) k_mlp_bwd_ws<0, 1, 2><<<grid, WS_NT, WS_BYTES, st>>>(f);
  else if (ng == 0 && na == 0) k_mlp_bwd_ws<0, 0, 0><<<grid, WS_NT, WS_BYTES, st>>>(f);
  else if (ng == 0 && na == 1) k_mlp_bwd_ws<0, 1, 0><<<grid, WS_NT, WS_BYTES, st>>>(f);
  else if (ng == 0) k_mlp_bwd_ws<0, 2, 0><<<grid, WS_NT, WS_BYTES, st>>>(f);
  else if (ng == 1) k_mlp_bwd_ws<1, 0, 0><<<grid, WS_NT, WS_BYTES, st>>>(f);
  else if (ng == 2) k_mlp_bwd_ws<2, 0, 0><<<grid, WS_NT, WS_BYTES, st>>>(f);
  else k_mlp_bwd_ws<3, 0, 0><<<grid, WS_NT, WS_BYTES, st>>>(f);
  return cudaPeekAtLastError();
}

}  // namespace saceo
