// tcgen05 (5th-generation tensor core) batched GEMM engine for the hidden x hidden per-agent
// contractions of the SAC-EO update (gemm_mode SACEO_GEMM_TCGEN05_BF16X3).
//
// fp32 parity on tensor cores: every fp32 operand x is split into bf16 hi = rn(x) and
// lo = rn(x - hi); the product is accumulated as hi.hi + hi.lo + lo.hi with fp32 accumulation in
// TMEM (three tcgen05.mma kind::f16 per K slab).  The dropped lo.lo term and the second-order
// residuals are O(2^-16) relative, far inside the 1e-3 parity budget that single-pass TF32 (2^-11
// per operand, truncated by the MMA) would consume after six chained GEMMs.
//
// Layout: one CTA owns a 128 x BN tile of C for one (agent, net).  All threads load a 64-wide K
// slab of both fp32 operands from global/L2, split it, and write the bf16 planes into shared memory
// in the canonical K-major SWIZZLE_128B UMMA layout (8-row x 128-byte atoms, 16-byte chunk index
// XOR row-in-atom) - whatever the storage order of the operand, so a single shared-memory
// descriptor format serves forward (X.W), input-gradient (dY.W^T) and weight-gradient (X^T.dY)
// GEMMs.  One thread issues the MMAs; tcgen05.commit on an mbarrier releases the stage to the
// loaders; the epilogue reads the accumulator with tcgen05.ld (32 lanes x 32 columns per warp) and
// applies the same fused epilogue as the SIMT engine (bias, addend, activation / activation
// derivative).  Rows that do not fill a 128-row tile (the E expert rows, the ones-row of the
// [dW; db] trick) are finished by the SIMT engine (GemmP::m_off).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>
#include "gemm_simt.cuh"

namespace saceo {

constexpr int TC_BM = 128, TC_BK = 64;

struct TcP {
  GemmP g;
  int m_rows;          // valid rows of op(A) handled by the tensor-core launch
  long long a_sr, a_sk, b_sr, b_sk;   // element strides of op(A)(m,k) and op(B)(k,n): (row=m|n, k)
  unsigned long long* dbg;            // optional per-CTA phase timestamps (globaltimer ns), 8 per CTA
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// explicit shared-window accesses (32-bit addresses): the swizzled / overlaid buffers are carved out of one
// dynamic allocation, so generic pointers would compile to generic LD/ST with 64-bit address math
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ float lds32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts128(uint32_t a, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts128f(uint32_t a, float x, float y, float z, float w) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  uint32_t spins = 0;
  do {
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    // a lost arrival must fail loudly instead of hanging the GPU (each try_wait already sleeps in hardware)
    if (!ok && ++spins > (1u << 24)) __trap();
  } while (!ok);
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
// start>>4 [0,14) | LBO>>4 [16,30) (=1, ignored for swizzled K-major) | SBO>>4 [32,46) (8 rows * 128 B)
// | version=1 [46,48) | layout_type=2 (SWIZZLE_128B) [61,64)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// instruction descriptor: D=F32 [4,6)=1, A=BF16 [7,10)=1, B=BF16 [10,13)=1, A/B K-major, N>>3 [17,23), M>>4 [24,29)
// fmt: 1 = bf16 operands (default), 0 = fp16 operands (forward passes, see split8)
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N, uint32_t fmt = 1u) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// fp32 -> (hi, lo) 16-bit pair for 8 consecutive-k values, packed conversions; hi = rn(x), lo = rn(x - hi).
//   F16 = false: bf16 planes (8 + 8 mantissa bits, residual 2^-17, full fp32 exponent range) - used wherever the
//                operand can be tiny (gradients).
//   F16 = true:  fp16 planes (11 + 11 bits, residual 2^-23 for |x| >= 2^-3, absolute 2^-25 below; saturating at
//                65504) - used by the FORWARD kernels, whose operands (normalised inputs, activations, weights) are
//                O(1): the pre-activations then carry fp32-level error, so ReLU masks / min(Q1,Q2) selections flip
//                no more often than between two fp32 implementations.  With bf16 planes (1e-5 forward error) a
//                handful of masks per layer flip and single gradient tensors can miss the 1e-3 parity bar.
template <bool F16 = false>
__device__ __forceinline__ void split8(const float (&x)[8], uint4& hi, uint4& lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (F16) {
      uint32_t hb, lb;
      asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hb) : "f"(x[2 * i + 1]), "f"(x[2 * i]));
      const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hb));
      asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lb) : "f"(x[2 * i + 1] - hf.y), "f"(x[2 * i] - hf.x));
      h[i] = hb; l[i] = lb;
    } else {
      const __nv_bfloat162 hp = __floats2bfloat162_rn(x[2 * i], x[2 * i + 1]);      // low half = x[2i]
      h[i] = *reinterpret_cast<const uint32_t*>(&hp);
      const float f0 = __uint_as_float(h[i] << 16), f1 = __uint_as_float(h[i] & 0xFFFF0000u);
      const __nv_bfloat162 lp = __floats2bfloat162_rn(x[2 * i] - f0, x[2 * i + 1] - f1);
      l[i] = *reinterpret_cast<const uint32_t*>(&lp);
    }
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// Register-staged slab loader.  A ROWS x 64 slab of a fp32 operand (element (r,k) at src[r*sr + k*sk],
// zero outside [0,rlim) x [0,klim)) is cut into ROWS*8 items of 8 consecutive k; thread t owns items
// t, t+NT, ...  The item -> (row, k-chunk) map, the global base pointer and the swizzled smem
// offset of every item are fixed for the whole K loop and computed once (init); ld() only ISSUES the
// global loads of one slab (so the next slab is in flight while the tensor core works on the current
// one); st() splits fp32 -> bf16 hi/lo and stores both planes in the K-major SWIZZLE_128B layout
// (conflict-free 16-byte stores for either storage order).
template <int ROWS, int NT>
struct Slab {
  static constexpr int ITEMS = ROWS * 8;
  static constexpr int PER = (ITEMS + NT - 1) / NT;
  float x[PER][8];
  const float* ptr[PER];     // element (row, kc*8) of slab 0
  int soff[PER];             // byte offset of the item's 16-byte chunk inside a plane; -1: item out of range
  int kc8[PER];              // kc*8
  long long sk;
  bool kcontig, vec;

  __device__ __forceinline__ void init(const float* __restrict__ src, long long sr, long long sk_, int r0, int rlim) {
    sk = sk_;
    kcontig = (sk_ == 1);
    vec = kcontig && ((sr & 3) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int it = threadIdx.x + i * NT;
      int r, kc;
      if (kcontig) { kc = it & 7; r = it >> 3; }          // 8 lanes cover one row's 256 contiguous bytes
      else { r = it % ROWS; kc = it / ROWS; }               // lanes walk rows: each scalar load is coalesced
      const int gr = r0 + r;
      const bool ok = (it < ITEMS);
      kc8[i] = kc * 8;
      ptr[i] = (ok && gr < rlim) ? src + (long long)gr * sr + (long long)(kc * 8) * sk_ : nullptr;
      soff[i] = ok ? (r >> 3) * 1024 + (r & 7) * 128 + ((kc ^ (r & 7)) << 4) : -1;
    }
  }
  __device__ __forceinline__ void ld(int k0, int klim) {
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const float* p = ptr[i];
      const int gk = k0 + kc8[i];
      if (p != nullptr && gk + 8 <= klim) {
        p += (long long)k0 * sk;
        if (vec) {
          const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
          x[i][0] = a.x; x[i][1] = a.y; x[i][2] = a.z; x[i][3] = a.w;
          x[i][4] = b.x; x[i][5] = b.y; x[i][6] = b.z; x[i][7] = b.w;
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) x[i][j] = __ldg(p + j * sk);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          x[i][j] = (p != nullptr && gk + j < klim) ? __ldg(p + ((long long)k0 + j) * sk) : 0.f;
      }
    }
  }
  template <bool F16 = false>
  __device__ __forceinline__ void st(uint32_t hi, uint32_t lo) const {
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      if (soff[i] < 0) continue;
      uint4 h, l;
      split8<F16>(x[i], h, l);
      sts128(hi + soff[i], h);
      sts128(lo + soff[i], l);
    }
  }
};

template <int BN, int NSTAGE, int NT>
struct TcSmem {
  static constexpr int A_PLANE = TC_BM * 128;       // bytes of one bf16 plane of the A slab
  static constexpr int B_PLANE = BN * 128;
  static constexpr int STAGE = 2 * A_PLANE + 2 * B_PLANE;
  static constexpr int NGRP = (BN / 32) < (NT / 128) ? (BN / 32) : (NT / 128);
  static constexpr int PATCH = NGRP * 4 * 32 * (BN / NGRP + 4) * 4;     // epilogue staging (overlays the stages)
  static constexpr int MAIN = NSTAGE * STAGE > PATCH ? NSTAGE * STAGE : PATCH;
  static constexpr int BYTES = MAIN + 1024 /*align slack*/ + 64 /*barriers + tmem ptr*/;
};

// ---- epilogue (shared by both kernels) -------------------------------------------------------------
// warp w owns TMEM lanes 32*(w%4).. (hardware rule) and column group w/4.  Phase 1: tcgen05.ld gives each
// thread 32 consecutive columns of ITS row; they are parked in a warp-private padded smem patch (the
// operand buffers are free once the last MMA has retired).  Phase 2: the warp walks the patch row-wise so
// that bias/addend/aux reads and the C stores are coalesced 16-byte accesses.
template <int BN, int NT>
__device__ __forceinline__ void tc_epilogue(const TcP& q, uint32_t sb, uint32_t tmem, int agent, int net,
                                            long long offC, int m0, int n0, int warp, int lane) {
  const GemmP& p = q.g;
  constexpr int NGRP = (BN / 32) < (NT / 128) ? (BN / 32) : (NT / 128);   // column groups
  constexpr int GCOLS = BN / NGRP;                 // columns per warp (32 or 64)
  constexpr int PSTR = GCOLS + 4;                  // padded patch row stride (floats), keeps 16-byte alignment
  const int grp = warp >> 2;
  if (grp >= NGRP) return;
  const float* bias = p.bias ? p.bias + agent * p.sba + net * p.sbn : nullptr;
  const float* addend = p.addend ? p.addend + offC : nullptr;
  const float* aux = p.aux ? p.aux + offC : nullptr;
  float* __restrict__ C = p.C + offC;
  const uint32_t patch = sb + (uint32_t)warp * 32 * PSTR * 4;
  const int cbase = grp * GCOLS;
#pragma unroll 1
  for (int c0 = 0; c0 < GCOLS; c0 += 32) {
    uint32_t v[32];
    const uint32_t taddr = tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(cbase + c0);
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                 "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    const uint32_t dst = patch + (uint32_t)(lane * PSTR + c0) * 4;
#pragma unroll
    for (int j = 0; j < 8; ++j) sts128(dst + j * 16, make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
  }
  __syncwarp();
  constexpr int LPR = GCOLS / 4;                 // lanes per row (float4 each)
  constexpr int RPI = 32 / LPR;                  // rows per warp instruction
  const int lr = lane / LPR, lc = (lane % LPR) * 4;
  const bool vec_ok = ((p.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0) &&
                      (!addend || (reinterpret_cast<uintptr_t>(addend) & 15) == 0) &&
                      (!aux || (reinterpret_cast<uintptr_t>(aux) & 15) == 0);
  const int gn = n0 + cbase + lc;
#pragma unroll 4
  for (int rr = 0; rr < 32; rr += RPI) {
    const int r = rr + lr;
    const int grow = m0 + (warp & 3) * 32 + r;
    if (grow >= q.m_rows || gn >= p.N) continue;
    const float4 acc = lds128(patch + (uint32_t)(r * PSTR + lc) * 4);
    float x[4] = {acc.x, acc.y, acc.z, acc.w};
    const long long o = (long long)grow * p.ldc + gn;
    const bool full = vec_ok && (gn + 4 <= p.N);
    float ad[4] = {0.f, 0.f, 0.f, 0.f}, ax[4] = {0.f, 0.f, 0.f, 0.f};
    if (full) {
      if (addend) { const float4 t4 = *reinterpret_cast<const float4*>(addend + o); ad[0] = t4.x; ad[1] = t4.y; ad[2] = t4.z; ad[3] = t4.w; }
      if (aux) { const float4 t4 = *reinterpret_cast<const float4*>(aux + o); ax[0] = t4.x; ax[1] = t4.y; ax[2] = t4.z; ax[3] = t4.w; }
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) if (gn + j < p.N) { if (addend) ad[j] = addend[o + j]; if (aux) ax[j] = aux[o + j]; }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (bias && gn + j < p.N) x[j] += __ldg(bias + gn + j);
      x[j] += ad[j];
      if (p.epi == EPI_ACT) x[j] = apply_act(p.act, x[j]);
      else if (p.epi == EPI_MUL_DACT) x[j] *= dact_from_out(p.act, ax[j]);
    }
    if (full) *reinterpret_cast<float4*>(C + o) = make_float4(x[0], x[1], x[2], x[3]);
    else {
#pragma unroll
      for (int j = 0; j < 4; ++j) if (gn + j < p.N) C[o + j] = x[j];
    }
  }
}

template <int BN, int NSTAGE, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) k_gemm_tc(TcP q) {
  using SM = TcSmem<BN, NSTAGE, NT>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;       // 1024-aligned base in the shared window
  const uint32_t bars = sb + SM::MAIN;                              // [NSTAGE] free + [1] done (8 bytes each)
  const uint32_t tmem_slot = bars + 8 * (NSTAGE + 1);

  const GemmP& p = q.g;
  const int z = blockIdx.z;
  const int agent = z / p.nnet, net = z - agent * p.nnet;
  const float* __restrict__ A = p.A + agent * p.sAa + net * p.sAn;
  const float* __restrict__ B = p.B + agent * p.sBa + net * p.sBn;
  const long long offC = agent * p.sCa + net * p.sCn;
  const int m0 = blockIdx.y * TC_BM, n0 = blockIdx.x * BN;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s <= NSTAGE; ++s) mbar_init(bars + 8 * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(BN) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = lds_u32(tmem_slot);

  const int nk = (p.K + TC_BK - 1) / TC_BK;
  const uint32_t IDESC = umma_idesc(TC_BM, BN, p.f16 ? 0u : 1u);
  Slab<TC_BM, NT> ra;
  Slab<BN, NT> rb;
  ra.init(A, q.a_sr, q.a_sk, m0, q.m_rows);
  rb.init(B, q.b_sr, q.b_sk, n0, p.N);
  ra.ld(0, p.K);
  rb.ld(0, p.K);
  for (int kc = 0; kc < nk; ++kc) {
    const int s = kc % NSTAGE;
    const uint32_t st = sb + s * SM::STAGE;
    if (kc >= NSTAGE) mbar_wait(bars + 8 * s, (uint32_t)((kc / NSTAGE - 1) & 1));   // MMAs of slab kc-NSTAGE retired
    if (p.f16) { ra.template st<true>(st, st + SM::A_PLANE); rb.template st<true>(st + 2 * SM::A_PLANE, st + 2 * SM::A_PLANE + SM::B_PLANE); }
    else       { ra.template st<false>(st, st + SM::A_PLANE); rb.template st<false>(st + 2 * SM::A_PLANE, st + 2 * SM::A_PLANE + SM::B_PLANE); }
    if (kc + 1 < nk) {          // next slab's global loads fly during the barrier, the MMA issue and the next wait
      ra.ld((kc + 1) * TC_BK, p.K);
      rb.ld((kc + 1) * TC_BK, p.K);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the tensor core
    __syncthreads();
    if (threadIdx.x == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t a_hi = st, a_lo = a_hi + SM::A_PLANE;
      const uint32_t b_hi = a_hi + 2 * SM::A_PLANE, b_lo = b_hi + SM::B_PLANE;
#pragma unroll
      for (int kk = 0; kk < TC_BK / 16; ++kk) {
        const uint32_t ko = kk * 32;               // 16 bf16 = 32 bytes along K inside the 128-byte swizzled row
        umma_f16(tmem, umma_desc(a_hi + ko), umma_desc(b_hi + ko), IDESC, (kc | kk) ? 1u : 0u);
        umma_f16(tmem, umma_desc(a_hi + ko), umma_desc(b_lo + ko), IDESC, 1u);
        umma_f16(tmem, umma_desc(a_lo + ko), umma_desc(b_hi + ko), IDESC, 1u);
      }
      umma_commit(bars + 8 * s);
      if (kc == nk - 1) umma_commit(bars + 8 * NSTAGE);
    }
  }
  mbar_wait(bars + 8 * NSTAGE, 0);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

  tc_epilogue<BN, NT>(q, sb, tmem, agent, net, offC, m0, n0, warp, lane);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(BN) : "memory");
  }
}

// ------------------------------------------------------------------------------------------
// Streaming variant for the hot shapes (full 128 x 256 tiles, K % 32 == 0, 16-byte aligned operands).
// The register-staged kernel above exposes one global-memory latency per K slab because all warps load,
// wait and convert in lock-step.  Here the raw fp32 slabs travel global -> shared with cp.async
// (LDGSTS, no registers), two 32-wide K slabs ahead of their use; the warps only do the
// fp32 -> bf16 hi/lo split shared -> shared into the half of the 64-wide SWIZZLE_128B stage that the
// tensor core is not reading, so copy, split and MMA of three consecutive slabs overlap.
//   smem: raw ring 2 x 48 KB | bf16 stage 96 KB (two 32-k halves) | barriers;  epilogue patch overlays all.
// ------------------------------------------------------------------------------------------
constexpr int TS_BN = 256, TS_BK = 32, TS_NT = 512;
constexpr int TS_RAW_A = TC_BM * TS_BK * 4, TS_RAW_B = TS_BN * TS_BK * 4, TS_RAW = TS_RAW_A + TS_RAW_B;   // 48 KB
constexpr int TS_APLANE = TC_BM * 128, TS_BPLANE = TS_BN * 128, TS_STAGE = 2 * TS_APLANE + 2 * TS_BPLANE; // 96 KB
constexpr int TS_MAIN = 2 * TS_RAW + TS_STAGE;
constexpr int TS_BYTES = TS_MAIN + 1024 + 64;

__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define TC_STAMP(i) do { if (q.dbg && threadIdx.x == 0) q.dbg[(size_t)((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 8 + (i)] = gtime(); } while (0)

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
// src_bytes = 0: nothing is read, the 16 destination bytes are zero-filled (rows past the end of a partial tile)
__device__ __forceinline__ void cp_async16z(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}

// Per-thread copy/convert plan of one operand with ROWS rows; KC: storage contiguous along k.
//   raw slab layout   KC: raw[r][32] (128 B per row)      else: raw[32][ROWS] (ROWS*4 B per k)
// Source pointers and shared offsets are computed once; each slab only advances the pointers.
template <int ROWS, bool KC>
struct TsPlan {
  static constexpr int NP = ROWS * 8 / TS_NT;     // 16-byte pieces per thread per slab
  static constexpr int NI = ROWS * 4 / TS_NT;     // (row, 8-k chunk) items per thread per slab
  const float* src[NP];
  uint32_t dst[NP];
  uint32_t rd[NI], wr[NI];
  uint32_t sz;               // bit i: piece i lies inside the operand (rows < rlim); other pieces are zero-filled
  long long kstep;

  // rlim: rows of the operand that exist (a partial last tile); the storage must be readable up to the 4-row group
  // that contains row rlim-1 (KC = false: leading dimension >= rlim rounded up to 4)
  __device__ __forceinline__ void init(const float* __restrict__ base, long long sr, long long sk, int r0, int rlim = 1 << 30) {
    kstep = KC ? TS_BK : (long long)TS_BK * sk;
    sz = 0;
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      const int pc = threadIdx.x + i * TS_NT;
      if (KC) {
        const int r = pc >> 3, c = pc & 7;
        const bool ok = r0 + r < rlim;
        src[i] = base + (long long)(ok ? r0 + r : r0) * sr + c * 4;
        dst[i] = (uint32_t)(r * 128 + c * 16);
        sz |= ok ? (1u << i) : 0u;
      } else {
        constexpr int PPR = ROWS / 4;
        const int k = pc / PPR, c = pc % PPR;
        const bool ok = r0 + c * 4 < rlim;
        src[i] = base + (long long)k * sk + r0 + (ok ? c * 4 : 0);
        dst[i] = (uint32_t)(k * (ROWS * 4) + c * 16);
        sz |= ok ? (1u << i) : 0u;
      }
    }
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int it = threadIdx.x + i * TS_NT;
      int r, kc4;
      if (KC) { kc4 = it & 3; r = it >> 2; rd[i] = (uint32_t)(r * 128 + kc4 * 32); }
      else { r = it % ROWS; kc4 = it / ROWS; rd[i] = (uint32_t)(((kc4 * 8) * ROWS + r) * 4); }
      wr[i] = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((kc4 ^ (r & 7)) << 4));   // k-half 0; half 1 = ^64
    }
  }
  __device__ __forceinline__ void issue(uint32_t raw) {
#pragma unroll
    for (int i = 0; i < NP; ++i) { cp_async16z(raw + dst[i], src[i], (sz >> i) & 1u ? 16u : 0u); src[i] += kstep; }
  }
  template <bool F16 = false>
  __device__ __forceinline__ void convert(uint32_t raw, int h, uint32_t hi, uint32_t lo) const {
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      float x[8];
      if (KC) {
        const float4 a = lds128(raw + rd[i]), b = lds128(raw + rd[i] + 16);
        x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = lds32(raw + rd[i] + j * (ROWS * 4));
      }
      uint4 hh, ll;
      split8<F16>(x, hh, ll);
      const uint32_t off = wr[i] ^ (uint32_t)(h << 6);
      sts128(hi + off, hh);
      sts128(lo + off, ll);
    }
  }
};

template <bool AKC, bool BKC>
__global__ void __launch_bounds__(TS_NT, 1) k_gemm_tc_stream(TcP q) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t stage = sb + 2 * TS_RAW;                          // bf16 planes (1024-aligned)
  const uint32_t bars = sb + TS_MAIN;                              // [2] half free + [1] done
  const uint32_t tmem_slot = bars + 24;

  TC_STAMP(0);
  const GemmP& p = q.g;
  const int z = blockIdx.z;
  const int agent = z / p.nnet, net = z - agent * p.nnet;
  const float* __restrict__ A = p.A + agent * p.sAa + net * p.sAn;
  const float* __restrict__ B = p.B + agent * p.sBa + net * p.sBn;
  const long long offC = agent * p.sCa + net * p.sCn;
  const int m0 = blockIdx.y * TC_BM, n0 = blockIdx.x * TS_BN;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < 3; ++s) mbar_init(bars + 8 * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(TS_BN) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  TsPlan<TC_BM, AKC> pa;
  TsPlan<TS_BN, BKC> pb;
  pa.init(A, q.a_sr, q.a_sk, m0, q.m_rows);        // a partial last row tile is zero-filled
  pb.init(B, q.b_sr, q.b_sk, n0);
  const int nslab = p.K / TS_BK;
  // prologue: two slabs in flight
  pa.issue(sb); pb.issue(sb + TS_RAW_A);
  asm volatile("cp.async.commit_group;" ::: "memory");
  if (nslab > 1) { pa.issue(sb + TS_RAW); pb.issue(sb + TS_RAW + TS_RAW_A); }
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = lds_u32(tmem_slot);
  TC_STAMP(1);
  const uint32_t IDESC = umma_idesc(TC_BM, TS_BN, p.f16 ? 0u : 1u);
  const uint32_t a_hi = stage, a_lo = stage + TS_APLANE, b_hi = stage + 2 * TS_APLANE, b_lo = b_hi + TS_BPLANE;

  for (int j = 0; j < nslab; ++j) {
    const int h = j & 1;
    const uint32_t raw = sb + h * TS_RAW;
    asm volatile("cp.async.wait_group 1;" ::: "memory");       // this thread's copies of slab j have landed
    __syncthreads();                                            // ... and everybody else's
    if (j >= 2) mbar_wait(bars + 8 * h, (uint32_t)((j / 2 - 1) & 1));     // MMAs that read half h (slab j-2) retired
    if (p.f16) { pa.template convert<true>(raw, h, a_hi, a_lo); pb.template convert<true>(raw + TS_RAW_A, h, b_hi, b_lo); }
    else       { pa.template convert<false>(raw, h, a_hi, a_lo); pb.template convert<false>(raw + TS_RAW_A, h, b_hi, b_lo); }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();                                            // stage half written, raw[h] free again
    if (j + 2 < nslab) { pa.issue(raw); pb.issue(raw + TS_RAW_A); }
    asm volatile("cp.async.commit_group;" ::: "memory");       // (possibly empty) keeps the group count uniform
    if (threadIdx.x == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
      for (int kk = 0; kk < 2; ++kk) {
        const uint32_t ko = (uint32_t)(h * 2 + kk) * 32;        // 16 bf16 = 32 bytes inside the 128-byte swizzled row
        umma_f16(tmem, umma_desc(a_hi + ko), umma_desc(b_hi + ko), IDESC, (j | kk) ? 1u : 0u);
        umma_f16(tmem, umma_desc(a_hi + ko), umma_desc(b_lo + ko), IDESC, 1u);
        umma_f16(tmem, umma_desc(a_lo + ko), umma_desc(b_hi + ko), IDESC, 1u);
      }
      umma_commit(bars + 8 * h);
      if (j == nslab - 1) umma_commit(bars + 16);
    }
  }
  TC_STAMP(2);
  mbar_wait(bars + 16, 0);
  TC_STAMP(3);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  tc_epilogue<TS_BN, TS_NT>(q, sb, tmem, agent, net, offC, m0, n0, warp, lane);
  TC_STAMP(4);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  TC_STAMP(5);
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TS_BN) : "memory");
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
// kernel variants: (BN, stages, threads, min CTAs/SM)
//   variant 0: 128 x 256 tile, 2 stages, 512 threads, 1 CTA/SM   (best operand reuse per CTA)
//   variant 1: 128 x 128 tile, 1 stage,  256 threads, 2 CTAs/SM  (two tiles per SM overlap each other's
//              load / MMA / epilogue phases; each SM keeps more bytes in flight)
#define TC_FOR_ALL(X) X(256, 2, 512, 1) X(128, 3, 512, 1) X(64, 4, 512, 1) X(128, 1, 256, 2) X(64, 1, 256, 2)
static inline cudaError_t tc_gemm_init() {
  static bool done_dev[64] = {};
  int dev_ = 0; cudaGetDevice(&dev_);
  bool& done = done_dev[dev_ & 63];       // cudaFuncSetAttribute is per device
  if (done) return cudaSuccess;
  cudaError_t e;
#define TC_ATTR(BN_, NS_, NT_, MB_) \
  e = cudaFuncSetAttribute(k_gemm_tc<BN_, NS_, NT_, MB_>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                           TcSmem<BN_, NS_, NT_>::BYTES); if (e) return e;
  TC_FOR_ALL(TC_ATTR)
#undef TC_ATTR
  e = cudaFuncSetAttribute(k_gemm_tc_stream<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TS_BYTES); if (e) return e;
  e = cudaFuncSetAttribute(k_gemm_tc_stream<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TS_BYTES); if (e) return e;
  e = cudaFuncSetAttribute(k_gemm_tc_stream<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TS_BYTES); if (e) return e;
  done = true;
  return cudaSuccess;
}

// rows of op(A) that go to the tensor-core launch.  The MMA itself is nearly free next to the operand traffic,
// so a partly empty 128-row tile (zero-filled rows) beats a CUDA-core tail as soon as the tail has >= 16 rows
// (the E expert rows, [dW0; db0] with S+A rows); only tiny tails (the single ones-row) stay off the tensor core.
static inline int tc_rows(bool ONES, const GemmP& p) {
  const int mmain = ONES ? p.M - 1 : p.M;
  int tiles = mmain / TC_BM;
  const int rem = mmain % TC_BM;
  if (rem >= 16 || (rem >= 4 && tiles >= 1)) tiles += 1;      // next to full tiles even a thin tail beats the CUDA-core pass
  const int r = tiles * TC_BM;
  return r < mmain ? r : mmain;
}
static inline bool tc_gemm_eligible(bool TA, bool TB, bool ONES, const GemmP& p) {
  (void)TA; (void)TB;
  const int r = tc_rows(ONES, p);
  // full tiles always; a lone partial tile only when the weight panel is big enough to amortise a 512-thread CTA
  return p.m_off == 0 && p.N > 32 && p.K >= 8 && (r >= 96 || (r >= 16 && (long long)p.N * p.K >= 128 * 128));
}

// Which tensor-core kernel takes a GEMM: the streaming kernel k_gemm_tc_stream<akc, bkc>, or the register-staged
// k_gemm_tc<bn, stages, threads, ...>.
struct TcRoute {
  bool stream;
  bool akc, bkc;               // streaming: op(A) / op(B) storage contiguous along k
  int bn, stages, threads;     // register-staged tile
};
static inline TcRoute tc_route(bool TA, bool TB, const GemmP& p, int variant) {
  TcRoute r{};
  r.akc = (TA ? p.lda : 1) == 1; r.bkc = (TB ? 1 : p.ldb) == 1;
  const bool aligned = ((p.lda & 3) == 0) && ((p.ldb & 3) == 0) && (((p.sAa | p.sAn | p.sBa | p.sBn) & 3) == 0) &&
                       ((reinterpret_cast<uintptr_t>(p.A) & 15) == 0) && ((reinterpret_cast<uintptr_t>(p.B) & 15) == 0);
  // both operands contiguous along k (dX = dY . W^T): the register-staged 64-k kernel reads whole 256-byte rows and wins
  // (134 vs 160 us on 256^3 x 512, tools/gemm_bench.py); every other orientation streams
  const bool both_kc = r.akc && r.bkc;
  r.stream = variant != 2 && aligned && !both_kc && (p.K % TS_BK) == 0 && (p.N % TS_BN) == 0;
  if (r.stream) return r;
  if (variant == 1) { r.bn = p.N > 64 ? 128 : 64; r.stages = 1; r.threads = 256; }
  else { r.bn = p.N > 128 ? 256 : p.N > 64 ? 128 : 64; r.stages = r.bn == 256 ? 2 : r.bn == 128 ? 3 : 4; r.threads = 512; }
  return r;
}

static unsigned long long* g_tc_dbg = nullptr;   // set by saceo_test_gemm_timed only
// launches the tensor-core part (rows [0, tc_rows)); the caller finishes rows [tc_rows, M). <0 on a launch error
static inline int tc_gemm_launch(bool TA, bool TB, bool ONES, const GemmP& p, int nagents, int variant, cudaStream_t st) {
  TcP q; q.g = p; q.dbg = g_tc_dbg;
  q.m_rows = tc_rows(ONES, p);
  q.a_sr = TA ? 1 : p.lda; q.a_sk = TA ? p.lda : 1;
  q.b_sr = TB ? p.ldb : 1; q.b_sk = TB ? 1 : p.ldb;
  const int mt = (q.m_rows + TC_BM - 1) / TC_BM;
#define TC_GO(BN_, NS_, NT_, MB_) do { dim3 grid((p.N + BN_ - 1) / BN_, mt, nagents * p.nnet); \
    k_gemm_tc<BN_, NS_, NT_, MB_><<<grid, NT_, TcSmem<BN_, NS_, NT_>::BYTES, st>>>(q); } while (0)
  const TcRoute r = tc_route(TA, TB, p, variant);
  if (r.stream) {
    dim3 grid(p.N / TS_BN, mt, nagents * p.nnet);
    if (r.akc) k_gemm_tc_stream<true, false><<<grid, TS_NT, TS_BYTES, st>>>(q);
    else if (r.bkc) k_gemm_tc_stream<false, true><<<grid, TS_NT, TS_BYTES, st>>>(q);
    else k_gemm_tc_stream<false, false><<<grid, TS_NT, TS_BYTES, st>>>(q);
  } else if (r.threads == 256) {
    if (r.bn == 128) TC_GO(128, 1, 256, 2); else TC_GO(64, 1, 256, 2);
  } else {
    if (r.bn == 256) TC_GO(256, 2, 512, 1); else if (r.bn == 128) TC_GO(128, 3, 512, 1); else TC_GO(64, 4, 512, 1);
  }
#undef TC_GO
  if (cudaPeekAtLastError() != cudaSuccess) return -1;
  return 0;
}

}  // namespace saceo
