// Fused expert-observation term through one frozen dynamics model for one agent:
//   forward   h1 = act0(Xm W0 + b0); h2 = act1(h1 W1 + b1); out = h2 W2 + b2                (base_world_model.py:65-87)
//   loss      pred = sE + clip(out[:, :S]) * max(std_d, 1e-8) + mean_d;  MSE partial          (SAC_expert.py:325-334)
//   backward  d(eps*MSE)/d(delta) -> dh2 -> dh1 -> gradient w.r.t. the ACTION columns of Xm   (weights frozen)
// The E/2 (<= 32) expert rows live in shared memory for the whole chain; every weight matrix is streamed
// exactly once per direction with coalesced reads (forward: lanes walk the output index; backward: one warp per
// output with lanes walking the contiguous input index + shuffle reduction), so the kernel is bound by the
// 2 x (W0 + W1 + W2) HBM read - the compulsory traffic of this term - instead of seven latency-bound launches.
#pragma once
#include "elem.cuh"
#include "model_term_mma.cuh"

namespace saceo {

constexpr int MT_THREADS = 512;

template <int MS>
__global__ void __launch_bounds__(MT_THREADS, 2) k_model_term(KCtx c, float* __restrict__ mse_part) {
  extern __shared__ float msm[];
  const int net = blockIdx.x, agent = blockIdx.y;
  const int S = c.S, A = c.A, SA = S + A, H1 = c.mh1, H2 = c.mh2, mo = c.mo, E = c.E;
  const int half = c.nmod == 2 ? E / 2 : E;             // rows handled by this model
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nwarp = MT_THREADS / 32;
  float* xs = msm;                      // [MS][SA]
  float* h1 = xs + MS * SA;             // [MS][H1]   (later dh1)
  float* h2 = h1 + MS * H1;             // [MS][H2]   (later dh2)
  float* ob = h2 + MS * H2;             // [MS][mo]   model output
  float* dd = ob + MS * mo;             // [MS][S]    d(eps*MSE)/d(delta)
  __shared__ float red[32];
  const float* th = c.T.model + ((long long)agent * 2 + net) * c.L.nm_stride;
  const float* W0 = th; const float* b0 = W0 + (long long)SA * H1;
  const float* W1 = b0 + H1; const float* b1 = W1 + (long long)H1 * H2;
  const float* W2 = b1 + H2; const float* b2 = W2 + (long long)H2 * mo;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  const float* Xm = c.Xm + ((long long)agent * 2 + net) * E * SA;

  for (int e = tid; e < MS * SA; e += MT_THREADS) { const int r = e / SA; xs[e] = r < half ? Xm[e] : 0.f; }
  __syncthreads();

  // ---- layer 0: thread j owns output column j -------------------------------------------------
  for (int j = tid; j < H1; j += MT_THREADS) {
    float acc[MS];
    const float bj = __ldg(b0 + j);
#pragma unroll
    for (int r = 0; r < MS; ++r) acc[r] = bj;
    for (int k = 0; k < SA; k += 8) {
      float w[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) w[u] = (k + u < SA) ? __ldg(W0 + (long long)(k + u) * H1 + j) : 0.f;   // 8 loads in flight
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (k + u < SA) {
#pragma unroll
          for (int r = 0; r < MS; ++r) acc[r] = fmaf(xs[r * SA + k + u], w[u], acc[r]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < MS; ++r) h1[r * H1 + j] = apply_act(c.mact0, acc[r]);
  }
  __syncthreads();
  // ---- layer 1 ---------------------------------------------------------------------------------
  for (int j = tid; j < H2; j += MT_THREADS) {
    float acc[MS];
    const float bj = __ldg(b1 + j);
#pragma unroll
    for (int r = 0; r < MS; ++r) acc[r] = bj;
    float wn[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) wn[u] = __ldg(W1 + (long long)u * H2 + j);
    for (int k = 0; k < H1; k += 8) {
      float w[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) w[u] = wn[u];
      if (k + 8 < H1) {
#pragma unroll
        for (int u = 0; u < 8; ++u) wn[u] = __ldg(W1 + (long long)(k + 8 + u) * H2 + j);   // next group flies during the FMAs
      }
#pragma unroll
      for (int r = 0; r < MS; ++r) {
        const float4 a = *reinterpret_cast<const float4*>(h1 + r * H1 + k);            // broadcast
        const float4 b = *reinterpret_cast<const float4*>(h1 + r * H1 + k + 4);
        acc[r] = fmaf(a.x, w[0], acc[r]); acc[r] = fmaf(a.y, w[1], acc[r]);
        acc[r] = fmaf(a.z, w[2], acc[r]); acc[r] = fmaf(a.w, w[3], acc[r]);
        acc[r] = fmaf(b.x, w[4], acc[r]); acc[r] = fmaf(b.y, w[5], acc[r]);
        acc[r] = fmaf(b.z, w[6], acc[r]); acc[r] = fmaf(b.w, w[7], acc[r]);
      }
    }
#pragma unroll
    for (int r = 0; r < MS; ++r) h2[r * H2 + j] = apply_act(c.mact1, acc[r]);
  }
  __syncthreads();
  // ---- layer 2: one warp per output column, lanes walk k ------------------------------------
  for (int col = warp; col < mo; col += nwarp) {
    float acc[MS];
#pragma unroll
    for (int r = 0; r < MS; ++r) acc[r] = 0.f;
    for (int k0 = lane; k0 < H2; k0 += 256) {
      float w[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) w[u] = (k0 + 32 * u < H2) ? __ldg(W2 + (long long)(k0 + 32 * u) * mo + col) : 0.f;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (k0 + 32 * u < H2) {
#pragma unroll
          for (int r = 0; r < MS; ++r) acc[r] = fmaf(h2[r * H2 + k0 + 32 * u], w[u], acc[r]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < MS; ++r) {
      float v = acc[r];
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) ob[r * mo + col] = v + __ldg(b2 + col);
    }
  }
  __syncthreads();
  // ---- loss and d(eps * MSE)/d(delta) -----------------------------------------------------------
  const float eps = agent_eps(c, agent);
  const float inv = 1.f / (float)half;
  float part = 0.f;
  for (int e = tid; e < MS * S; e += MT_THREADS) {
    const int i = e / S, j = e - i * S;
    float g = 0.f;
    if (i < half) {
      const int src = c.perm[(long long)agent * E + net * half + i];
      float delta = ob[i * mo + j];
      float cm = 1.f;
      if (c.delta_clip > 0.f) {
        cm = (delta >= -c.delta_clip && delta <= c.delta_clip) ? 1.f : 0.f;
        delta = fminf(fmaxf(delta, -c.delta_clip), c.delta_clip);
      }
      const float sd = nstd(nr[c.L.off_m_d_std + j]);
      const float pred = c.expert_s[((long long)agent * E + src) * S + j] + (delta * sd + nr[c.L.off_m_d_mean + j]);
      const float err = c.expert_sp[((long long)agent * E + src) * S + j] - pred;
      part += 0.5f * err * err;
      g = (-err * inv * eps) * sd * cm;
    }
    dd[e] = g;
  }
  part = block_sum(part, red);
  if (tid == 0) mse_part[agent * 2 + net] = part * inv;
  __syncthreads();
  // ---- layer 2 transposed: thread j reads its own (contiguous) row of W2 ----------------------
  for (int j = tid; j < H2; j += MT_THREADS) {
    float acc[MS];
#pragma unroll
    for (int r = 0; r < MS; ++r) acc[r] = 0.f;
    for (int cc = 0; cc < S; cc += 8) {
      float w[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) w[u] = (cc + u < S) ? __ldg(W2 + (long long)j * mo + cc + u) : 0.f;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (cc + u < S) {
#pragma unroll
          for (int r = 0; r < MS; ++r) acc[r] = fmaf(dd[r * S + cc + u], w[u], acc[r]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < MS; ++r) h2[r * H2 + j] = acc[r] * dact_from_out(c.mact1, h2[r * H2 + j]);   // own column only
  }
  __syncthreads();
  // ---- layer 1 transposed: thread i owns input index i and streams ITS contiguous W1 row (32-byte pieces = whole
  // sectors), the dz2 rows are broadcast from shared memory - the same loop shape as the forward layer.  (The earlier
  // warp-per-row mapping re-read all of dz2 from shared memory with distinct addresses for every pair of rows and took
  // 2.3x the forward time: 133 us vs 58 us per CTA, measured with clock64 stamps.)
  for (int i = tid; i < H1; i += MT_THREADS) {
    float acc[MS];
#pragma unroll
    for (int r = 0; r < MS; ++r) acc[r] = 0.f;
    const float4* __restrict__ wrow = reinterpret_cast<const float4*>(W1 + (long long)i * H2);
    float4 wn0 = __ldg(wrow), wn1 = __ldg(wrow + 1);
    for (int j = 0; j < H2; j += 8) {
      const float4 w0 = wn0, w1 = wn1;
      if (j + 8 < H2) { wn0 = __ldg(wrow + ((j + 8) >> 2)); wn1 = __ldg(wrow + ((j + 8) >> 2) + 1); }   // next piece flies during the FMAs
#pragma unroll
      for (int r = 0; r < MS; ++r) {
        const float4 a = *reinterpret_cast<const float4*>(h2 + r * H2 + j);            // broadcast
        const float4 g = *reinterpret_cast<const float4*>(h2 + r * H2 + j + 4);
        acc[r] = fmaf(a.x, w0.x, acc[r]); acc[r] = fmaf(a.y, w0.y, acc[r]);
        acc[r] = fmaf(a.z, w0.z, acc[r]); acc[r] = fmaf(a.w, w0.w, acc[r]);
        acc[r] = fmaf(g.x, w1.x, acc[r]); acc[r] = fmaf(g.y, w1.y, acc[r]);
        acc[r] = fmaf(g.z, w1.z, acc[r]); acc[r] = fmaf(g.w, w1.w, acc[r]);
      }
    }
#pragma unroll
    for (int r = 0; r < MS; ++r) h1[r * H1 + i] = acc[r] * dact_from_out(c.mact0, h1[r * H1 + i]);   // own column only
  }
  __syncthreads();
  // ---- layer 0 transposed, action rows only: one warp per action ------------------------------
  float* out = c.mdXa + ((long long)agent * 2 + net) * E * A;
  for (int a = warp; a < A; a += nwarp) {
    float acc[MS];
#pragma unroll
    for (int r = 0; r < MS; ++r) acc[r] = 0.f;
    const float* wrow = W0 + (long long)(S + a) * H1;
    for (int j0 = lane; j0 < H1; j0 += 256) {
      float w[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) w[u] = (j0 + 32 * u < H1) ? __ldg(wrow + j0 + 32 * u) : 0.f;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (j0 + 32 * u < H1) {
#pragma unroll
          for (int r = 0; r < MS; ++r) acc[r] = fmaf(h1[r * H1 + j0 + 32 * u], w[u], acc[r]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < MS; ++r) {
      float v = acc[r];
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0 && r < half) out[r * A + a] = v;
    }
  }
}

static inline int model_term_ms(const KCtx& c) {
  const int half = c.nmod == 2 ? c.E / 2 : c.E;
  return half <= 4 ? 4 : half <= 8 ? 8 : half <= 12 ? 12 : half <= 16 ? 16 : 32;
}
static inline size_t model_term_smem(const KCtx& c, int ms);
static inline bool model_term_eligible(const KCtx& c) {
  const int half = c.nmod == 2 ? c.E / 2 : c.E;
  return c.nmod > 0 && c.mnh == 2 && half <= 32 && (c.mh1 % 8) == 0 && (c.mh2 % 8) == 0 && ((c.L.nm_stride % 4) == 0) &&
         (((long long)(c.S + c.A) * c.mh1) % 4) == 0 &&
         model_term_smem(c, model_term_ms(c)) <= 200 * 1024;
}
static inline cudaError_t model_term_init() {
  static bool done_dev[64] = {};
  int dev_ = 0; cudaGetDevice(&dev_);
  bool& done = done_dev[dev_ & 63];       // cudaFuncSetAttribute is per device
  if (done) return cudaSuccess;
  cudaError_t e;
#define MT_ATTR(MSV) e = cudaFuncSetAttribute(k_model_term<MSV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); if (e) return e;
  MT_ATTR(4) MT_ATTR(8) MT_ATTR(12) MT_ATTR(16) MT_ATTR(32)
#undef MT_ATTR
#define MT_ATTR(MSV) e = cudaFuncSetAttribute(k_model_term_mma<MSV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024); if (e) return e;
  MT_ATTR(4) MT_ATTR(8) MT_ATTR(12) MT_ATTR(16)
#undef MT_ATTR
  done = true;
  return cudaSuccess;
}
static inline size_t model_term_smem(const KCtx& c, int ms) {
  return (size_t)ms * (c.S + c.A + c.mh1 + c.mh2 + c.mo + c.S) * sizeof(float);
}
static inline bool model_term_mma_ok(const KCtx& c) {
  const int half = c.nmod == 2 ? c.E / 2 : c.E;
  return half <= 16 && (c.mh1 % 32) == 0 && (c.mh2 % 32) == 0 && ((c.L.nm_stride % 4) == 0) &&
         (((long long)(c.S + c.A) * c.mh1 + c.mh1) % 4) == 0 && c.mo <= 32 && model_term_mma_smem(c, 16) <= 224 * 1024;
}
static bool g_mt_fp32 = false;      // test-only: k_model_term even where k_model_term_mma applies (saceo_test_set_mt_fp32)
// For shapes model_term_eligible accepts: the hidden layer on the tensor cores (k_model_term_mma) where the shape allows,
// else the fp32 CUDA-core kernel.
static inline cudaError_t model_term_launch(const KCtx& c, float* mse_part, cudaStream_t st) {
  const int half = c.nmod == 2 ? c.E / 2 : c.E;
  dim3 grid(c.nmod, c.n_agents);
  if (!g_mt_fp32 && model_term_mma_ok(c)) {
    const int nthr = MTM_THREADS;
#define MT_GOM(MSV) do { k_model_term_mma<MSV><<<grid, nthr, model_term_mma_smem(c, MSV), st>>>(c, mse_part, g_mt_dbg); } while (0)
    if (half <= 4) MT_GOM(4);
    else if (half <= 8) MT_GOM(8);
    else if (half <= 12) MT_GOM(12);
    else MT_GOM(16);
#undef MT_GOM
    return cudaPeekAtLastError();
  }
#define MT_GO(MSV) do { k_model_term<MSV><<<grid, MT_THREADS, model_term_smem(c, MSV), st>>>(c, mse_part); } while (0)
  if (half <= 4) MT_GO(4);
  else if (half <= 8) MT_GO(8);
  else if (half <= 12) MT_GO(12);
  else if (half <= 16) MT_GO(16);
  else MT_GO(32);
#undef MT_GO
  return cudaPeekAtLastError();
}

}  // namespace saceo
