// Element-wise / reduction kernels of the SAC-EO update: replay row gather, input staging
// (normalise + concat), tanh-Gaussian head forward/backward, TD target, loss reductions,
// Keras-Adam (+ Polyak) and the temperature step.  Every kernel covers the whole population
// (blockIdx.y or .z = agent).  Reference citations are relative to /root/reference/.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "../../include/saceo.h"
#include "gemm_simt.cuh"
#include "rng.cuh"
#include "planes.cuh"

namespace saceo {

struct KCtx {
  int n_agents, S, A, Ao, mo, B, E, R, nmod, per_state_std, sep_reward;
  float eps_force;   // >= 0: expert weight used instead of hyper[5] (behaviour cloning = 1), < 0: per-agent table value
  int ldXc, ldXp;    // leading dimensions of Xc (S+A -> multiple of 4) and Xpi (S -> multiple of 4): 16-byte aligned rows, pad columns stay zero
  int Rs;   // row stride of the per-agent [R rows] actor buffers (R rounded up to 32; the pad rows stay zero)
  int mh1, mh2, mact0, mact1;
  int mnh;           // hidden layers of the models; mh1 / mh2 / mact0 / mact1 describe them only when mnh == 2
  float delta_clip;
  int cap;
  saceo_layout L;
  saceo_tables T;
  // workspace (per-agent arrays; strides derive from the dims above)
  long long* idx; float* noise; int* perm;
  float *mb_s, *mb_a, *mb_sp, *mb_r, *mb_omd;
  float *Xpi, *aOut, *daOut, *dls;
  float *Xc, *cQ, *cdQ, *cdXa;
  float *Xc2;        // live-critic input [N_s(s) | N_a(a)] (Xc holds the target-critic input [N_s(sp) | N_a(a')])
  float *Xc3;        // actor-phase critic input [N_s(s) | N_a(pi(s))]: state columns written by the gather, action columns by the head
  float *Xm, *mOut, *mdOut, *mdXa;
  float *y, *nlp;
  float *g_q, *g_actor;
  float *lrt, *losses, *mse_part;
  unsigned long long* step_ctr;
  // expert rows actually used (bound table or host-staged copy)
  const float *expert_s, *expert_sp;
};

__device__ __forceinline__ float agent_eps(const KCtx& c, int agent) {
  return c.eps_force >= 0.f ? c.eps_force : c.T.hyper[(long long)agent * c.L.hyper_stride + 5];
}

constexpr float kLog2Pi = 1.8378770664093453f;
constexpr float kLog2 = 0.6931471805599453f;
constexpr float kMinLogStd = -5.0f, kMaxLogStd = 2.0f;   // continuous_actors.py:250-251
constexpr float kB1 = 0.9f, kB2 = 0.999f, kAdamEps = 1e-7f;  // tf.keras Adam defaults
// keras/optimizers/adam.py::update_step multiplies by the Python double (1 - beta) rounded to fp32 (0.001 -> 0.00100000005),
// not by fp32(1) - fp32(beta) (0.00099998713): pinned by tests/test_reference_pin.py against the reference's own code
constexpr float kOmB1 = (float)(1.0 - 0.9), kOmB2 = (float)(1.0 - 0.999);

__device__ __forceinline__ float softplusf(float x) {
  return x > 0.f ? x + log1pf(expf(-x)) : log1pf(expf(x));
}
__device__ __forceinline__ float nstd(float s) { return fmaxf(s, 1e-8f); }  // normalizer.py:37

__device__ __forceinline__ float block_sum(float v, float* sh) {
  // deterministic block reduction (fixed tree), blockDim.x multiple of 32, <= 1024
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) sh[w] = v;
  __syncthreads();
  float r = 0.f;
  if (w == 0) {
    r = l < nw ? sh[l] : 0.f;
    for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
    if (l == 0) sh[0] = r;
  }
  __syncthreads();
  r = sh[0];
  return r;
}

// ------------------------------------------------------------------------------------------
// step bookkeeping: Adam step counters and bias-corrected step sizes for the four optimisers
// (SAC_expert.py:108-115).  grid: ceil(n_agents*4/128)
// ------------------------------------------------------------------------------------------
__global__ void k_step_begin(KCtx c, int advance_rng) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && advance_rng) c.step_ctr[0] += 1ull;
  if (i >= c.n_agents * 4) return;
  const int agent = i >> 2, opt = i & 3;
  const int t = c.T.adam_t[i] + 1;
  c.T.adam_t[i] = t;
  const float* hy = c.T.hyper + (long long)agent * c.L.hyper_stride;
  const float lr = opt < 2 ? hy[2] : (opt == 2 ? hy[3] : hy[4]);
  const double b1t = pow((double)kB1, (double)t), b2t = pow((double)kB2, (double)t);
  c.lrt[i] = (float)((double)lr * sqrt(1.0 - b2t) / (1.0 - b1t));
}

// behaviour-cloning step (BC.py:309-363): only the actor optimiser advances.  grid: ceil(n_agents/128)
__global__ void k_bc_begin(KCtx c, int advance_rng) {
  const int agent = blockIdx.x * blockDim.x + threadIdx.x;
  if (agent == 0 && advance_rng) c.step_ctr[0] += 1ull;
  if (agent >= c.n_agents) return;
  const int t = c.T.adam_t[agent * 4 + 2] + 1;
  c.T.adam_t[agent * 4 + 2] = t;
  const float lr = c.T.hyper[(long long)agent * c.L.hyper_stride + 3];
  const double b1t = pow((double)kB1, (double)t), b2t = pow((double)kB2, (double)t);
  c.lrt[agent * 4 + 2] = (float)((double)lr * sqrt(1.0 - b2t) / (1.0 - b1t));
}
// BC_MSE_loss bookkeeping (BC.py:360-363): losses[3] = losses[4] = MSE.  grid: ceil(n_agents/128)
__global__ void k_bc_loss(KCtx c) {
  const int agent = blockIdx.x * blockDim.x + threadIdx.x;
  if (agent >= c.n_agents) return;
  float* ls = c.losses + (long long)agent * c.L.n_losses;
  const float mse = c.mse_part[agent * 2] + (c.nmod == 2 ? c.mse_part[agent * 2 + 1] : 0.f);
  ls[3] = mse; ls[4] = mse; ls[7] = 1.f;
}

// ------------------------------------------------------------------------------------------
// in-kernel draws (perf mode): idx, noise, expert permutation.  grid: (ceil(max_items/256), n_agents)
// ------------------------------------------------------------------------------------------
__global__ void k_set_seed(KCtx c, unsigned long long seed) { c.step_ctr[1] = seed; }
__global__ void k_rng_fill(KCtx c, int skip_idx) {
  const unsigned long long seed = c.step_ctr[1];
  const int agent = blockIdx.y;
  const unsigned step = (unsigned)c.step_ctr[0];
  const int q = blockIdx.x * blockDim.x + threadIdx.x;   // one Philox block (4 values) per thread
  const unsigned size = (unsigned)c.T.replay_size[agent];
  const int n_idx4 = (c.B + 3) / 4;
  const int n_noise = (3 * c.B + c.E) * c.A;
  const int n_noise4 = (n_noise + 3) / 4;
  uint32_t r[4];
  if (q < n_idx4 && !skip_idx) {      // skip_idx: the minibatch indices come from the host (np.random.randint)
    Philox::gen(seed, (uint32_t)q, (uint32_t)agent, step, 0u, r);
    for (int j = 0; j < 4; ++j) {
      const int b = 4 * q + j;
      if (b < c.B) c.idx[(long long)agent * c.B + b] = (long long)below(r[j], size);
    }
  }
  if (q < n_noise4) {
    Philox::gen(seed, (uint32_t)q, (uint32_t)agent, step, 1u, r);
    float z[4];
    normal4(r, z);
    for (int j = 0; j < 4; ++j) {
      const int e = 4 * q + j;
      if (e < n_noise) c.noise[(long long)agent * n_noise + e] = z[j];
    }
  }
  if (q == 0 && c.E > 0) {
    // Fisher-Yates shuffle of arange(E) (two-model branch only; SAC_expert.py:301-303)
    int* pm = c.perm + (long long)agent * c.E;
    for (int i = 0; i < c.E; ++i) pm[i] = i;
    if (c.nmod == 2) {
      for (int i = c.E - 1; i > 0; --i) {
        Philox::gen(seed, (uint32_t)i, (uint32_t)agent, step, 2u, r);
        const int j = (int)below(r[0], (uint32_t)(i + 1));
        const int tmp = pm[i]; pm[i] = pm[j]; pm[j] = tmp;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// replay row gather (buffers.py:135-142).  One warp per (agent, batch row): the AoS row is read
// as contiguous 16-byte vectors and scattered to the SoA outputs.  Bit-exact word copies.
// grid: (ceil(B/8), n_agents), block 256.  out_d (f64 raw words) xor omd (float 1-d) may be set.
// stage != 0 (the update path): the normalised network inputs of the critic phase are written in the same pass
// (normalizer.py:26-37, critics.py:89-93): Xpi[b] = Xc[b, :S] = N_s(sp[b]);  Xc2[b] = [N_s(s[b]) | N_a(a[b])].
// ------------------------------------------------------------------------------------------
__global__ void k_gather(KCtx c, const long long* __restrict__ idx, float* __restrict__ out_s,
                         float* __restrict__ out_a, float* __restrict__ out_sp,
                         float* __restrict__ out_r, double* __restrict__ out_d,
                         float* __restrict__ out_omd, int stage) {
  const int agent = blockIdx.y;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= c.B) return;
  long long li = idx[(long long)agent * c.B + b];
  const int start = c.T.replay_start ? c.T.replay_start[agent] : 0;
  long long phys = li + start;
  if (phys >= c.cap) phys -= c.cap;
  const int rw = c.L.row_words;
  const float4* __restrict__ row = reinterpret_cast<const float4*>(
      c.T.replay + ((long long)agent * c.cap + phys) * rw);
  const long long ob = (long long)agent * c.B + b;
  const int S = c.S, A = c.A;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  for (int v = lane; v < (rw >> 2); v += 32) {
    const float4 q = __ldg(row + v);
    const float w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int i = 4 * v + j;
      if (i < c.L.off_a) {
        if (out_s) out_s[ob * S + i] = w[j];
        if (stage) {
          const float x = (w[j] - nr[c.L.off_s_mean + i]) / nstd(nr[c.L.off_s_std + i]);
          c.Xc2[ob * c.ldXc + i] = x;
          c.Xc3[ob * c.ldXc + i] = x;
        }
      } else if (i < c.L.off_sp) {
        const int a = i - c.L.off_a;
        if (out_a) out_a[ob * A + a] = w[j];
        if (stage) c.Xc2[ob * c.ldXc + S + a] = (w[j] - nr[c.L.off_a_mean + a]) / nstd(nr[c.L.off_a_std + a]);
      } else if (i < c.L.off_r) {
        const int t = i - c.L.off_sp;
        if (out_sp) out_sp[ob * S + t] = w[j];
        if (stage) {
          const float x = (w[j] - nr[c.L.off_s_mean + t]) / nstd(nr[c.L.off_s_std + t]);
          c.Xpi[((long long)agent * c.Rs + b) * c.ldXp + t] = x;
          c.Xc[ob * c.ldXc + t] = x;
        }
      } else if (i == c.L.off_r) { if (out_r) out_r[ob] = w[j]; }
    }
    // d is an 8-byte-aligned f64 inside the row, so both words are in the same float4
    if (c.L.off_d >= 4 * v && c.L.off_d < 4 * v + 4) {
      const int j = c.L.off_d - 4 * v;
      const double d = __hiloint2double(__float_as_int(w[j + 1]), __float_as_int(w[j]));
      if (out_d) out_d[ob] = d;
      if (out_omd) out_omd[ob] = (float)(1.0 - d);   // (1-done) formed in f64 then cast, SAC_expert.py:227
    }
  }
}

// ------------------------------------------------------------------------------------------
// population-wide replay append (TrajectoryBuffer.add, buffers.py:41-71; SAC_expert.py:793-801): k new AoS rows per
// agent go behind the newest row of that agent's ring; when the ring is full the OLDEST rows are overwritten, which is
// the reference's keep-the-last-buffer_size truncation (:60-66).  Two stream-ordered launches: rows, then the ring
// bookkeeping (size / start), so that every block of the first sees the same ring state.
// grid: (ceil(k * row_words / 4 / 256), n_agents)
// ------------------------------------------------------------------------------------------
__global__ void k_replay_append_rows(KCtx c, const float* __restrict__ rows, int k, float* __restrict__ replay,
                                     const int* __restrict__ rsize, const int* __restrict__ rstart) {
  const int agent = blockIdx.y;
  const int rw4 = c.L.row_words >> 2;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;          // float4 index inside the agent's [k, row_words] block
  if (e >= k * rw4) return;
  const int i = e / rw4, v = e - i * rw4;
  const int size = rsize[agent], start = rstart ? rstart[agent] : 0;
  long long pos = (long long)start + size + i;                  // logical slot behind the newest row
  pos %= c.cap;
  const float4 q = reinterpret_cast<const float4*>(rows + ((long long)agent * k + i) * c.L.row_words)[v];
  reinterpret_cast<float4*>(replay + ((long long)agent * c.cap + pos) * c.L.row_words)[v] = q;
}
__global__ void k_replay_append_commit(KCtx c, int k, int* __restrict__ rsize, int* __restrict__ rstart) {
  const int agent = blockIdx.x * blockDim.x + threadIdx.x;
  if (agent >= c.n_agents) return;
  const int size = rsize[agent], start = rstart[agent];
  const long long tot = (long long)size + k;
  const int over = tot > c.cap ? (int)(tot - c.cap) : 0;
  rsize[agent] = tot > c.cap ? c.cap : (int)tot;
  rstart[agent] = (int)(((long long)start + over) % c.cap);
}

// ------------------------------------------------------------------------------------------
// input staging of the actor phase: normalise into the GEMM operand matrices (the critic-phase inputs are staged by
// k_gather):  Xpi[b] = N_s(s[b]);  Xpi[B+i] = N_s(sE[perm i]);  Xm[net][il,:S] = N_s^M(sE[perm i])
// grid: (ceil(R*S/256), n_agents)
// ------------------------------------------------------------------------------------------
__global__ void k_stage(KCtx c) {
  const int agent = blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int S = c.S, SA = S + c.A, B = c.B;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  const float* smean = nr + c.L.off_s_mean; const float* sstd = nr + c.L.off_s_std;
  if (e >= c.R * S) return;
  const int row = e / S, j = e - row * S;
  if (row < B) {
    c.Xpi[((long long)agent * c.Rs + row) * c.ldXp + j] =
        (c.mb_s[((long long)agent * B + row) * S + j] - smean[j]) / nstd(sstd[j]);
  } else {
    const int i = row - B;
    const int src = c.perm[(long long)agent * c.E + i];
    const float x = c.expert_s[((long long)agent * c.E + src) * S + j];
    c.Xpi[((long long)agent * c.Rs + row) * c.ldXp + j] = (x - smean[j]) / nstd(sstd[j]);
    const int half = c.nmod == 2 ? c.E / 2 : c.E;
    const int net = i / half, il = i - net * half;
    c.Xm[(((long long)agent * 2 + net) * c.E + il) * SA + j] =
        (x - nr[c.L.off_m_s_mean + j]) / nstd(nr[c.L.off_m_s_std + j]);
  }
}

// generic: Xpi[row] = N_s(obs[row]) for the inference entry points.  grid (ceil(rows*S/256), n_agents)
__global__ void k_stage_obs(KCtx c, const float* __restrict__ obs, int rows_total, int row0, int rows,
                            float* __restrict__ X, int ldx, long long sXa, int model_norm) {
  const int agent = blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= rows * c.S) return;
  const int r = e / c.S, j = e - r * c.S;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  const float mean = nr[(model_norm ? c.L.off_m_s_mean : c.L.off_s_mean) + j];
  const float sd = nr[(model_norm ? c.L.off_m_s_std : c.L.off_s_std) + j];
  X[agent * sXa + (long long)r * ldx + j] =
      (obs[((long long)agent * rows_total + row0 + r) * c.S + j] - mean) / nstd(sd);
}
// X[row, S + j] = N_a(act[row, j])   (critic / model action columns for the inference entry points)
__global__ void k_stage_act(KCtx c, const float* __restrict__ act, int rows_total, int row0, int rows,
                            float* __restrict__ X, int ldx, long long sXa, int model_norm) {
  const int agent = blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= rows * c.A) return;
  const int r = e / c.A, j = e - r * c.A;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  const float mean = nr[(model_norm ? c.L.off_m_a_mean : c.L.off_a_mean) + j];
  const float sd = nr[(model_norm ? c.L.off_m_a_std : c.L.off_a_std) + j];
  X[agent * sXa + (long long)r * ldx + c.S + j] =
      (act[((long long)agent * rows_total + row0 + r) * c.A + j] - mean) / nstd(sd);
}

// ------------------------------------------------------------------------------------------
// tanh-Gaussian head forward: SquashedGaussianActor.evaluate / .sample
// (continuous_actors.py:270-306, 327-379).  One thread per row.
//   rows [0, nmain): evaluate -> neglogp, squashed action normalised into Xc[:, S:]   (write_xc)
//   rows [nmain, nrows): sample (expert rows) -> normalised into Xm[net][il, S:]
//   act_out != null: raw pi rows are also written there (inference entry point)
// noise_row0: row offset of this pass inside the per-agent noise block (u1|u2|uE|u5).
// grid: (ceil(nrows/128), n_agents)
// ------------------------------------------------------------------------------------------
__global__ void k_head_fwd(KCtx c, int nrows, int nmain, const float* __restrict__ noise,
                           long long noise_agent_stride, int noise_row0, int write_xc,
                           float* __restrict__ act_out, float* __restrict__ nlp_out,
                           long long out_agent_stride_rows, int out_row0) {
  const int agent = blockIdx.y;
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= nrows) return;
  const int A = c.A, Ao = c.Ao, S = c.S, SA = S + A;
  const float* out = c.aOut + ((long long)agent * c.Rs + row) * Ao;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  const float* lsv = c.T.actor + (long long)agent * c.L.na_stride + (c.L.na - A);
  const float* u = noise ? noise + agent * noise_agent_stride + (long long)(noise_row0 + row) * A : nullptr;
  float acc_g = 0.f, acc_c = 0.f;
  const bool expert = row >= nmain;
  int net = 0, il = 0;
  if (expert) {
    const int i = row - nmain;
    const int half = c.nmod == 2 ? c.E / 2 : c.E;
    net = i / half; il = i - net * half;
  }
  for (int j = 0; j < A; ++j) {
    const float mean = out[j];
    const float ls_raw = c.per_state_std ? out[A + j] : lsv[j];
    const float ls = fminf(fmaxf(ls_raw, kMinLogStd), kMaxLogStd);
    const float sd = expf(ls);
    const float z = u ? mean + sd * u[j] : mean;
    const float qn = (z - mean) / sd;
    acc_g += qn * qn + 2.f * ls + kLog2Pi;
    acc_c += 2.f * (kLog2 - z - softplusf(-2.f * z));
    const float pi = nr[c.L.off_act_limit + j] * tanhf(z);
    if (act_out) act_out[((long long)agent * out_agent_stride_rows + out_row0 + row) * A + j] = pi;
    if (!expert) {
      if (write_xc)
        (write_xc == 2 ? c.Xc2 : c.Xc)[((long long)agent * c.B + row) * c.ldXc + S + j] =
            (pi - nr[c.L.off_a_mean + j]) / nstd(nr[c.L.off_a_std + j]);
    } else {
      c.Xm[(((long long)agent * 2 + net) * c.E + il) * SA + S + j] =
          (pi - nr[c.L.off_m_a_mean + j]) / nstd(nr[c.L.off_m_a_std + j]);
    }
  }
  const float nlp = 0.5f * acc_g + acc_c;
  if (!expert) c.nlp[(long long)agent * c.Rs + row] = nlp;
  if (nlp_out) nlp_out[(long long)agent * out_agent_stride_rows + out_row0 + row] = nlp;
}

// TD target (SAC_expert.py:211-229): y = r + gamma * ((1-d) * (min(Qt1,Qt2)*max(ret_std,1e-8) + alpha*nlp))
// alpha is the RAW variable (no exp).  grid: (ceil(B/128), n_agents)
__global__ void k_td_target(KCtx c) {
  const int agent = blockIdx.y;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= c.B) return;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  const float ret = nstd(nr[c.L.off_ret_std]);
  const float gamma = c.T.hyper[(long long)agent * c.L.hyper_stride + 0];
  const float alpha = c.T.alpha[agent];
  const float q0 = c.cQ[((long long)agent * 2 + 0) * c.B + b] * ret;
  const float q1 = c.cQ[((long long)agent * 2 + 1) * c.B + b] * ret;
  const float nv = fminf(q0, q1) + alpha * c.nlp[(long long)agent * c.Rs + b];
  const long long o = (long long)agent * c.B + b;
  c.y[o] = c.mb_r[o] + gamma * (c.mb_omd[o] * nv);
}

// critic loss + dL/dq (SAC_expert.py:238-250): L = mean_b 0.5 (q - y)^2, dq = (q - y)/B.
// grid: (2, n_agents), block 256
__global__ void k_critic_loss(KCtx c) {
  __shared__ float sh[32];
  const int net = blockIdx.x, agent = blockIdx.y;
  const long long o = ((long long)agent * 2 + net) * c.B;
  const float invB = 1.f / (float)c.B;
  float acc = 0.f;
  for (int b = threadIdx.x; b < c.B; b += blockDim.x) {
    const float d = c.cQ[o + b] - c.y[(long long)agent * c.B + b];
    acc += 0.5f * d * d;
    c.cdQ[o + b] = d * invB;
  }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) c.losses[(long long)agent * c.L.n_losses + net] = acc * invB;
}

// actor main loss (SAC_expert.py:312-319): L_pi = mean(-alpha*nlp - min(Q1,Q2)); dL/dq_k with
// reduce_min tie-splitting; scaled by (1-eps) when the expert term is on.  grid: (n_agents), block 256
__global__ void k_actor_q(KCtx c) {
  __shared__ float sh[32];
  const int agent = blockIdx.x;
  const float alpha = c.T.alpha[agent];
  const float eps = agent_eps(c, agent);
  const float wpi = c.nmod > 0 ? 1.f - eps : 1.f;
  const float sc = -wpi / (float)c.B;
  float acc = 0.f;
  for (int b = threadIdx.x; b < c.B; b += blockDim.x) {
    const float q0 = c.cQ[((long long)agent * 2 + 0) * c.B + b];
    const float q1 = c.cQ[((long long)agent * 2 + 1) * c.B + b];
    const float s0 = q0 < q1 ? 1.f : (q0 == q1 ? 0.5f : 0.f);
    c.cdQ[((long long)agent * 2 + 0) * c.B + b] = sc * s0;
    c.cdQ[((long long)agent * 2 + 1) * c.B + b] = sc * (1.f - s0);
    acc += -alpha * c.nlp[(long long)agent * c.Rs + b] - fminf(q0, q1);
  }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) {
    c.losses[(long long)agent * c.L.n_losses + 2] = acc / (float)c.B;
    if (c.nmod == 0) c.losses[(long long)agent * c.L.n_losses + 3] = 0.f;
  }
}

// expert-observation term (SAC_expert.py:325-335; base_world_model.py:65-87; continuous_models.py:244-254):
// pred = sE + clip(delta)*max(std_d,1e-8) + mean_d; MSE = mean_i 0.5 sum_j err^2 (both halves summed);
// writes d(eps*MSE)/d(delta) into mdOut.  grid: (n_agents), block 256
__global__ void k_model_loss(KCtx c) {
  __shared__ float sh[32];
  const int agent = blockIdx.x;
  const int S = c.S, E = c.E;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  const float eps = agent_eps(c, agent);
  const int half = c.nmod == 2 ? E / 2 : E;
  const float inv = 1.f / (float)half;
  float acc = 0.f;
  for (int e = threadIdx.x; e < E * S; e += blockDim.x) {
    const int i = e / S, j = e - i * S;
    const int net = i / half, il = i - net * half;
    const int src = c.perm[(long long)agent * E + i];
    float delta = c.mOut[(((long long)agent * 2 + net) * E + il) * c.mo + j];
    float cm = 1.f;
    if (c.delta_clip > 0.f) {
      cm = (delta >= -c.delta_clip && delta <= c.delta_clip) ? 1.f : 0.f;
      delta = fminf(fmaxf(delta, -c.delta_clip), c.delta_clip);
    }
    const float sd = nstd(nr[c.L.off_m_d_std + j]);
    const float pred = c.expert_s[((long long)agent * E + src) * S + j] + (delta * sd + nr[c.L.off_m_d_mean + j]);
    const float err = c.expert_sp[((long long)agent * E + src) * S + j] - pred;
    acc += 0.5f * err * err;
    c.mdOut[(((long long)agent * 2 + net) * E + il) * S + j] = (-err * inv * eps) * sd * cm;
  }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) { c.mse_part[agent * 2] = acc * inv; c.mse_part[agent * 2 + 1] = 0.f; }
}

// head backward (SURVEY.md App. A): dL/d(out) from dL/d(pi) and dL/d(neglogp).  One thread per row.
//   main rows:   g_pi = (dXa[q1] + dXa[q2]) / max(a_std,1e-8),  g_nlp = -alpha*(1-eps)/B
//   expert rows: g_pi = mdXa / max(a_std^M,1e-8),               g_nlp = 0
// grid: (ceil(R/128), n_agents)
__global__ void k_head_bwd(KCtx c, int nrows) {
  const int agent = blockIdx.y;
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= nrows) return;
  const int A = c.A, Ao = c.Ao, B = c.B;
  const float* out = c.aOut + ((long long)agent * c.Rs + row) * Ao;
  float* dout = c.daOut + ((long long)agent * c.Rs + row) * Ao;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  const float* lsv = c.T.actor + (long long)agent * c.L.na_stride + (c.L.na - A);
  const float alpha = c.T.alpha[agent];
  const float eps = agent_eps(c, agent);
  const float wpi = c.nmod > 0 ? 1.f - eps : 1.f;
  const bool expert = row >= B;
  const float g_nlp = expert ? 0.f : -alpha * wpi / (float)B;
  const int n_noise = (3 * B + c.E) * A;
  // actor-phase noise: u2 rows [B,2B), expert rows [2B, 2B+E)
  const float* u = c.noise + (long long)agent * n_noise + (long long)(B + row) * A;
  int net = 0, il = 0;
  if (expert) {
    const int i = row - B;
    const int half = c.nmod == 2 ? c.E / 2 : c.E;
    net = i / half; il = i - net * half;
  }
  for (int j = 0; j < A; ++j) {
    const float mean = out[j];
    const float ls_raw = c.per_state_std ? out[A + j] : lsv[j];
    const float ls = fminf(fmaxf(ls_raw, kMinLogStd), kMaxLogStd);
    const float sd = expf(ls);
    const float z = mean + sd * u[j];
    const float t = tanhf(z);
    float g_pi;
    if (!expert) {
      g_pi = (c.cdXa[(((long long)agent * 2 + 0) * B + row) * A + j] +
              c.cdXa[(((long long)agent * 2 + 1) * B + row) * A + j]) / nstd(nr[c.L.off_a_std + j]);
    } else {
      g_pi = c.mdXa[(((long long)agent * 2 + net) * c.E + il) * A + j] / nstd(nr[c.L.off_m_a_std + j]);
    }
    const float dz = g_pi * nr[c.L.off_act_limit + j] * (1.f - t * t) + g_nlp * (-2.f * t);
    const float mask = (ls_raw >= kMinLogStd && ls_raw <= kMaxLogStd) ? 1.f : 0.f;
    const float dl = (dz * sd * u[j] + g_nlp) * mask;
    dout[j] = dz;
    if (c.per_state_std) dout[A + j] = dl;
    else c.dls[((long long)agent * c.Rs + row) * A + j] = dl;
  }
}

// state-independent logstd gradient: column sums of dls in fixed row order (deterministic).
// grid: (n_agents), block >= A
__global__ void k_lsv_reduce(KCtx c, int nrows) {
  const int agent = blockIdx.x, j = threadIdx.x;
  if (j >= c.A) return;
  float acc = 0.f;
  for (int r = 0; r < nrows; ++r) acc += c.dls[((long long)agent * c.Rs + r) * c.A + j];
  c.g_actor[(long long)agent * c.L.na_stride + (c.L.na - c.A) + j] = acc;
}

// Keras Adam (epsilon outside the bias correction) fused with the Polyak target update
// (SAC_expert.py:243,250,338; 362-373).  grid: (ceil(n/256), nnet, n_agents)
// launch bounds: <= 64 registers (48 used, no spills; (256, 6) = 40 registers spilled 1.2 M local loads per launch)
__global__ void __launch_bounds__(256, 4) k_adam(float* __restrict__ theta, float* __restrict__ m, float* __restrict__ v,
                       const float* __restrict__ g, float* __restrict__ target,
                       const float* __restrict__ lrt, const float* __restrict__ hyper, int hyper_stride,
                       int opt0, long long n, long long stride, int nnet, int do_polyak,
                       uint8_t* __restrict__ planes, uint8_t* __restrict__ tplanes, int K0, int nout) {
  // planes / tplanes (nullable): fp16 hi/lo weight-plane images of theta / target (planes.cuh), one image per
  // (agent, net), kept current here so that no forward / backward pass ever converts a weight again
  // one float4 (4 consecutive parameters) per thread: every table row is 128-byte aligned (strides are multiples of 32)
  const int agent = blockIdx.z, net = blockIdx.y;
  const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 >= n) return;
  const long long o = ((long long)agent * nnet + net) * stride + i4;
  const float lr_t = lrt[agent * 4 + opt0 + net];
  const float4 g4 = *reinterpret_cast<const float4*>(g + o);
  float4 m4 = *reinterpret_cast<const float4*>(m + o);
  float4 v4 = *reinterpret_cast<const float4*>(v + o);
  float4 t4 = *reinterpret_cast<const float4*>(theta + o);
  float4 q4 = do_polyak ? *reinterpret_cast<const float4*>(target + o) : make_float4(0.f, 0.f, 0.f, 0.f);
  const float tau = do_polyak ? hyper[(long long)agent * hyper_stride + 1] : 0.f;
  const float one_m = (float)(1.0 - (double)tau);
  const float gi[4] = {g4.x, g4.y, g4.z, g4.w};
  float mi[4] = {m4.x, m4.y, m4.z, m4.w}, vi[4] = {v4.x, v4.y, v4.z, v4.w}, th[4] = {t4.x, t4.y, t4.z, t4.w},
        tg[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (i4 + j < n) {          // words past n are padding (the actor's last pad word carries g_alpha): left untouched
      mi[j] = kB1 * mi[j] + kOmB1 * gi[j];
      vi[j] = kB2 * vi[j] + kOmB2 * gi[j] * gi[j];
      th[j] = th[j] - lr_t * mi[j] / (sqrtf(vi[j]) + kAdamEps);
      // NumPy fp32: two rounded products, one rounded sum (no FMA contraction)
      tg[j] = __fadd_rn(__fmul_rn(tg[j], one_m), __fmul_rn(th[j], tau));
    }
  }
  *reinterpret_cast<float4*>(m + o) = make_float4(mi[0], mi[1], mi[2], mi[3]);
  *reinterpret_cast<float4*>(v + o) = make_float4(vi[0], vi[1], vi[2], vi[3]);
  *reinterpret_cast<float4*>(theta + o) = make_float4(th[0], th[1], th[2], th[3]);
  if (do_polyak) *reinterpret_cast<float4*>(target + o) = make_float4(tg[0], tg[1], tg[2], tg[3]);
  if (planes) {
    const long long ib = ((long long)agent * nnet + net) * ws_image_bytes(K0, nout);
    ws_planes_store4(planes + ib, K0, nout, i4, th);
    if (do_polyak && tplanes) ws_planes_store4(tplanes + ib, K0, nout, i4, tg);
  }
}

// temperature step + loss bookkeeping (SAC_expert.py:341-356).  grid: (n_agents), block 256
//   L_alpha = -alpha * mean(-nlp3 + H);  g = -mean(-nlp3 + H);  Adam;  alpha = max(alpha, 1e-5)
__global__ void k_alpha_step(KCtx c, int apply) {
  __shared__ float sh[32];
  const int agent = blockIdx.x;
  const float* hy = c.T.hyper + (long long)agent * c.L.hyper_stride;
  const float te = hy[6];
  float acc = 0.f;
  for (int b = threadIdx.x; b < c.B; b += blockDim.x) acc += -c.nlp[(long long)agent * c.Rs + b] + te;
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) {
    float* ls = c.losses + (long long)agent * c.L.n_losses;
    const float alpha = c.T.alpha[agent];
    const float mean_term = acc / (float)c.B;
    const float g = -mean_term;
    ls[5] = -alpha * mean_term;
    const float eps = hy[5];
    if (c.nmod > 0) ls[3] = c.mse_part[agent * 2] + (c.nmod == 2 ? c.mse_part[agent * 2 + 1] : 0.f);   // fixed order
    ls[4] = c.nmod > 0 ? (1.f - eps) * ls[2] + eps * ls[3] : ls[2];
    ls[7] = eps;
    c.g_actor[(long long)agent * c.L.na_stride + c.L.na_stride - 1] = g;   // last padded word: g_alpha (DP all-reduce rides along)
    if (apply) {
      const float lr_t = c.lrt[agent * 4 + 3];
      const float mi = kB1 * c.T.alpha_m[agent] + kOmB1 * g;
      const float vi = kB2 * c.T.alpha_v[agent] + kOmB2 * g * g;
      float a = alpha - lr_t * mi / (sqrtf(vi) + kAdamEps);
      a = fmaxf(a, 1e-5f);
      c.T.alpha_m[agent] = mi; c.T.alpha_v[agent] = vi; c.T.alpha[agent] = a;
      ls[6] = a;
    }
  }
}
// apply-only half for the data-parallel mode (g_alpha already all-reduced in g_actor's last word)
__global__ void k_alpha_apply(KCtx c) {
  const int agent = blockIdx.x * blockDim.x + threadIdx.x;
  if (agent >= c.n_agents) return;
  const float g = c.g_actor[(long long)agent * c.L.na_stride + c.L.na_stride - 1];
  const float lr_t = c.lrt[agent * 4 + 3];
  const float mi = kB1 * c.T.alpha_m[agent] + kOmB1 * g;
  const float vi = kB2 * c.T.alpha_v[agent] + kOmB2 * g * g;
  float a = c.T.alpha[agent] - lr_t * mi / (sqrtf(vi) + kAdamEps);
  a = fmaxf(a, 1e-5f);
  c.T.alpha_m[agent] = mi; c.T.alpha_v[agent] = vi; c.T.alpha[agent] = a;
  c.losses[(long long)agent * c.L.n_losses + 6] = a;
}

// critic.value scaling / model.sample epilogue for the inference entry points
__global__ void k_scale_ret(KCtx c, float* __restrict__ q, int rows) {
  const int agent = blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= 2 * rows) return;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  q[(long long)agent * 2 * rows + e] *= nstd(nr[c.L.off_ret_std]);
}
// sp_out[agent, net, row0+r, j] = obs + clip(delta)*max(std_d,1e-8) + mean_d
__global__ void k_model_out(KCtx c, const float* __restrict__ obs, int rows_total, int row0, int rows,
                            float* __restrict__ sp_out) {
  const int agent = blockIdx.y, net = blockIdx.z;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= rows * c.S) return;
  const int r = e / c.S, j = e - r * c.S;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  float delta = c.mOut[(((long long)agent * 2 + net) * c.E + r) * c.mo + j];
  if (c.delta_clip > 0.f) delta = fminf(fmaxf(delta, -c.delta_clip), c.delta_clip);
  const float x = obs[((long long)agent * rows_total + row0 + r) * c.S + j];
  sp_out[(((long long)agent * 2 + net) * rows_total + row0 + r) * c.S + j] =
      x + (delta * nstd(nr[c.L.off_m_d_std + j]) + nr[c.L.off_m_d_mean + j]);
}

}  // namespace saceo
