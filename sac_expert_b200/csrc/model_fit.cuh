// Dynamics-model fitting for the whole population (SURVEY.md §8f rank 1):
//   MBRLOnPolicyAlg._apply_model_grads   sac_eo/algs/mbrl_onpolicy_alg.py:301-319
//   MSEModel.get_loss                    sac_eo/models/continuous_models.py:280-302
//   BaseWorldModel._forward(clip=False)  sac_eo/models/base_world_model.py:65-87
// One "fit step" = for every agent: every model's loss on its own minibatch of replay rows, summed;
// optional tf.clip_by_global_norm over ALL models' tensors; one joint Keras Adam step.
// The MLP forward / backward / weight-gradient GEMMs are the generic ones of saceo.cu; this file holds
// the row staging, the loss + output gradient, the global-norm reduction and the Adam step.
#pragma once
#include "elem.cuh"

namespace saceo {

enum { FIT_LR = 0, FIT_RCOEF = 1, FIT_DCLIP = 2, FIT_RCLIP = 3, FIT_MAXNORM = 4, FIT_RMEAN = 5, FIT_RSTD = 6, FIT_SCALE = 7, FIT_HYPER = 8 };

struct FitCtx {
  // caller tables (saceo_fit_tables)
  float *model, *m, *v; int* t; const float* hyper;
  float *ls, *ls_m, *ls_v;   // GaussianModel.logstd [n_agents, 2, S] and its Adam slots (NULL: MSEModel loss)
  float *g_ls;               // workspace: gradient of logstd [n_agents, 2, S]
  // workspace, all [n_agents, 2, ...]
  float *X, *T, *Out, *dOut, *g;
  float *loss_part;      // [n_agents, 2]
  float *gscale;         // [n_agents] gradient scale of clip_by_global_norm (1 when clipping is off)
  float *gnorm;          // [n_agents] global gradient norm (diagnostic)
  float *lrt;            // [n_agents] bias-corrected Adam step size
  int S, mb, mbs, nmod, use_clip;     // mbs: row stride of the minibatch buffers (mb rounded up to 32, pad rows stay zero)
  long long nm, nm_stride;
  // separate_reward_nn: the reward network of every model (caller tables + workspace), NULL otherwise
  float *rw, *rw_m, *rw_v, *g_r;
  float *rOut, *rdOut;
  long long nr, nr_stride;
};

// Adam step counter and step size of the joint model optimiser.  grid: ceil(n_agents/128)
__global__ void k_fit_begin(FitCtx f, int n_agents) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_agents) return;
  const int t = f.t[i] + 1;
  f.t[i] = t;
  const float lr = f.hyper[i * FIT_HYPER + FIT_LR];
  const double b1t = pow((double)kB1, (double)t), b2t = pow((double)kB2, (double)t);
  f.lrt[i] = (float)((double)lr * sqrt(1.0 - b2t) / (1.0 - b1t));
  f.gscale[i] = 1.f;
}

// Gathers the minibatch rows of every (agent, model) from the device replay table (same logical ->
// physical ring mapping as k_gather) and stages the normalised network input and regression target:
//   X[row] = [ N_s(s) | N_a(a) ]                         base_world_model.py:67-70
//   T[row] = [ clip(N_delta(sp - s)) | clip(N_r(r)) ]    continuous_models.py:284-296
// grid: (ceil(mb*(2S+A+1)/256), nmod, n_agents)
__global__ void k_fit_stage(KCtx c, FitCtx f, const long long* __restrict__ idx) {
  const int agent = blockIdx.z, net = blockIdx.y;
  const int S = c.S, A = c.A, SA = S + A, W = SA + S + 1;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= f.mb * W) return;
  const int row = e / W, col = e - row * W;
  const long long an = (long long)agent * 2 + net;
  const long long li = idx[((long long)agent * f.nmod + net) * f.mb + row];
  const int start = c.T.replay_start ? c.T.replay_start[agent] : 0;
  long long phys = li + start;
  if (phys >= c.cap) phys -= c.cap;
  const float* __restrict__ src = c.T.replay + ((long long)agent * c.cap + phys) * c.L.row_words;
  const float* nr = c.T.norm + (long long)agent * c.L.norm_stride;
  const float* hy = f.hyper + (long long)agent * FIT_HYPER;
  if (col < S) {
    f.X[(an * f.mbs + row) * SA + col] = (src[c.L.off_s + col] - nr[c.L.off_m_s_mean + col]) / nstd(nr[c.L.off_m_s_std + col]);
  } else if (col < SA) {
    const int j = col - S;
    f.X[(an * f.mbs + row) * SA + col] = (src[c.L.off_a + j] - nr[c.L.off_m_a_mean + j]) / nstd(nr[c.L.off_m_a_std + j]);
  } else if (col < SA + S) {
    const int j = col - SA;
    const float d = src[c.L.off_sp + j] - src[c.L.off_s + j];
    float dn = (d - nr[c.L.off_m_d_mean + j]) / nstd(nr[c.L.off_m_d_std + j]);
    const float cl = hy[FIT_DCLIP];
    if (cl > 0.f) dn = fminf(fmaxf(dn, -cl), cl);
    f.T[(an * f.mbs + row) * (S + 1) + j] = dn;
  } else {
    float rn = (src[c.L.off_r] - hy[FIT_RMEAN]) / nstd(hy[FIT_RSTD]);
    const float cl = hy[FIT_RCLIP];
    if (cl > 0.f) rn = fminf(fmaxf(rn, -cl), cl);
    f.T[(an * f.mbs + row) * (S + 1) + S] = rn;
  }
}

// loss and its gradient w.r.t. the network output.  grid: (nmod, n_agents), block 256
//   MSEModel (continuous_models.py:280-302):
//     L = mean_b( 0.5*sum_j (T_j - P_j)^2 + coef*0.5*(T_r - P_r)^2 );  dP_j = (P_j - T_j) / mb
//   GaussianModel (continuous_models.py:101-131), logstd ls[S] trainable and unclipped:
//     L = mean_b( sc*0.5*sum_j(((T_j - P_j)/exp(ls_j))^2 + 2 ls_j + log 2pi) + coef*0.5*(T_r - P_r)^2 )
//     sc = stop_gradient(mean_j exp(ls_j)^2) if scale_model_loss else 1
//     dP_j = sc (P_j - T_j) exp(-2 ls_j) / mb;   dL/dls_j = sc * mean_b(1 - (T_j - P_j)^2 exp(-2 ls_j))
__global__ void k_fit_loss(KCtx c, FitCtx f, float* __restrict__ losses_out) {
  __shared__ float sh[32];
  __shared__ float w[512];              // exp(-2 ls_j) per output column (S <= 512 checked at bind time)
  __shared__ float sc_s, lsum_s;
  const int agent = blockIdx.y, net = blockIdx.x;
  const int S = c.S, mt = S + 1;                 // target rows: [delta (S) | reward]
  const int mo = f.rw ? S : S + 1;               // model output width (separate_reward_nn: delta columns only)
  const long long an = (long long)agent * 2 + net;
  const float* hy = f.hyper + (long long)agent * FIT_HYPER;
  const float coef = hy[FIT_RCOEF];
  const float inv = 1.f / (float)f.mb;
  const float* ls = f.ls ? f.ls + an * S : nullptr;
  if (ls) {
    for (int j = threadIdx.x; j < S; j += blockDim.x) w[j] = expf(-2.f * ls[j]);
    if (threadIdx.x == 0) {             // fixed-order scalars
      float var = 0.f, lsum = 0.f;
      for (int j = 0; j < S; ++j) { const float sd = expf(ls[j]); var += sd * sd; lsum += 2.f * ls[j] + kLog2Pi; }
      sc_s = hy[FIT_SCALE] != 0.f ? var / (float)S : 1.f;
      lsum_s = lsum;
    }
  } else {
    for (int j = threadIdx.x; j < S; j += blockDim.x) w[j] = 1.f;
    if (threadIdx.x == 0) { sc_s = 1.f; lsum_s = 0.f; }
  }
  __syncthreads();
  const float sc = sc_s;
  float acc = 0.f;
  for (int row = threadIdx.x; row < f.mb; row += blockDim.x) {
    const float* P = f.Out + (an * f.mbs + row) * mo;
    const float* T = f.T + (an * f.mbs + row) * mt;
    float* dP = f.dOut + (an * f.mbs + row) * mo;
    float dl = 0.f;
    for (int j = 0; j < S; ++j) {
      const float e = P[j] - T[j];
      dl += e * e * w[j];
      dP[j] = sc * e * w[j] * inv;
    }
    const float er = (f.rw ? f.rOut[an * f.mbs + row] : P[S]) - T[S];
    if (f.rw) f.rdOut[an * f.mbs + row] = coef * er * inv;
    else dP[S] = coef * er * inv;
    acc += sc * (0.5f * (dl + lsum_s)) + coef * (0.5f * er * er);
  }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) {
    const float L = acc * inv;
    f.loss_part[an] = L;
    if (losses_out) losses_out[(long long)agent * f.nmod + net] = L;
  }
  if (ls) {                             // dL/dls_j: one thread per column, rows in fixed order
    for (int j = threadIdx.x; j < S; j += blockDim.x) {
      float g = 0.f;
      for (int row = 0; row < f.mb; ++row) {
        const float e = f.Out[(an * f.mbs + row) * mo + j] - f.T[(an * f.mbs + row) * mt + j];
        g += 1.f - e * e * w[j];
      }
      f.g_ls[an * S + j] = sc * g * inv;
    }
  }
}

// tf.clip_by_global_norm over every tensor of every model of one agent (mbrl_onpolicy_alg.py:315-317):
// scale = clip * min(1/||g||, 1/clip), clip = model_max_grad_norm * num_models.  grid: (n_agents), block 1024
__global__ void k_fit_gnorm(FitCtx f) {
  __shared__ float sh[32];
  const int agent = blockIdx.x;
  float acc = 0.f;
  for (int net = 0; net < f.nmod; ++net) {
    const float* g = f.g + ((long long)agent * 2 + net) * f.nm_stride;
    for (long long i = threadIdx.x; i < f.nm; i += blockDim.x) { const float x = g[i]; acc += x * x; }
    if (f.ls) {
      const float* gl = f.g_ls + ((long long)agent * 2 + net) * f.S;
      for (int i = threadIdx.x; i < f.S; i += blockDim.x) { const float x = gl[i]; acc += x * x; }
    }
    if (f.rw) {
      const float* gr = f.g_r + ((long long)agent * 2 + net) * f.nr_stride;
      for (long long i = threadIdx.x; i < f.nr; i += blockDim.x) { const float x = gr[i]; acc += x * x; }
    }
  }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) {
    const float norm = sqrtf(acc);
    f.gnorm[agent] = norm;
    const float mgn = f.hyper[(long long)agent * FIT_HYPER + FIT_MAXNORM];
    if (mgn > 0.f) {
      const float clip = mgn * (float)f.nmod;
      f.gscale[agent] = clip * fminf(1.f / norm, 1.f / clip);
    }
  }
}

// joint Keras Adam over all model tensors (one step counter per agent).  grid: (ceil(ceil(nm/4)/256), nmod, n_agents)
// reward != 0: the same step on the reward networks' tensors (separate_reward_nn).
__global__ void k_fit_adam(FitCtx f, int reward) {
  const int agent = blockIdx.z, net = blockIdx.y;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const float lr_t = f.lrt[agent];
  if (reward) { f.model = f.rw; f.m = f.rw_m; f.v = f.rw_v; f.g = f.g_r; f.nm = f.nr; f.nm_stride = f.nr_stride; f.ls = nullptr; }
  if (f.ls && blockIdx.x == 0) {                           // the logstd variable rides in the first block
    for (int j = threadIdx.x; j < f.S; j += blockDim.x) {
      const long long o = ((long long)agent * 2 + net) * f.S + j;
      const float gi = f.g_ls[o] * f.gscale[agent];
      const float mi = kB1 * f.ls_m[o] + kOmB1 * gi;
      const float vi = kB2 * f.ls_v[o] + kOmB2 * gi * gi;
      f.ls[o] = f.ls[o] - lr_t * mi / (sqrtf(vi) + kAdamEps);
      f.ls_m[o] = mi; f.ls_v[o] = vi;
    }
  }
  const long long i4 = i * 4;             // one float4 per thread (rows are 128-byte aligned, nm_stride % 32 == 0)
  if (i4 >= f.nm) return;
  const long long o = ((long long)agent * 2 + net) * f.nm_stride + i4;
  const float gs = f.gscale[agent];
  const float4 g4 = *reinterpret_cast<const float4*>(f.g + o);
  const float4 m4 = *reinterpret_cast<const float4*>(f.m + o);
  const float4 v4 = *reinterpret_cast<const float4*>(f.v + o);
  const float4 t4 = *reinterpret_cast<const float4*>(f.model + o);
  const float gi[4] = {g4.x * gs, g4.y * gs, g4.z * gs, g4.w * gs};
  float mi[4] = {m4.x, m4.y, m4.z, m4.w}, vi[4] = {v4.x, v4.y, v4.z, v4.w}, th[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (i4 + j < f.nm) {
      mi[j] = kB1 * mi[j] + kOmB1 * gi[j];
      vi[j] = kB2 * vi[j] + kOmB2 * gi[j] * gi[j];
      th[j] = th[j] - lr_t * mi[j] / (sqrtf(vi[j]) + kAdamEps);
    }
  }
  *reinterpret_cast<float4*>(f.m + o) = make_float4(mi[0], mi[1], mi[2], mi[3]);
  *reinterpret_cast<float4*>(f.v + o) = make_float4(vi[0], vi[1], vi[2], vi[3]);
  *reinterpret_cast<float4*>(f.model + o) = make_float4(th[0], th[1], th[2], th[3]);
}

}  // namespace saceo
