// Fisher-vector product pieces and the conjugate-gradient recurrences.
//   F x = (1/N) sum_s J_s^T diag(exp(-2 logstd_s), 2) J_s x + damp x       (SURVEY.md App. B)
// which equals the reference's double back-prop of the mean forward KL at theta_ref = theta
// (sac_eo/algs/model_free/trpo.py:200-227 with GaussianActor.kl / ._forward,
//  sac_eo/actors/continuous_actors.py:74-100,159-184).  The GEMMs (tangent forward, VJP backward)
// are issued by saceo.cu; here are the per-row metric and the per-agent vector recurrences of
// cg() (sac_eo/common/update_utils.py:4-24).
#pragma once
#include "elem.cuh"

namespace saceo {

struct FvpWs {
  int N;
  float *Out, *Tmp, *TOut, *G, *gls;
  float *p, *r, *z, *x, *sc;   // CG vectors [n, na_stride]; sc[agent*8 + {0: rr, 1: active}]
};

// per (agent, state row): G = M . (J x) / N in the GaussianActor._forward parameterisation
//   per-state std: logstd = log(softplus(o2)) + log(std_mult) - log(log 2), floor log(1e-3)
//   state-indep:   logstd = logstd_var + log(std_mult),                    floor log(1e-3)
// grid: (ceil(N/128), n_agents)
__global__ void k_fvp_metric(KCtx c, FvpWs f, const float* __restrict__ xin, float std_mult) {
  const int agent = blockIdx.y;
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= f.N) return;
  const int A = c.A, Ao = c.Ao;
  const float invN = 1.f / (float)f.N;
  const float floor_ls = logf(1e-3f);
  const float* out = f.Out + ((long long)agent * f.N + row) * Ao;
  const float* tout = f.TOut + ((long long)agent * f.N + row) * Ao;
  float* g = f.G + ((long long)agent * f.N + row) * Ao;
  const float* theta = c.T.actor + (long long)agent * c.L.na_stride;
  const float* tang = xin + (long long)agent * c.L.na_stride;
  for (int j = 0; j < A; ++j) {
    if (c.per_state_std) {
      const float o2 = out[A + j];
      const float sp = softplusf(o2);
      float ls = logf(sp) + (logf(std_mult) - logf(kLog2));
      const float mask = ls >= floor_ls ? 1.f : 0.f;
      ls = fmaxf(ls, floor_ls);
      const float dls = (1.f / (1.f + expf(-o2))) / sp * mask;     // d logstd / d o2
      g[j] = expf(-2.f * ls) * tout[j] * invN;
      g[A + j] = 2.f * (tout[A + j] * dls) * invN * dls;
    } else {
      float ls = theta[c.L.na - A + j] + logf(std_mult);
      const float mask = ls >= floor_ls ? 1.f : 0.f;
      ls = fmaxf(ls, floor_ls);
      g[j] = expf(-2.f * ls) * tout[j] * invN;
      f.gls[((long long)agent * f.N + row) * A + j] = 2.f * (tang[c.L.na - A + j] * mask) * invN * mask;
    }
  }
}

// Fx[logstd_var] = column sums (fixed order), then Fx += damp * x.  grid: (ceil(na/256), n_agents)
__global__ void k_fvp_finish(KCtx c, FvpWs f, const float* __restrict__ xin, float damp, float* __restrict__ Fx) {
  const int agent = blockIdx.y;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.L.na) return;
  const long long o = (long long)agent * c.L.na_stride + i;
  float v;
  if (!c.per_state_std && i >= c.L.na - c.A) {
    const int j = (int)(i - (c.L.na - c.A));
    v = 0.f;
    for (int r = 0; r < f.N; ++r) v += f.gls[((long long)agent * f.N + r) * c.A + j];
  } else {
    v = Fx[o];
  }
  Fx[o] = v + damp * xin[o];
}

// cg(): p = r = b, x = 0, rdotr = r.r            update_utils.py:6-9.   grid: (n_agents), block 256
__global__ void k_cg_init(KCtx c, FvpWs f, const float* __restrict__ b) {
  __shared__ float sh[32];
  const int agent = blockIdx.x;
  const long long o = (long long)agent * c.L.na_stride;
  float acc = 0.f;
  for (long long i = threadIdx.x; i < c.L.na; i += blockDim.x) {
    const float v = b[o + i];
    f.p[o + i] = v; f.r[o + i] = v; f.x[o + i] = 0.f;
    acc += v * v;
  }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) { f.sc[agent * 8 + 0] = acc; f.sc[agent * 8 + 1] = 1.f; }
}

// one loop body after z = F(p):  v = rr/(p.z); x += v p; r -= v z; rr' = r.r; mu = rr'/rr;
// p = r + mu p; rr = rr'; break if rr < tol (latched per agent).   update_utils.py:11-22
__global__ void k_cg_step(KCtx c, FvpWs f, float tol) {
  __shared__ float sh[32];
  const int agent = blockIdx.x;
  if (f.sc[agent * 8 + 1] == 0.f) return;
  const long long o = (long long)agent * c.L.na_stride;
  const float rr = f.sc[agent * 8 + 0];
  float acc = 0.f;
  for (long long i = threadIdx.x; i < c.L.na; i += blockDim.x) acc += f.p[o + i] * f.z[o + i];
  const float pz = block_sum(acc, sh);
  const float v = rr / pz;
  acc = 0.f;
  for (long long i = threadIdx.x; i < c.L.na; i += blockDim.x) {
    f.x[o + i] += v * f.p[o + i];
    const float rn = f.r[o + i] - v * f.z[o + i];
    f.r[o + i] = rn;
    acc += rn * rn;
  }
  const float rr2 = block_sum(acc, sh);
  const float mu = rr2 / rr;
  for (long long i = threadIdx.x; i < c.L.na; i += blockDim.x) f.p[o + i] = f.r[o + i] + mu * f.p[o + i];
  if (threadIdx.x == 0) {
    f.sc[agent * 8 + 0] = rr2;
    if (rr2 < tol) f.sc[agent * 8 + 1] = 0.f;
  }
}

// vFv = x . F(x)   (trpo.py:185)
__global__ void k_cg_vfv(KCtx c, FvpWs f, float* __restrict__ vfv) {
  __shared__ float sh[32];
  const int agent = blockIdx.x;
  const long long o = (long long)agent * c.L.na_stride;
  float acc = 0.f;
  for (long long i = threadIdx.x; i < c.L.na; i += blockDim.x) acc += f.x[o + i] * f.z[o + i];
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) vfv[agent] = acc;
}

}  // namespace saceo
