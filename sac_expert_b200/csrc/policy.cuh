// Acting for a set of P independent policies of any depth (saceo_policy_act): an expert policy is only ever rolled out
// (SAC_exp._collect_expert_data, sac_eo/algs/SAC_expert.py:156-209), so it needs a forward pass and the reference's two
// policy heads, not the two-hidden-layer training engine.
//
//   x = (s - s_mean) / max(s_std, 1e-8)                                  RunningNormalizer.normalize (normalizer.py:26-41)
//   h_l = act_l(h_{l-1} . W_l + b_l),  l < n_hidden;  out = h . W_n + b_n     Keras Sequential of Dense (nn_utils.py:86-138)
//   squash = 0  GaussianActor._forward + .sample (continuous_actors.py:74-123): logstd = log(softplus(out[A:])) + log(std_mult)
//               - log(log 2) (per-state std) or logstd_var + log(std_mult); logstd = max(logstd, log 1e-3);
//               a = mean (+ exp(logstd) u)
//   squash = 1  SquashedGaussianActor.sample (:270-306): logstd clipped to [-5, 2]; z = mean (+ exp(logstd) u);
//               a = act_limit tanh(z)
//
// Exact fp32 on CUDA cores: every output is one thread's FMA chain over k = 0 .. in-1 in order, then + bias (the order of
// k_gemm_simt), so a policy's actions do not depend on the grid, on the row tile or on the other policies of the set.
// One launch per call: grid (row tiles, P), activations ping-pong between two shared-memory buffers of `ld` floats per
// row.  Weights are read along output columns (coalesced), 16 bytes at a time when the layer's offset and width allow.
#pragma once
#include "elem.cuh"

namespace saceo {

constexpr int POL_MAX_HIDDEN = SACEO_POLICY_MAX_HIDDEN;
constexpr int POL_MAX_WIDTH = 1024;
constexpr int POL_THREADS = 256;
constexpr int POL_RB = 4;           // rows per thread item (a 4 x 4 register tile of outputs)

struct PolicyP {
  const float* params; const float* norm; const float* obs; const float* noise; float* out;
  long long pstride;                // floats per policy in params
  int nstride;                      // floats per policy in norm: s_mean(S) | s_std(S) | act_limit(A)
  int rows, rt, ld;                 // rows per policy, rows per tile (multiple of POL_RB), shared row stride (floats)
  int S, A, Ao, nl;                 // nl = n_hidden + 1 dense layers
  int width[POL_MAX_HIDDEN + 2];    // width[0] = S, width[l + 1] = output width of layer l
  int act[POL_MAX_HIDDEN + 1];      // ACT_* per layer, ACT_LINEAR for the output layer
  long long off[POL_MAX_HIDDEN + 2];  // offset of W_l in the flat layout; off[nl] = logstd variable
  int squash, per_state_std;
  float ls_add;                     // log(std_mult) (- log(log 2) with per-state std)
};

// One dense layer for the rows of a tile: dst[r][n] = act(sum_k src[r][k] W[k][n] + b[n]).
// A thread item is (4-row block, 4 consecutive columns): 16 independent FMA chains, one 16-byte weight load per k when
// VEC (width and offset multiples of 4), four coalesced scalar loads otherwise.
template <bool VEC>
__device__ __forceinline__ void pol_layer(const float* __restrict__ W, const float* __restrict__ b, int in, int outw,
                                          int act, const float* src, float* dst, int ld, int nrb) {
  const int groups = (outw + 3) >> 2;
  for (int item = threadIdx.x; item < groups * nrb; item += blockDim.x) {
    const int g = item % groups, rb = item / groups;
    const int n0 = g * 4;
    const float* s0 = src + (rb * POL_RB) * ld;
    float acc[POL_RB][4];
#pragma unroll
    for (int r = 0; r < POL_RB; ++r)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[r][j] = 0.f;
#pragma unroll 4
    for (int k = 0; k < in; ++k) {
      float w[4];
      if (VEC) {
        const float4 w4 = __ldg(reinterpret_cast<const float4*>(W + (long long)k * outw + n0));
        w[0] = w4.x; w[1] = w4.y; w[2] = w4.z; w[3] = w4.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) w[j] = n0 + j < outw ? __ldg(W + (long long)k * outw + n0 + j) : 0.f;
      }
#pragma unroll
      for (int r = 0; r < POL_RB; ++r) {
        const float h = s0[r * ld + k];
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[r][j] = fmaf(h, w[j], acc[r][j]);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (n0 + j >= outw) continue;
      const float bj = __ldg(b + n0 + j);
#pragma unroll
      for (int r = 0; r < POL_RB; ++r) dst[(rb * POL_RB + r) * ld + n0 + j] = apply_act(act, acc[r][j] + bj);
    }
  }
}

// grid (ceil(rows / rt), P), block POL_THREADS, dynamic shared memory 2 * rt * ld floats
__global__ void __launch_bounds__(POL_THREADS, 4) k_policy_forward(PolicyP p) {
  extern __shared__ __align__(16) float pol_sm[];
  const int pol = blockIdx.y;
  const int r0 = blockIdx.x * p.rt;
  const int nr = min(p.rt, p.rows - r0);
  const int nrb = (nr + POL_RB - 1) / POL_RB;
  const float* theta = p.params + (long long)pol * p.pstride;
  const float* nrm = p.norm + (long long)pol * p.nstride;
  const int half = p.rt * p.ld;         // buffer b starts at pol_sm + b * half

  // stage the normalised observations; rows past the end of the tile are zero (computed, never stored)
  const float* obs = p.obs + ((long long)pol * p.rows + r0) * p.S;
  for (int e = threadIdx.x; e < nrb * POL_RB * p.S; e += blockDim.x) {
    const int r = e / p.S, j = e - r * p.S;
    pol_sm[r * p.ld + j] = r < nr ? (obs[(long long)r * p.S + j] - nrm[j]) / nstd(nrm[p.S + j]) : 0.f;
  }
  __syncthreads();

  int cur = 0;
  for (int l = 0; l < p.nl; ++l) {
    const int in = p.width[l], outw = p.width[l + 1];
    const float* W = theta + p.off[l];
    const float* b = W + (long long)in * outw;
    if (((outw | (int)(p.off[l] & 3)) & 3) == 0) pol_layer<true>(W, b, in, outw, p.act[l], pol_sm + cur * half, pol_sm + (cur ^ 1) * half, p.ld, nrb);
    else pol_layer<false>(W, b, in, outw, p.act[l], pol_sm + cur * half, pol_sm + (cur ^ 1) * half, p.ld, nrb);
    cur ^= 1;
    __syncthreads();
  }

  // head: one thread per (row, action dimension)
  const float* o = pol_sm + cur * half;
  const int A = p.A;
  const float* lsv = theta + p.off[p.nl];
  for (int e = threadIdx.x; e < nr * A; e += blockDim.x) {
    const int r = e / A, j = e - r * A;
    const long long g = ((long long)pol * p.rows + r0 + r) * A + j;
    const float mean = o[r * p.ld + j];
    float ls = p.per_state_std ? o[r * p.ld + A + j] : __ldg(lsv + j);
    float a;
    if (p.squash) {
      ls = fminf(fmaxf(ls, kMinLogStd), kMaxLogStd);
      const float sd = expf(ls);
      const float z = p.noise ? mean + sd * p.noise[g] : mean;
      a = nrm[2 * p.S + j] * tanhf(z);
    } else {
      ls = (p.per_state_std ? logf(softplusf(ls)) : ls) + p.ls_add;
      ls = fmaxf(ls, logf(1e-3f));
      a = p.noise ? mean + expf(ls) * p.noise[g] : mean;
    }
    p.out[g] = a;
  }
}

}  // namespace saceo
