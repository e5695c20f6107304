// hrl_normalize.cuh - running observation statistics and return-based reward scaling (hrl_obs_moments, hrl_reward_scale;
// DESIGN.md section 4, kernel 8).  SB3 VecNormalize's statistics, on the device, in float64, without atomics.
//
// Both reductions over a batch run in ONE thread-block cluster (16 CTAs of 1024 threads, 8 where the device cannot
// co-schedule 16; hrl_b200.cu norm_cluster_size): the CTAs reduce
// their share of the batch and CTA 0 merges the CTA partials through distributed shared memory in rank order.  So no
// scratch memory outside the cluster is needed (the calls are reentrant: concurrent calls on other streams share nothing),
// and the order of every merge is fixed: the same inputs give the same bytes on every call.
//
// Partials are (n, mean, M2).  Inside a thread the data are summed as deviations from a sample of the same data (the
// thread's first value): s1 = sum (x - K), s2 = sum (x - K)^2, then mean = K + s1 / n, M2 = s2 - s1^2 / n.  K lies inside
// the data, so s2 and s1^2 / n do not cancel the way raw sums of squares do (a column with mean 1e3 and std 1e-2 keeps its
// digits).  Above the thread, partials merge with Chan's rule:
//   n = na + nb,  d = mb - ma,  mean = ma + d nb / n,  M2 = M2a + M2b + d^2 na nb / n.
#pragma once
#include <cooperative_groups.h>
#include "hrl_math.cuh"

#define HRL_NORM_THREADS 1024
#define HRL_NORM_MAX_D 64
#define HRL_NORM_U 16  // loads in flight per thread in the reductions (the cluster has few SMs: latency bounds them)

struct Moments {
  double n, m, M2;
};

__device__ __forceinline__ void chan_merge(Moments& a, const Moments& b) {
  if (b.n == 0.0) return;
  if (a.n == 0.0) { a = b; return; }
  const double n = a.n + b.n, d = b.m - a.m;
  a.m = a.m + d * (b.n / n);
  a.M2 = a.M2 + b.M2 + d * d * (a.n * b.n / n);
  a.n = n;
}

// SB3 RunningMeanStd.update_from_moments on {count, mean, var} with a batch (bm, bv, bc), in numpy's order of operations
__device__ __forceinline__ void sb3_merge(double& count, double& mean, double& var, double bm, double bv, double bc) {
  const double delta = __dsub_rn(bm, mean), tot = __dadd_rn(count, bc);
  const double new_mean = __dadd_rn(mean, __ddiv_rn(__dmul_rn(delta, bc), tot));
  const double m2 = __dadd_rn(__dadd_rn(__dmul_rn(var, count), __dmul_rn(bv, bc)),
                              __ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(delta, delta), count), bc), tot));
  mean = new_mean;
  var = __ddiv_rn(m2, tot);
  count = tot;
}

__device__ __forceinline__ Moments shifted_to_moments(double n, double K, double s1, double s2) {
  Moments p;
  p.n = n;
  p.m = n > 0.0 ? K + s1 / n : 0.0;
  p.M2 = n > 0.0 ? fmax(s2 - s1 * s1 / n, 0.0) : 0.0;
  return p;
}

// ---- hrl_obs_moments: x f32[M, D] merged into mom f64[1 + 2D] = {count, mean[D], var[D]} ----------------------------
// CTA c of the cluster owns rows [c M / C, (c + 1) M / C).  Thread t < R D (R = 1024 / D rows per sweep) owns column t % D
// and rows r0 + t / D, r0 + t / D + R, ...: a sweep reads R D consecutive floats (coalesced).  The R partials of a column
// merge in a fixed tree in shared memory, then CTA 0 merges the C CTA partials in rank order.
__global__ void __launch_bounds__(HRL_NORM_THREADS)
obs_moments_kernel(int M, int D, const float* __restrict__ x, double* __restrict__ mom, float eps, float* __restrict__ mean_f,
                   float* __restrict__ rstd_f) {
  namespace cg = cooperative_groups;
  cg::cluster_group cl = cg::this_cluster();
  __shared__ Moments part[HRL_NORM_THREADS];
  const int C = (int)cl.num_blocks(), c = (int)cl.block_rank(), t = threadIdx.x;
  const int R = HRL_NORM_THREADS / D, col = t % D, sub = t / D;
  const size_t r0 = (size_t)M * c / C, r1 = (size_t)M * (c + 1) / C;
  Moments p = {0.0, 0.0, 0.0};
  if (sub < R) {
    double n = 0.0, K = 0.0, s1 = 0.0, s2 = 0.0;
    size_t r = r0 + sub;
    const size_t step = (size_t)R * D;
    const float* px = x + r * D + col;
    if (r < r1) K = (double)*px;
    // HRL_NORM_U loads issued together: one memory round trip per HRL_NORM_U rows, not per row
    for (; r + (size_t)(HRL_NORM_U - 1) * R < r1; r += (size_t)HRL_NORM_U * R, px += HRL_NORM_U * step) {
      float v[HRL_NORM_U];
#pragma unroll
      for (int u = 0; u < HRL_NORM_U; u++) v[u] = __ldg(px + u * step);
#pragma unroll
      for (int u = 0; u < HRL_NORM_U; u++) {
        const double d = (double)v[u] - K;
        s1 += d;
        s2 = fma(d, d, s2);
      }
      n += (double)HRL_NORM_U;
    }
    for (; r < r1; r += R, px += step) {
      const double d = (double)*px - K;
      s1 += d;
      s2 = fma(d, d, s2);
      n += 1.0;
    }
    p = shifted_to_moments(n, K, s1, s2);
  }
  part[t] = p;
  __syncthreads();
  for (int s = 1; s < R; s *= 2) {  // sub-row r takes r + s for r % 2s == 0: a fixed tree
    if (sub < R && sub % (2 * s) == 0 && sub + s < R) chan_merge(part[t], part[t + s * D]);
    __syncthreads();
  }
  cl.sync();  // every CTA's column partials (part[0 .. D)) are final
  if (c == 0 && t < D) {
    Moments b = part[t];
    for (int k = 1; k < C; k++) chan_merge(b, *cl.map_shared_rank(&part[t], k));
    double count = mom[0], mean = mom[1 + t], var = mom[1 + D + t];
    sb3_merge(count, mean, var, b.m, b.M2 / b.n, b.n);
    mom[1 + t] = mean;
    mom[1 + D + t] = var;
    mean_f[t] = (float)mean;
    rstd_f[t] = (float)(1.0 / sqrt(var + (double)eps));
  }
  cl.sync();  // the other CTAs keep their shared memory until CTA 0 has read it, and every column has read the old count
  if (c == 0 && t == 0) mom[0] = __dadd_rn(mom[0], (double)M);
}

// ---- hrl_reward_scale ------------------------------------------------------------------------------------------------
// Launch 1: per-env scan over T, one thread per env (coalesced on [T, N]); R in float64, in numpy's order R gamma + r.
// Writes R rounded to float32 into out and the carry (zeroed where done[T - 1]) into ret.
__global__ void __launch_bounds__(256)
return_scan_kernel(int T, int N, double gamma, const float* __restrict__ rew, const uint8_t* __restrict__ done,
                   double* __restrict__ ret, float* __restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  double R = ret[e];
  for (int t0 = 0; t0 < T; t0 += HRL_NORM_U) {  // the loads of HRL_NORM_U steps are issued together
    float r[HRL_NORM_U];
    bool d[HRL_NORM_U];
#pragma unroll
    for (int u = 0; u < HRL_NORM_U; u++) {
      const size_t i = (size_t)(t0 + u) * N + e;
      r[u] = t0 + u < T ? rew[i] : 0.f;
      d[u] = t0 + u < T && done[i] != 0;
    }
#pragma unroll
    for (int u = 0; u < HRL_NORM_U; u++) {
      if (t0 + u < T) {
        const size_t i = (size_t)(t0 + u) * N + e;
        R = __dadd_rn(__dmul_rn(R, gamma), (double)r[u]);
        out[i] = (float)R;
        if (d[u]) R = 0.0;
      }
    }
  }
  ret[e] = R;
}

// Launch 2 (one cluster): per step t the mean and population variance of R over the N envs, then SB3's chain of merges
// into rm = {count, mean, var} in step order; work[t] = s_t = (float)(1 / sqrt(var + eps)).  CTA c owns envs
// [c N / C, (c + 1) N / C); its 32 warps take 32 steps at a time, warp w step t0 + w, the lanes striding over the envs
// with the CTA's first env as the shift.  CTA 0 merges the CTA partials of each step in rank order, lane l for step t0 + l,
// and lane 0 runs the chain.
__global__ void __launch_bounds__(HRL_NORM_THREADS)
return_moments_kernel(int T, int N, float eps, const float* __restrict__ R, double* __restrict__ rm, double* __restrict__ work) {
  namespace cg = cooperative_groups;
  cg::cluster_group cl = cg::this_cluster();
  __shared__ Moments part[32];
  __shared__ double chain[3];  // CTA 0: {count, mean, var} of the returns, carried across the groups of 32 steps
  const int C = (int)cl.num_blocks(), c = (int)cl.block_rank();
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e0 = (int)((long long)N * c / C), e1 = (int)((long long)N * (c + 1) / C);
  if (c == 0 && threadIdx.x == 0) { chain[0] = rm[0]; chain[1] = rm[1]; chain[2] = rm[2]; }
  for (int t0 = 0; t0 < T; t0 += 32) {
    const int t = t0 + w;
    Moments p = {0.0, 0.0, 0.0};
    if (t < T && e1 > e0) {
      const float* row = R + (size_t)t * N;
      const double K = (double)row[e0];
      double s1 = 0.0, s2 = 0.0;
      int e = e0 + lane;
      for (; e + 32 * (HRL_NORM_U - 1) < e1; e += 32 * HRL_NORM_U) {
        float v[HRL_NORM_U];
#pragma unroll
        for (int u = 0; u < HRL_NORM_U; u++) v[u] = row[e + 32 * u];
#pragma unroll
        for (int u = 0; u < HRL_NORM_U; u++) {
          const double d = (double)v[u] - K;
          s1 += d;
          s2 = fma(d, d, s2);
        }
      }
      for (; e < e1; e += 32) {
        const double d = (double)row[e] - K;
        s1 += d;
        s2 = fma(d, d, s2);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {  // a fixed tree: the same sums on every call
        s1 += __shfl_down_sync(HRL_FULL_MASK, s1, o);
        s2 += __shfl_down_sync(HRL_FULL_MASK, s2, o);
      }
      p = shifted_to_moments((double)(e1 - e0), K, s1, s2);
    }
    if (lane == 0) part[w] = p;
    cl.sync();
    if (c == 0 && w == 0) {
      Moments b = part[lane];
      for (int k = 1; k < C; k++) chan_merge(b, *cl.map_shared_rank(&part[lane], k));
      const double bm = b.m, bv = b.n > 0.0 ? b.M2 / b.n : 0.0;
      double count = chain[0], mean = chain[1], var = chain[2];
      for (int j = 0; j < 32 && t0 + j < T; j++) {
        const double m = __shfl_sync(HRL_FULL_MASK, bm, j), v = __shfl_sync(HRL_FULL_MASK, bv, j);
        sb3_merge(count, mean, var, m, v, (double)N);   // every lane runs the chain; lane 0 writes it
        if (lane == 0) work[t0 + j] = (double)(float)(1.0 / sqrt(var + (double)eps));
      }
      if (lane == 0) { chain[0] = count; chain[1] = mean; chain[2] = var; }
    }
    cl.sync();  // part[] is rewritten by the next 32 steps, and read remotely until here
  }
  if (c == 0 && threadIdx.x == 0) { rm[0] = chain[0]; rm[1] = chain[1]; rm[2] = chain[2]; }
}

// Launch 3: out[t, e] = clamp(rew[t, e] * s_t, -clip, clip) in float32; blockIdx.y strides over t, x over the envs
__global__ void __launch_bounds__(256)
reward_apply_kernel(int T, int N, float clip, const float* __restrict__ rew, const double* __restrict__ work, float* __restrict__ out) {
  for (int t = blockIdx.y; t < T; t += gridDim.y) {
    const float s = (float)work[t];
    const size_t row = (size_t)t * N;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < N; e += gridDim.x * blockDim.x)
      out[row + e] = fminf(fmaxf(__fmul_rn(rew[row + e], s), -clip), clip);
  }
}
