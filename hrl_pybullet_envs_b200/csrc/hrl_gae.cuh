// hrl_gae.cuh - GAE(lambda) advantages and returns over a [T, N] rollout buffer (hrl_gae; DESIGN.md section 4, kernel 7).
//
// Backwards in time the recurrence is an affine map per env:  A_t = delta_t + c_t A_{t+1},  c_t = gamma lam (1 - done_t),
// A_T = 0.  Maps compose associatively, (c1, d1) o (c2, d2) = (c1 c2, d1 + c1 d2), so T is split as well as N:
// a CTA owns 32 consecutive envs (one per lane: every access to a time slice [t, e0 : e0 + 32] is one coalesced 128-byte
// line in the [T, N] layout) and its W warps own W contiguous chunks of T.
//   pass 1  each lane runs its chunk backwards and composes the chunk's map (C, D), writing delta_t to adv; the chunk that
//           ends at T starts from A_T = 0, so its D already is A_t and it writes the final adv / ret right away;
//   combine the W maps of each env meet in shared memory, and each chunk applies the maps of the chunks after it to A_T = 0;
//   pass 2  the other chunks run again from that A, reading delta_t back from adv, and write adv and ret.
// Every choice between a value and a value not meant to be used is a select: a NaN in a row that is not selected (a stale
// terminal-value row, the value after a termination, the A of the next episode) is never an operand.
#pragma once
#include "hrl_math.cuh"

#define HRL_GAE_MAX_WARPS 16    // chunks of T per env = warps per CTA
#define HRL_GAE_MIN_CHUNK 8     // no split below 8 steps per chunk: pass 2 and the combine would cost more than they hide
#define HRL_GAE_WARPS_PER_SM 16 // resident warps per SM at which the launch is wide enough without splitting T

// warps per CTA for T steps of N envs on `sms` SMs: split T (powers of two) until the grid holds HRL_GAE_WARPS_PER_SM warps
// per SM, while every chunk keeps at least HRL_GAE_MIN_CHUNK steps.  W = 1 whenever the envs alone fill the machine.
static inline int gae_warps(int T, int N, int sms) {
  const long long G = (N + 31) / 32;
  int W = 1;
  while (W < HRL_GAE_MAX_WARPS && G * W < (long long)sms * HRL_GAE_WARPS_PER_SM && T >= 2 * W * HRL_GAE_MIN_CHUNK) W *= 2;
  return W;
}

#define HRL_GAE_U 8             // steps whose loads are issued together: one memory round trip per 8 steps, not per step

// L = ceil(T / W) steps per chunk; info / tval both NULL (every done terminates) or both non-NULL; ret may be NULL
__global__ void __launch_bounds__(32 * HRL_GAE_MAX_WARPS)
gae_kernel(int T, int N, int L, float gamma, float gl, const float* __restrict__ rew, const uint8_t* __restrict__ done,
           const float* __restrict__ info, const float* __restrict__ values, const float* __restrict__ tval,
           float* __restrict__ adv, float* __restrict__ ret) {
  __shared__ float2 chunk_map[HRL_GAE_MAX_WARPS][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, W = blockDim.x >> 5;
  const int e = blockIdx.x * 32 + lane;
  const bool ok = e < N;
  const int t0 = min(w * L, T), t1 = min(t0 + L, T);
  HRL_CHECK(w < HRL_GAE_MAX_WARPS && W <= HRL_GAE_MAX_WARPS && t0 <= t1 && t1 <= T);
  const bool last = t1 == T;  // A_{t1} = A_T = 0 is known: pass 1 writes the results (a chunk past T is empty)
  const size_t n = (size_t)N;
  float C = 1.f, D = 0.f;     // the chunk's map A_{t0} = D + C A_{t1}
  if (ok && t0 < t1) {
    float vnext = values[(size_t)t1 * n + e];
    for (int tg = t1; tg > t0; tg -= HRL_GAE_U) {  // steps tg - 1, tg - 2, ... of this group, j = 0 first
      const int nt = min(HRL_GAE_U, tg - t0);
      float r[HRL_GAE_U], v[HRL_GAE_U], tv[HRL_GAE_U];
      bool d[HRL_GAE_U], tr[HRL_GAE_U];
#pragma unroll
      for (int j = 0; j < HRL_GAE_U; j++) {
        const size_t i = (size_t)(tg - 1 - j) * n + e;
        d[j] = j < nt && done[i] != 0;
        r[j] = j < nt ? rew[i] : 0.f;
        v[j] = j < nt ? values[i] : 0.f;
      }
#pragma unroll
      for (int j = 0; j < HRL_GAE_U; j++) {  // the flag and the terminal value are read only where a done can select them
        const size_t i = (size_t)(tg - 1 - j) * n + e;
        tr[j] = tval && d[j] && ((int)info[4 * i + 2] & 1);
        tv[j] = tval && d[j] ? tval[i] : 0.f;
      }
#pragma unroll
      for (int j = 0; j < HRL_GAE_U; j++) {
        if (j < nt) {
          const size_t i = (size_t)(tg - 1 - j) * n + e;
          const float next = d[j] ? (tr[j] ? tv[j] : 0.f) : vnext;
          const float delta = fmaf(gamma, next, r[j]) - v[j];
          D = d[j] ? delta : fmaf(gl, D, delta);
          C = d[j] ? 0.f : gl * C;
          adv[i] = last ? D : delta;
          if (last && ret) ret[i] = D + v[j];
          vnext = v[j];
        }
      }
    }
  }
  chunk_map[w][lane] = make_float2(C, D);
  __syncthreads();
  if (!ok || last) return;
  float A = 0.f;  // A_{t1}: the maps of the later chunks applied to A_T = 0
  for (int k = W - 1; k > w; k--) {
    HRL_CHECK(k < HRL_GAE_MAX_WARPS);
    const float2 m = chunk_map[k][lane];
    A = m.x == 0.f ? m.y : fmaf(m.x, A, m.y);
  }
  for (int tg = t1; tg > t0; tg -= HRL_GAE_U) {
    const int nt = min(HRL_GAE_U, tg - t0);
    float dl[HRL_GAE_U], v[HRL_GAE_U];
    bool d[HRL_GAE_U];
#pragma unroll
    for (int j = 0; j < HRL_GAE_U; j++) {
      const size_t i = (size_t)(tg - 1 - j) * n + e;
      d[j] = j < nt && done[i] != 0;
      dl[j] = j < nt ? adv[i] : 0.f;
      v[j] = j < nt && ret ? values[i] : 0.f;
    }
#pragma unroll
    for (int j = 0; j < HRL_GAE_U; j++) {
      if (j < nt) {
        const size_t i = (size_t)(tg - 1 - j) * n + e;
        A = d[j] ? dl[j] : fmaf(gl, A, dl[j]);
        adv[i] = A;
        if (ret) ret[i] = A + v[j];
      }
    }
  }
}
