// hrl_b200.cu - fused env-step kernels (sm_100a) and the C-ABI of include/hrl_b200.h.
//
// Layout: one 4-lane group per env (lane = leg), 8 envs per warp, one warp per CTA by default so
// that 4096 envs become 512 CTAs spread over the 148 SMs x 4 schedulers.  Per-warp shared memory
// (37.4 KB) holds the whitened constraint rows of the sub-step + impulses, the contact candidates and
// the cube-collider scratch; after the last sub-step the row buffer is reused for the sensor bins and
// the observation staging tile, which is written back with fully coalesced float4 stores.
// No CPU fallback: every entry point fails with HRL_E_CUDA when no device / kernel is available.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <utility>

#include "../../include/hrl_b200.h"
#include "hrl_ant.cuh"
#include "hrl_ant_wide.cuh"
#include "hrl_gae.cuh"
#include "hrl_math.cuh"
#include "hrl_normalize.cuh"
#include "hrl_sensors.cuh"

#ifndef HRL_WARPS_PER_CTA
#define HRL_WARPS_PER_CTA 1
#endif
#define HRL_OBS_STAGE 64  // floats per env in the staging tile = the widest observation hrl_create accepts

// ------------------------------------------------------------------------------------------
// device state (internal SoA layout; the public layout of hrl_get_state is converted by kernels)
// ------------------------------------------------------------------------------------------
struct DevState {
  float4* base;   // [N][4]: (pos.xyz, initial_z) (quat xyzw) (vel.xyz, potential) (ang.xyz, wtd)
  float4* leg;    // [N][4 legs]: (q_hip, q_ankle, qd_hip, qd_ankle)
  float4* items;  // [N][4 lanes][2]: items 4k..4k+3 as (x0,y0,x1,y1)(x2,y2,x3,y3)
  float4* miscf;  // [N][2]: (target.x, target.y, running return, sum of finished returns) (feet0..3)
  int4* misci;    // [N][2]: (t, episode, steps_total, goals_left) (since, rewarded, -, -)
  unsigned long long* stats;  // [4]: contacts, limit rows, env-substeps, non-finite resets
  // completion signal of the zero-copy host path: the last CTA to finish writes fin_seq to the
  // pinned host word fin_flag (NULL: no signalling), so the host can poll instead of paying a
  // driver-level stream synchronisation
  unsigned int* fin_count;
  unsigned int* fin_flag;
  unsigned int fin_seq;
#ifdef HRL_WARP_TIMES
  // profiling build only: per warp (cycles of the launch, cycles of the physics loop, solver trips, task-layer passes)
  unsigned long long* wt;
#endif
};

struct hrl_handle {
  hrl_config cfg;
  int device, N, D, A;
  DevState st;
  float* d_bounds;  // lidar bound lines [7][4]
  int n_lines;
  // staging for hrl_step_host: ONE device block laid out [obs | rew | info | done] so that a host
  // buffer with the same layout (hrl_host_layout) comes back with a single copy
  float *s_act, *s_obs, *s_rew, *s_info;
  uint8_t* s_done;
  size_t s_out_bytes;
  int sub;        // lane mapping of the ant kernels: 1 = 4 lanes per env, 2 = 8, 4 = 16 (hrl_set_lanes_per_env)
  int compact;    // 4-lane mapping with compact solver rows (7 CTAs per SM): chosen when that saves a wave of CTAs
  int host_mode;  // HRL_HOST_AUTO / HRL_HOST_COPY / HRL_HOST_ZEROCOPY
  unsigned int* h_flag;  // pinned host word polled by hrl_step_host (zero-copy mode)
  unsigned int seq;
  // small cache of (host pointer -> device alias) so that steady-state steps skip cudaPointerGetAttributes
  const void* alias_key[12];
  void* alias_val[12];
  int alias_n;
};

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

static int set_err(int code, const char* msg) {
  snprintf(g_err, sizeof g_err, "%s", msg);
  return code;
}
static int set_err(int code, const char* fn, const char* msg) {  // "fn: msg"
  snprintf(g_err, sizeof g_err, "%s: %s", fn, msg);
  return code;
}
static int cuda_fail(cudaError_t e, const char* where) {
  snprintf(g_err, sizeof g_err, "%s: %s", where, cudaGetErrorString(e));
  return HRL_E_CUDA;
}
#define CK(call)                                    \
  do {                                              \
    cudaError_t _e = (call);                        \
    if (_e != cudaSuccess) return cuda_fail(_e, #call); \
  } while (0)

// Every entry point runs on the handle's device and puts the caller's current device back on return (a process that
// drives several GPUs, or PyTorch's own notion of the current device, must not be disturbed by a step on cuda:1).
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) {
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess) { cudaGetLastError(); cur = -1; }
    if (cur != dev) { err = cudaSetDevice(dev); prev = cur; }
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};
#define ON_DEVICE(dev)                                             \
  DeviceGuard _guard(dev);                                         \
  if (_guard.err != cudaSuccess) return cuda_fail(_guard.err, "cudaSetDevice")

// ------------------------------------------------------------------------------------------
// task-layer helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float clip5(float x) { return fminf(fmaxf(x, -5.f), 5.f); }

// Flagrun goal j of episode ep: ant_flagrun_env.py:71-78; the stream is shared by all envs (:39)
// rarely executed: kept out of line so that the hot task-layer code stays compact in the I-cache
// `gen` counts the create_targets() calls of the env (ant_flagrun_env.py:91-96 draws fresh goals from the stream each time)
__device__ __noinline__ void flag_goal(const hrl_config& cfg, int ep, int j, int gen, float& gx, float& gy) {
  const float half = cfg.flag_size * 0.5f;
  for (uint32_t attempt = 0;; attempt++) {
    float u[4];
    rng_u4(cfg.flag_seed, (uint32_t)gen, STREAM_FLAG, attempt, (uint32_t)(ep * 128 + j), u);
    gx = -half + 2.f * half * u[0]; gy = -half + 2.f * half * u[1];
    if (sqrtf(gx * gx + gy * gy) < 0.5f && attempt + 1 < HRL_MAX_PLACE_ATTEMPTS) continue;
    return;
  }
}

// create_close_target (ant_flagrun_env.py:80-89, max_targets <= 0): per-axis offset of magnitude
// U(tol, max_target_dist / 2) with a random sign around the true torso xy, redrawn until strictly inside the world
__device__ __noinline__ void flag_close_target(const hrl_config& cfg, uint32_t genv, int steps_total, int at_reset, float px,
                                               float py, float& gx, float& gy) {
  const float wb = cfg.flag_size * 0.5f, lo = cfg.tol, hi = cfg.flag_max_target_dist * 0.5f;
  float g0 = wb + 1.f, g1 = wb + 1.f;
  bool inside = false;
  for (uint32_t attempt = 0; attempt < HRL_MAX_CLOSE_ATTEMPTS && !inside; attempt++) {
    float u[4];
    rng_u4(cfg.flag_seed, genv, STREAM_FLAG_CLOSE, (uint32_t)steps_total, attempt * 2 + (at_reset ? 1u : 0u), u);
    g0 = (lo + (hi - lo) * u[0]) * (u[2] < 0.5f ? -1.f : 1.f) + px;
    g1 = (lo + (hi - lo) * u[1]) * (u[3] < 0.5f ? -1.f : 1.f) + py;
    inside = -wb < g0 && g0 < wb && -wb < g1 && g1 < wb;
  }
  if (!inside) {  // the reference redraws for ever; after 64 rejected draws the goal is pulled inside the world instead
    const float lim = wb - 1e-3f;
    g0 = fminf(fmaxf(g0, -lim), lim); g1 = fminf(fmaxf(g1, -lim), lim);
  }
  gx = g0; gy = g1;
}

// gather_scene.py:52-62: uniform on the (size-1)^2 square, rejected while closer than `spacing`
// to (ax, ay).  Evaluated in double from 24-bit uniforms and rounded to f32 (bit-identical to the oracle).
__device__ __noinline__ void place_item(const hrl_config& cfg, uint32_t genv, uint32_t stream, uint32_t draw,
                                           int item, float ax, float ay, float& ox, float& oy) {
  const double sx = (double)cfg.world_size[0] - 1.0, sy = (double)cfg.world_size[1] - 1.0;
  for (int attempt = 0;; attempt++) {
    float u[4];
    rng_u4(cfg.seed, genv, stream, draw, (uint32_t)(item * 64 + attempt), u);
    double x = (double)u[0] * sx - sx / 2, y = (double)u[1] * sy - sy / 2;
    double dx = (double)ax - x, dy = (double)ay - y;
    if (sqrt(dx * dx + dy * dy) < (double)cfg.robot_object_spacing && attempt + 1 < HRL_MAX_PLACE_ATTEMPTS) continue;
    ox = (float)x; oy = (float)y;
    return;
  }
}

struct TaskRegs {  // replicated per-env task state held in registers
  float initial_z, potential, wtd, tx, ty;
  float ret, ret_sum;  // episode-return accumulators (HRL_SF_RETURN, HRL_SF_RETURN_SUM)
  float feet[4];
  int t, episode, steps_total, goals_left, since, rewarded, gen;
};

// Flagrun next_target() (ant_flagrun_env.py:112-120): pop the next pre-drawn goal, or draw a close one
// when max_targets <= 0; the potential restarts from the STALE walk_target_dist (quirk Q3).
// false = goal list exhausted (the reference's IndexError -> done).
__device__ __forceinline__ bool flag_next(const hrl_config& cfg, uint32_t genv, TaskRegs& T, float px, float py, int at_reset) {
  float gx, gy;  // out-of-line callees write to locals: T itself must stay in registers
  if (cfg.flag_max_targets < 1) flag_close_target(cfg, genv, T.steps_total, at_reset, px, py, gx, gy);
  else {
    if (T.goals_left <= 0) return false;
    T.goals_left--;
    flag_goal(cfg, T.episode - 1, T.goals_left, T.gen, gx, gy);
  }
  T.tx = gx; T.ty = gy;
  T.rewarded = 0;
  T.potential = -T.wtd / cfg.dt;
  return true;
}

// ------------------------------------------------------------------------------------------
// fused Ant step kernel
//   FAMILY 0: AntGather.  FAMILY 1: walker family (AntMaze, AntFlagrun, AntMj, AntMazeMj).
//   mode 0: full env step (+ auto-reset), mode 1: n_sub physics sub-steps only,
//   mode 2: reset the masked envs and emit their observation, mode 3: observe only.
// ------------------------------------------------------------------------------------------
#define SMEM_PER_WARP_FLOATS (HRL_SMEM_FLOATS_PER_WARP + HRL_ITEM_SCRATCH_FLOATS)
static_assert(HRL_EPW == 8, "the 4-lane mapping fills a warp with 8 envs");

// Lane mapping of the fused kernel.  SUB = lanes per leg: 1 = 4 lanes per env, 8 envs per warp (hrl_ant.cuh);
// 2 / 4 = the wide mappings of hrl_ant_wide.cuh (8 / 16 lanes per env, 4 / 2 envs per warp).
template <int SUB>
struct Map : WideMap<SUB> {
  static constexpr int ROW_F4 = HRLW_ROW_F4, ENV_F4 = HRLW_ENV_F4;
  static constexpr int MIN_CTAS = (SUB == 4 ? 14 : 7) / HRL_WARPS_PER_CTA;  // all 4096 envs resident in one wave
};
template <>
struct Map<0> {  // 4 lanes per env with COMPACT solver rows: 30.1 KB per warp, 7 CTAs per SM (batches larger than one wave)
  static constexpr int LPE = 4, EPW = 8, IPL = 4, ROW_F4 = 3, ENV_F4 = HRL_ENV_F4_COMPACT;
  static constexpr int ROWS_FLOATS = HRL_EPW * HRL_ENV_F4_COMPACT * 4, LAM_FLOATS = HRL_LAM_FLOATS_PER_WARP;
  static constexpr int CAND_FLOATS = HRL_MAXC * HRL_CAND_F * 32, ITEM_FLOATS = HRL_ITEM_SCRATCH_FLOATS;
  static constexpr int SMEM_FLOATS = ROWS_FLOATS + LAM_FLOATS + CAND_FLOATS + ITEM_FLOATS;
  static constexpr int MIN_CTAS = 7 / HRL_WARPS_PER_CTA;
};
template <>
struct Map<1> {
  static constexpr int LPE = 4, EPW = 8, IPL = 4, ROW_F4 = 4, ENV_F4 = HRL_ENV_F4;
  static constexpr int ROWS_FLOATS = HRL_ROWS_FLOATS_PER_WARP, LAM_FLOATS = HRL_LAM_FLOATS_PER_WARP;
  static constexpr int CAND_FLOATS = HRL_MAXC * HRL_CAND_F * 32, ITEM_FLOATS = HRL_ITEM_SCRATCH_FLOATS;
  static constexpr int SMEM_FLOATS = SMEM_PER_WARP_FLOATS;
  static constexpr int MIN_CTAS = 1;
};
template <int SUB>
constexpr bool tiles_fit() { return Map<SUB>::ROWS_FLOATS >= Map<SUB>::EPW * HRL_OBS_STAGE + 2 * Map<SUB>::EPW * 2 * HRL_MAX_BINS; }
static_assert(tiles_fit<0>() && tiles_fit<1>() && tiles_fit<2>() && tiles_fit<4>(), "task-layer tiles must fit in the row buffer");

// ------------------------------------------------------------------------------------------
// fused rollout (SURVEY.md 8f item 4, "policy-inference fusion"): T steps in ONE launch, the actions of every step
// computed in-kernel by a small MLP policy from the observation the previous step left in shared memory
//   a = tanh(W3 tanh(W2 tanh(W1 obs + b1) + b2) + b3) + sigma[c] * N(0, 1)
// weights packed input-major: W1[D][H] b1[H] W2[H][H] b2[H] W3[H][A] b3[A], H = 32 or 64, A = 8 (Ant) or 2 (PointGather).
// The 4 lanes of an env split the hidden units (H / 4 each); lane k ends up with the two actions of ITS leg.
// ------------------------------------------------------------------------------------------
struct RollArgs {
  int T, H;
  const float* w;
  float sigma;            // noise scale of every action component, used when sigma_v is NULL
  const float* sigma_v;   // [A] per-component noise scale, or NULL
  unsigned long long seed;
  float* act_out;  // [T][N][A]
  // ROLL = 2 only: the policy reads clamp((obs - mean) * rstd, -clip, clip) (hrl_rollout_mlp_norm)
  const float* obs_mean;  // [D]
  const float* obs_rstd;  // [D]
  float obs_clip;
  // members (hrl_evaluate_mlp): env e runs the policy at w + (e / m_envs) * nw; a CTA holds envs of one member only
  int m_envs;
  // per-env results over the launch up to the first done (hrl_evaluate_mlp), or NULL: return, length, finished flag
  float* ev_ret;
  int32_t* ev_len;
  uint8_t* ev_fin;
};
enum { STREAM_POLICY = 6 };

// The weights live in shared memory (staged once per launch, shared by the warps of the CTA).  Lane k owns the float4
// groups g = 4 q + k of a layer's H / 4 groups: for a fixed q the 4 lanes of an env read 64 contiguous bytes (no bank
// conflict; the 8 envs of the warp read the same addresses: broadcast).
template <int HQ>
__device__ __forceinline__ void mlp_layer(const float* __restrict__ w, const float* __restrict__ b, int n_in, const float* __restrict__ x,
                                          int k, float* __restrict__ out) {
  constexpr int H = 4 * HQ;
  float acc[HQ];
#pragma unroll
  for (int q = 0; q < HQ / 4; q++) {
    const float4 bv = *reinterpret_cast<const float4*>(b + (4 * q + k) * 4);
    acc[4 * q] = bv.x; acc[4 * q + 1] = bv.y; acc[4 * q + 2] = bv.z; acc[4 * q + 3] = bv.w;
  }
#pragma unroll 4
  for (int j = 0; j < n_in; j++) {
    const float xj = x[j];
#pragma unroll
    for (int q = 0; q < HQ / 4; q++) {
      const float4 wv = *reinterpret_cast<const float4*>(w + j * H + (4 * q + k) * 4);
      acc[4 * q] = fmaf(xj, wv.x, acc[4 * q]); acc[4 * q + 1] = fmaf(xj, wv.y, acc[4 * q + 1]);
      acc[4 * q + 2] = fmaf(xj, wv.z, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(xj, wv.w, acc[4 * q + 3]);
    }
  }
#pragma unroll
  for (int q = 0; q < HQ / 4; q++)
    *reinterpret_cast<float4*>(out + (4 * q + k) * 4) = make_float4(tanhf(acc[4 * q]), tanhf(acc[4 * q + 1]), tanhf(acc[4 * q + 2]), tanhf(acc[4 * q + 3]));
}
// w: the packed weights in shared memory; obs: this env's staged observation, scratch: 2 x 64 floats of this env (shared memory)
template <int HQ>
__device__ __forceinline__ float2 mlp_policy(const float* __restrict__ w, int D, const float* __restrict__ obs, float* __restrict__ scratch, int k) {
  constexpr int H = 4 * HQ;
  const float* w1 = w, *b1 = w1 + D * H, *w2 = b1 + H, *b2 = w2 + H * H, *w3 = b2 + H, *b3 = w3 + H * 8;
  mlp_layer<HQ>(w1, b1, D, obs, k, scratch);
  __syncwarp();
  mlp_layer<HQ>(w2, b2, H, scratch, k, scratch + 64);
  __syncwarp();
  float2 o = *reinterpret_cast<const float2*>(b3 + 2 * k);
#pragma unroll 8
  for (int j = 0; j < H; j++) {
    const float xj = scratch[64 + j];
    const float2 wv = *reinterpret_cast<const float2*>(w3 + j * 8 + 2 * k);
    o.x = fmaf(xj, wv.x, o.x); o.y = fmaf(xj, wv.y, o.y);
  }
  __syncwarp();
  return make_float2(tanhf(o.x), tanhf(o.y));
}
// Normalized policy input of obs component i: subtract, multiply, clamp, each rounded on its own (no FMA can form), so
// torch.clamp((obs - mean) * rstd, -clip, clip) gives the same bits.  stat: mean[D] then rstd[D], staged in shared memory.
__device__ __forceinline__ float norm_obs(float o, const float* __restrict__ stat, int D, int i, float clip) {
  return fminf(fmaxf(__fmul_rn(__fsub_rn(o, stat[i]), stat[D + i]), -clip), clip);
}
#define HRL_ROLL_WARPS 2                       // warps per CTA of the fused-rollout instantiations (they share the weights)
#define HRL_MLP_MAX_FLOATS (HRL_OBS_STAGE * 64 + 64 + 64 * 64 + 64 + 64 * 8 + 8)   // obs_dim <= HRL_OBS_STAGE, H <= 64

#ifdef HRL_DEBUG_CONTACTS
__device__ float* g_dbg_contacts = nullptr;  // [N][4 legs][40]: candidate lists of the first sub-step of the last launch
#endif

// ROLL = 1: the fused rollout; ROLL = 2: the same with a normalized policy input (hrl_rollout_mlp_norm)
template <int FAMILY, int SUB, int ROLL = 0>
__global__ void __launch_bounds__(32 * (ROLL ? HRL_ROLL_WARPS : HRL_WARPS_PER_CTA), ROLL ? 2 : Map<SUB>::MIN_CTAS)
ant_env_kernel(const __grid_constant__ hrl_config cfg, DevState st, const float* __restrict__ bounds_g, int n_lines,
               const float* __restrict__ actions, const uint8_t* __restrict__ mask, float* __restrict__ obs_out_g,
               float* __restrict__ rew_out_g, uint8_t* __restrict__ done_out_g, float* __restrict__ info_out_g,
               float* __restrict__ term_out_g, int mode_g, int n_sub, int D, RollArgs ra = RollArgs()) {
  extern __shared__ __align__(16) float smem[];
  typedef Map<SUB> M;
  constexpr int LPE = M::LPE, EPW = M::EPW, IPL = M::IPL;
  // l: lane within the env, k: leg, sub: sub-lane of the leg (wide mappings), ew = es: env slot in the warp
  constexpr int WPC = ROLL ? HRL_ROLL_WARPS : HRL_WARPS_PER_CTA;   // warps per CTA
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, l = lane & (LPE - 1), k = l & 3, sub = l >> 2, ew = lane / LPE, es = ew;
  float* rows = smem + warp * M::SMEM_FLOATS;
  const float* wsm = smem + WPC * M::SMEM_FLOATS;   // ROLL: the policy weights, behind the warps' own regions
  // ROLL = 2: the observation statistics (mean[D], rstd[D]) behind the weights
  const float* nstat = wsm + (ROLL == 2 ? D * ra.H + ra.H + ra.H * ra.H + ra.H + ra.H * 8 + 8 : 0);
  if (ROLL) {
    const int nw = D * ra.H + ra.H + ra.H * ra.H + ra.H + ra.H * 8 + 8;
    const float* wg = ra.w + (size_t)((int)blockIdx.x * WPC * EPW / ra.m_envs) * nw;   // this CTA's member
    for (int i = threadIdx.x; i < nw; i += 32 * WPC) const_cast<float*>(wsm)[i] = __ldg(wg + i);
    if (ROLL == 2)
      for (int i = threadIdx.x; i < 2 * D; i += 32 * WPC) const_cast<float*>(nstat)[i] = __ldg(i < D ? ra.obs_mean + i : ra.obs_rstd + (i - D));
    __syncthreads();
  }
  float* cands = rows + M::ROWS_FLOATS + M::LAM_FLOATS;
  HRL_CHECK(D > 0 && D <= HRL_OBS_STAGE && n_lines >= 0 && 4 * n_lines <= 32 && cfg.n_bins <= HRL_MAX_BINS && cfg.n_food + cfg.n_poison <= 16);
  // the task layer runs after the last sub-step, when the solver rows are dead: its observation staging tile and
  // the sensor bins alias the row buffer (keeps a warp at < 37.8 KB so that 6 CTAs fit an SM at large batch sizes)
  float* sobs = rows;                                                                   // [EPW][HRL_OBS_STAGE]
  unsigned long long* sbins = (unsigned long long*)(rows + EPW * HRL_OBS_STAGE);   // [EPW][2][HRL_MAX_BINS]
  float* iscr = cands + M::CAND_FLOATS;  // cube-collider scratch: lives across the sub-steps
  const int N = cfg.num_envs, kind = cfg.env_kind;
  const int env0 = (blockIdx.x * WPC + warp) * EPW;  // first env of this warp
  const int env_raw = env0 + ew;
  const bool active = env_raw < N;
  // the lane groups of a ragged tail shadow the last env (same trip counts, stores suppressed)
  const int e = active ? env_raw : N - 1;
  const uint32_t genv = (uint32_t)(cfg.env_index_offset + e);
  const LegConst lc = leg_const(k);

#ifdef HRL_WARP_TIMES
  const long long wt_t0 = clock64();
  long long wt_t1 = wt_t0;
  int wt_trips = 0, wt_passes = 0, wt_resets = 0;
#endif
  // ---- load ----
  AntLane s;
  TaskRegs T;
  {
    const float4 b0 = st.base[e * 4 + 0], b1 = st.base[e * 4 + 1], b2 = st.base[e * 4 + 2], b3 = st.base[e * 4 + 3];
    const float4 lg = st.leg[e * 4 + k];
    const float4 m0 = st.miscf[e * 2 + 0], m1 = st.miscf[e * 2 + 1];
    const int4 i0 = st.misci[e * 2 + 0], i1 = st.misci[e * 2 + 1];
    s.O = mk(b0.x, b0.y, b0.z); T.initial_z = b0.w;
    s.qx = b1.x; s.qy = b1.y; s.qz = b1.z; s.qw = b1.w;
    s.v = mk(b2.x, b2.y, b2.z); T.potential = b2.w;
    s.w = mk(b3.x, b3.y, b3.z); T.wtd = b3.w;
    s.q1 = lg.x; s.q2 = lg.y; s.qd1 = lg.z; s.qd2 = lg.w;
    T.tx = m0.x; T.ty = m0.y; T.ret = m0.z; T.ret_sum = m0.w;
    T.feet[0] = m1.x; T.feet[1] = m1.y; T.feet[2] = m1.z; T.feet[3] = m1.w;
    T.t = i0.x; T.episode = i0.y; T.steps_total = i0.z; T.goals_left = i0.w; T.since = i1.x; T.rewarded = i1.y; T.gen = i1.z;
  }
  // ROLL: the launch's first episode - its return (rewards added in step order) and length ev_n while it runs, ~length
  // once a done has ended it (one register for the length and the flag)
  float ev_ret = 0.f;
  int ev_n = 0;
  float it_x[IPL], it_y[IPL];  // this lane's items IPL * l .. IPL * l + IPL - 1 (food 0-7, poison 8-15)
  if (FAMILY == 0) {
    if (IPL == 4) {
      const float4 a = st.items[(e * 4 + l) * 2 + 0], b = st.items[(e * 4 + l) * 2 + 1];
      it_x[0] = a.x; it_y[0] = a.y; it_x[1] = a.z; it_y[1] = a.w; it_x[IPL - 2] = b.x; it_y[IPL - 2] = b.y; it_x[IPL - 1] = b.z; it_y[IPL - 1] = b.w;
    } else if (IPL == 2) {
      const float4 a = st.items[e * 8 + l];
      it_x[0] = a.x; it_y[0] = a.y; it_x[IPL - 1] = a.z; it_y[IPL - 1] = a.w;
    } else {
      const float2 a = reinterpret_cast<const float2*>(st.items)[e * 16 + l];
      it_x[0] = a.x; it_y[0] = a.y;
    }
  }

  // ROLL: step -1 composes the initial observation (what hrl_observe does), steps 0 .. T-1 are full env steps whose
  // actions come from the in-kernel policy; the robot / task state stays in registers in between.  Otherwise ONE pass.
#pragma unroll 1
  for (int step = ROLL ? -1 : 0; step < (ROLL ? ra.T : 1); step++) {
  const int mode = ROLL ? (step < 0 ? 3 : 0) : mode_g;
  // ROLL: every per-step buffer may be NULL (hrl_evaluate_mlp passes none)
  float* __restrict__ obs_out = ROLL && obs_out_g ? obs_out_g + (size_t)(step + 1) * N * D : obs_out_g;
  float* __restrict__ rew_out = ROLL && rew_out_g ? rew_out_g + (size_t)max(step, 0) * N : rew_out_g;
  uint8_t* __restrict__ done_out = ROLL && done_out_g ? done_out_g + (size_t)max(step, 0) * N : done_out_g;
  float* __restrict__ info_out = ROLL && info_out_g ? info_out_g + (size_t)max(step, 0) * N * 4 : info_out_g;
  float* __restrict__ term_out = ROLL && term_out_g ? term_out_g + (size_t)max(step, 0) * N * D : term_out_g;
  const float* __restrict__ bounds = bounds_g;
  // ---- physics ----
  float act1 = 0.f, act2 = 0.f;
  int feet_ground = 0;
  int touch[IPL];
#pragma unroll
  for (int i = 0; i < IPL; i++) touch[i] = 0;
  if (mode <= 1) {
    // idle solver visits read the two all-zero rows HRL_ROW_ZERO, HRL_ROW_ZERO+1 and the idle impulse / mu slots
    // behind the real ones: zero those (2 x 4 float4 per env) and the whole impulse array, nothing else
    for (int i = lane; i < 2 * M::ROW_F4 * EPW; i += 32)
      reinterpret_cast<float4*>(rows)[(i / (2 * M::ROW_F4)) * M::ENV_F4 + HRL_ROW_ZERO * M::ROW_F4 + (i % (2 * M::ROW_F4))] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = lane; i < M::LAM_FLOATS / 4; i += 32)
      reinterpret_cast<float4*>(rows + M::ROWS_FLOATS)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncwarp();
    float2 a;
    if (ROLL) {  // the policy reads the observation the previous pass staged in shared memory (sobs is dense: [EPW][D])
      float* scr = cands + es * 128;
      const float* x = sobs + es * D;
      if (ROLL == 2) {  // normalized input in the scratch's upper half: layer 1 reads it, layer 2 overwrites it; sobs stays raw
        HRL_CHECK(D <= 64 && es >= 0 && es < EPW);
        for (int i = l; i < D; i += LPE) scr[64 + i] = norm_obs(sobs[es * D + i], nstat, D, i, ra.obs_clip);
        __syncwarp();
        x = scr + 64;
      }
      a = ra.H == 64 ? mlp_policy<16>(wsm, D, x, scr, k) : mlp_policy<8>(wsm, D, x, scr, k);
      if (ra.sigma_v || ra.sigma > 0.f) {  // exploration noise: Box-Muller on the counter RNG, keyed by (seed, env), addressed by the env's step count
        const float s1 = ra.sigma_v ? __ldg(ra.sigma_v + 2 * k) : ra.sigma, s2 = ra.sigma_v ? __ldg(ra.sigma_v + 2 * k + 1) : ra.sigma;
        float u[4];
        rng_u4(ra.seed, genv, STREAM_POLICY, (uint32_t)T.steps_total, (uint32_t)k, u);
        const float r0 = sqrtf(-2.f * logf(u[0] + 2.98e-8f));
        float sn, cs;
        sincosf(6.2831853f * u[1], &sn, &cs);
        a.x += s1 * r0 * cs; a.y += s2 * r0 * sn;
      }
      if (active && sub == 0 && ra.act_out) reinterpret_cast<float2*>(ra.act_out)[((size_t)step * N + e) * 4 + k] = a;
    } else {
      a = reinterpret_cast<const float2*>(actions)[e * 4 + k];
    }
    act1 = a.x; act2 = a.y;
    // WalkerBase.apply_action [3P-MEM]: clip to +-1, torque = power * power_coef * a
    const float tau1 = cfg.torque_scale * fminf(fmaxf(act1, -1.f), 1.f);
    const float tau2 = cfg.torque_scale * fminf(fmaxf(act2, -1.f), 1.f);
    const SubstepParams P = make_params(cfg);
    int sc = 0, sl = 0;
    const int ns = mode == 0 ? cfg.substeps : n_sub;
    for (int i = 0; i < ns; i++) {
      const bool on = (i == 0) || !cfg.torque_first_substep_only;
      // cube colliders (FAMILY 0): the contact points of the LAST sub-step are what getContactPoints reports
      // (ant_gather_env.py:114)
      if (SUB <= 1)
        ant_substep<FAMILY == 0, SUB == 0>(s, P, lc, on ? tau1 : 0.f, on ? tau2 : 0.f, rows, cands, lane, k, es, feet_ground, sc, sl, it_x, it_y,
                                 iscr, mode == 0 && i == ns - 1
#if defined(HRL_WARP_TIMES) || defined(HRL_DEBUG_CONTACTS)
#ifdef HRL_WARP_TIMES
                                 , &wt_trips
#else
                                 , nullptr, (g_dbg_contacts && i == 0) ? g_dbg_contacts + (size_t)(e * 4 + k) * 40 : nullptr
#endif
#endif
        );
      else
        ant_substep_w<(SUB > 1 ? SUB : 2), FAMILY == 0>(s, P, lc, on ? tau1 : 0.f, on ? tau2 : 0.f, rows, cands, lane, l, k, sub, es, feet_ground,
                                                        sc, sl, it_x, it_y, iscr, mode == 0 && i == ns - 1
#ifdef HRL_DEBUG_CONTACTS
                                                        , (g_dbg_contacts && i == 0) ? g_dbg_contacts + (size_t)(e * 4 + k) * 40 : nullptr
#endif
        );
    }
    if (FAMILY == 0 && P.item_contacts && mode == 0) {  // this lane's 4 cubes: contact points of the last sub-step
      __syncwarp();
      const unsigned long long* tw = reinterpret_cast<const unsigned long long*>(iscr + EPW * 32) + 2 * es;
#pragma unroll
      for (int i = 0; i < IPL; i++) touch[i] = HRL_TOUCH_GET(tw, IPL * l + i);
      __syncwarp();
    }
    if (st.stats) {  // warp-uniform: inactive tail lanes contribute zeros (never guard a *_sync by `active`)
      const int na = __popc(__ballot_sync(HRL_FULL_MASK, active && l == 0));
      sc = __reduce_add_sync(HRL_FULL_MASK, active ? sc : 0); sl = __reduce_add_sync(HRL_FULL_MASK, active ? sl : 0);
      if (lane == 0) {
        atomicAdd(&st.stats[0], (unsigned long long)sc); atomicAdd(&st.stats[1], (unsigned long long)sl);
        atomicAdd(&st.stats[2], (unsigned long long)(ns * na));
      }
    }
  }

#ifdef HRL_WARP_TIMES
  wt_t1 = clock64();
#endif
  // the lidar's bound lines (<= 7 x 4 floats): fetched once per warp and parked in shared memory (the contact
  // candidates are dead by now) - the ray loop would otherwise wait for a global load per line and ray
  if (FAMILY == 1) {
    const float bv = (lane < 4 * n_lines) ? bounds[lane] : 0.f;
    __syncwarp();
    cands[lane] = bv;
    __syncwarp();
    bounds = cands;
  }

  // ---- task layer: observation / reward / done / reset state machine ----
  // todo: 0 nothing, 1 compose+commit obs, 2 Flagrun reset stage 1 (stale-target calc_state)
  int todo = (mode == 1) ? 0 : 1;
  bool first = (mode == 0);       // first compose of a full step carries the reward logic
  bool set_pot = false;           // potential <- -wtd/dt when the obs is committed (walker reset)
  int done = 0;
  bool pend_reset = false;
  if (mode == 2) {
    const bool m = mask ? (mask[e] != 0) : true;
    todo = m ? 3 : 0;  // 3: reset request
  }

  for (int guard = 0; guard < 6; guard++) {
    // reset requests are executed first (register state only)
    if (todo == 3) {
      T.t = 0; T.ret = 0.f;
      s.O = mk(cfg.start_pos[0], cfg.start_pos[1], cfg.start_pos[2]);
      s.qx = s.qy = s.qz = 0.f; s.qw = 1.f;
      s.v = mk(0.f, 0.f, 0.f); s.w = mk(0.f, 0.f, 0.f);
#pragma unroll
      for (int i = 0; i < 4; i++) T.feet[i] = 0.f;
      {  // WalkerBase.robot_specific_reset: joints ~ U(-0.1, 0.1), zero velocity
        float u[4];
        rng_u4(cfg.seed, genv, STREAM_JOINT, (uint32_t)T.episode, (uint32_t)(k >> 1), u);
        s.q1 = -0.1f + 0.2f * u[(k & 1) * 2]; s.q2 = -0.1f + 0.2f * u[(k & 1) * 2 + 1];
        s.qd1 = 0.f; s.qd2 = 0.f;
      }
      T.initial_z = s.O.z;
      if (FAMILY == 0) {
        // gather_scene.py:38-50: every item re-randomised, avoiding (0,0)
#pragma unroll
        for (int i = 0; i < IPL; i++) {
          const int gi = IPL * l + i;
          if (gi < cfg.n_food + cfg.n_poison) place_item(cfg, genv, STREAM_ITEM_RESET, (uint32_t)T.episode, gi, 0.f, 0.f, it_x[i], it_y[i]);
        }
        T.tx = 0.f; T.ty = 0.f;
        todo = 1;
      } else {
        if (kind == HRL_ANT_MAZE || kind == HRL_ANT_MAZE_MJ) {
          float u[4];
          rng_u4(cfg.seed, genv, STREAM_GOAL, (uint32_t)T.episode, 0u, u);
          int idx = (int)(u[0] * (float)cfg.n_targets);  // rs.randint(0, len(targets)) ant_maze_bullet_env.py:110
          if (idx >= cfg.n_targets) idx = cfg.n_targets - 1;
          T.tx = cfg.targets[idx][0]; T.ty = cfg.targets[idx][1];
        }
        if (kind == HRL_ANT_MJ) { T.tx = 1000.f; T.ty = 0.f; }
        if (kind == HRL_ANT_FLAGRUN) {
          if (T.episode == 0) { T.tx = 1000.f; T.ty = 0.f; }  // WalkerBase default walk target
          T.rewarded = 0;
          // goal generation of the episode: reset() itself draws generation 0; in manual mode nothing is drawn yet, so
          // the caller's first create_targets() (generation += 1) draws what the automatic mode would have drawn
          if (cfg.flag_manual_goals) { T.goals_left = 0; T.gen = -1; set_pot = true; todo = 1; }  // ant_flagrun_env.py:150-153: no goals drawn, target kept
          else { T.goals_left = cfg.flag_max_targets; T.gen = 0; todo = 2; }
        } else { set_pot = true; todo = 1; }
      }
      T.episode++;
    }
    if (!__any_sync(HRL_FULL_MASK, todo != 0)) break;

    // ---------------- calc_state of the current register state ----------------
    float roll, pitch, yaw, cyw, syw;
    quat_to_rpy(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw, cyw, syw);
    const float vbx = cyw * s.v.x + syw * s.v.y, vby = cyw * s.v.y - syw * s.v.x;  // Rz(-yaw) v
    const float o_z = clip5(s.O.z - T.initial_z);
    const float o_v0 = clip5(0.3f * vbx), o_v1 = clip5(0.3f * vby), o_v2 = clip5(0.3f * s.v.z);
    const float o_r = clip5(roll), o_p = clip5(pitch);
    const float mid2 = 0.5f * (lc.lo2 + lc.hi2);
    const float rel1 = 2.f * s.q1 / (ant::HIP_HI - ant::HIP_LO), rel2 = 2.f * (s.q2 - mid2) / (lc.hi2 - lc.lo2);
    const float sp1 = 0.1f * s.qd1, sp2 = 0.1f * s.qd2;
    float wtd_new = 0.f, sin_t = 0.f, cos_t = 1.f;
    if (FAMILY == 1) {
      // body_xyz = mean over the 13 link COMs (+ scene bodies, quirk Q1)
      const LegKin K = leg_fk(s, lc);
      const V3 part = 2.5f * K.rh + 3.f * K.r1 + K.r2;  // (leg + aux + foot COMs) - 3 O
      const float sx = gsum(part.x) + 13.f * s.O.x + cfg.scene_parts_sum[0];
      const float sy = gsum(part.y) + 13.f * s.O.y + cfg.scene_parts_sum[1];
      const float inv_np = 1.0f / (float)(13 + cfg.n_scene_parts);
      const float bx = sx * inv_np, by = sy * inv_np;
      const float dx = T.tx - bx, dy = T.ty - by;
      wtd_new = sqrtf(dx * dx + dy * dy);
      // sin / cos of (atan2(dy, dx) - yaw) by rotating the unit target direction with Rz(-yaw)
      if (wtd_new > 0.f) {
        const float iw = 1.0f / wtd_new;
        cos_t = (dx * cyw + dy * syw) * iw; sin_t = (dy * cyw - dx * syw) * iw;
      } else { cos_t = cyw; sin_t = -syw; }
    }
#ifdef HRL_BOUNDS
    struct ObsRow {  // HRL_BOUNDS builds: every index into the staging row is asserted
      float* p; int n;
      __device__ float& operator[](int i) const { assert(i >= 0 && i < n); return p[i]; }
    };
    const ObsRow so = {sobs + es * D, D};
#else
    float* so = sobs + es * D;  // dense staging: the warp's observations are one contiguous span
#endif
    const bool commit = (todo == 1);
    int fin = 1;       // finite flag (this lane's values)
    int switched = 0;  // Flagrun: the target changed in this step

    if (FAMILY == 0) {
      // ---------------- AntGather: ant_gather_env.py:76-119 ----------------
      float food_rew = 0.f;
      if (first && todo == 1) {
        // pickups in item order; each lane owns 4 items (:86-92, gather_scene.py:95-114)
#pragma unroll
        for (int i = 0; i < IPL; i++) {
          const int gi = IPL * l + i;
          if (gi >= cfg.n_food + cfg.n_poison) continue;
          const double dx = __dsub_rn((double)it_x[i], (double)s.O.x), dy = __dsub_rn((double)it_y[i], (double)s.O.y);
          const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
          if (d2 < (double)cfg.robot_coll_dist) {
            food_rew += (gi < cfg.n_food) ? 1.f : -1.f;
            if (cfg.respawn) place_item(cfg, genv, STREAM_ITEM, (uint32_t)T.steps_total, gi, s.O.x, s.O.y, it_x[i], it_y[i]);
            else { it_x[i] = 100.f; it_y[i] = 0.f; }  // fake_kill_pos gather_scene.py:13
          }
        }
      }
      const bool touch_pickup = first && todo == 1 && !(cfg.robot_coll_dist > 0.f);
      if (touch_pickup) {  // ant_gather_env.py:113-116: one reward_collision per contact POINT of the robot with a cube
#pragma unroll
        for (int i = 0; i < IPL; i++)
          if (IPL * l + i < cfg.n_food + cfg.n_poison) food_rew += (float)touch[i] * ((IPL * l + i < cfg.n_food) ? 1.f : -1.f);
      }
      food_rew = esum<LPE>(food_rew);
      const int nb = cfg.n_bins;
      if (commit) {
        if (l == 0) {
          so[0] = o_z; so[1] = o_v0; so[2] = o_v1; so[3] = o_v2; so[4] = o_r; so[5] = o_p;
          so[22] = T.feet[0]; so[23] = T.feet[1]; so[24] = T.feet[2]; so[25] = T.feet[3];
        }
        if (sub == 0) { so[6 + 4 * k] = clip5(rel1); so[7 + 4 * k] = clip5(sp1); so[8 + 4 * k] = clip5(rel2); so[9 + 4 * k] = clip5(sp2); }
      }
      if (cfg.use_sensor) {
        // sector sensor (:128-177): nearest item wins per bin
        for (int i = lane; i < EPW * 2 * HRL_MAX_BINS; i += 32) sbins[i] = 0x7ff0000000000000ull;
        __syncwarp();
#pragma unroll
        for (int i = 0; i < IPL; i++) {
          const int gi = IPL * l + i;
          if (gi >= cfg.n_food + cfg.n_poison) continue;
          double d2;
          const int b = gather_item_bin(s.O.x, s.O.y, yaw, it_x[i], it_y[i], nb, cfg.sensor_range, cfg.sensor_span, &d2);
          HRL_CHECK(b < nb && nb <= HRL_MAX_BINS);
          if (b >= 0) atomicMin(&sbins[(es * 2 + (gi < cfg.n_food ? 0 : 1)) * HRL_MAX_BINS + b], (unsigned long long)__double_as_longlong(d2));
        }
        __syncwarp();
        if (commit) {
          for (int b = l; b < 2 * nb; b += LPE) {
            const int ty = b / nb, bb = b - ty * nb;
            const unsigned long long bits = sbins[(es * 2 + ty) * HRL_MAX_BINS + bb];
            so[26 + b] = bits == 0x7ff0000000000000ull ? 0.f : (float)(1.0 - __longlong_as_double((long long)bits) / (double)cfg.sensor_range);
          }
        }
      } else {
        // use_sensor=False -> get_abs_pos (:179-196): world xy of the min(n_bins, n) nearest food items, then
        // poison items, each sorted by squared distance (stable).  Rank = number of same-type items that sort
        // before this one; the 16 exact float64 distances are exchanged through shared memory.
        double* sd2 = reinterpret_cast<double*>(sbins + es * 2 * HRL_MAX_BINS);
        double d2v[IPL];
#pragma unroll
        for (int i = 0; i < IPL; i++) {
          const double dx = __dsub_rn((double)it_x[i], (double)s.O.x), dy = __dsub_rn((double)it_y[i], (double)s.O.y);
          d2v[i] = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
          sd2[IPL * l + i] = d2v[i];
        }
        __syncwarp();
        if (commit) {
          const int keep_f = min(nb, cfg.n_food), keep_p = min(nb, cfg.n_poison);
#pragma unroll
          for (int i = 0; i < IPL; i++) {
            const int gi = IPL * l + i;
            if (gi >= cfg.n_food + cfg.n_poison) continue;
            const bool poison = gi >= cfg.n_food;
            const int first = poison ? cfg.n_food : 0, cnt = poison ? cfg.n_poison : cfg.n_food;
            int rank = 0;
            for (int j = first; j < first + cnt; j++) rank += (sd2[j] < d2v[i] || (sd2[j] == d2v[i] && j < gi)) ? 1 : 0;
            if (rank < (poison ? keep_p : keep_f)) {
              const int at = 26 + (poison ? 2 * keep_f : 0) + 2 * rank;
              so[at] = it_x[i]; so[at + 1] = it_y[i];
            }
          }
        }
        __syncwarp();
      }
      if (touch_pickup) {  // the cube moves AFTER the observation of this step was built (:96 before :113)
#pragma unroll
        for (int i = 0; i < IPL; i++) {
          const int gi = IPL * l + i;
          if (gi >= cfg.n_food + cfg.n_poison || touch[i] == 0) continue;
          if (cfg.respawn) place_item(cfg, genv, STREAM_ITEM, (uint32_t)T.steps_total, gi, s.O.x, s.O.y, it_x[i], it_y[i]);
          else { it_x[i] = 100.f; it_y[i] = 0.f; }
        }
      }
      fin = isfinite(o_z) && isfinite(o_v0) && isfinite(o_v1) && isfinite(o_v2) && isfinite(o_r) && isfinite(o_p) &&
            isfinite(rel1) && isfinite(sp1) && isfinite(rel2) && isfinite(sp2);
      fin = (gsum(fin ? 0.f : 1.f) == 0.f);
      if (first && todo == 1) {
        const int alive = (o_z + T.initial_z) > 0.26f;  // Ant.alive_bonus on state[0] + initial_z (:99)
        done = !alive || !fin;                          // :100-103
        const float dead_rew = alive ? 0.f : cfg.dying_cost;
        T.t++; T.steps_total++;
        float trunc = 0.f;
        if (cfg.max_episode_steps > 0 && T.t >= cfg.max_episode_steps) { trunc = done ? 0.f : 1.f; done = 1; }
        T.ret += food_rew + dead_rew;
        if (done) { T.ret_sum += T.ret; T.ret = 0.f; }
        if (ROLL && ev_n >= 0) { ev_ret += food_rew + dead_rew; ev_n = done ? ~(ev_n + 1) : ev_n + 1; }
        if (active && l == 0) {
          if (!ROLL || rew_out) rew_out[e] = food_rew + dead_rew;
          if (!ROLL || done_out) done_out[e] = (uint8_t)done;
          if (info_out) reinterpret_cast<float4*>(info_out)[e] = make_float4(food_rew, dead_rew, trunc, (float)T.t);
        }
      }
    } else {
      // ---------------- walker family ----------------
      const bool mj = (kind == HRL_ANT_MJ || kind == HRL_ANT_MAZE_MJ);
      if (commit) {
        if (mj) {
          // MjAnt.calc_state envs/MjAnt.py:17-25: [pos3, quat4, q8, lin3, ang3, qd8] unclipped
          if (l == 0) {
            so[0] = s.O.x; so[1] = s.O.y; so[2] = s.O.z; so[3] = s.qx; so[4] = s.qy; so[5] = s.qz; so[6] = s.qw;
            so[15] = s.v.x; so[16] = s.v.y; so[17] = s.v.z; so[18] = s.w.x; so[19] = s.w.y; so[20] = s.w.z;
          }
          if (sub == 0) { so[7 + 2 * k] = s.q1; so[8 + 2 * k] = s.q2; so[21 + 2 * k] = s.qd1; so[22 + 2 * k] = s.qd2; }
          if (kind == HRL_ANT_MAZE_MJ) {  // ant_maze_mj_env.py:57-64
            const int nb = cfg.n_bins;
            for (int b = l; b < nb; b += LPE) {
              so[29 + b] = lidar_ray(b, nb, cfg.sensor_span, cfg.sensor_range, n_lines, bounds, s.O.x, s.O.y, yaw);
              so[29 + nb + b] = 0.f; so[29 + 2 * nb + b] = 0.f;
            }
            if (l == 0) so[29 + 3 * nb] = (float)T.t * 0.001f;
          }
        } else {
          const int off = (kind == HRL_ANT_FLAGRUN) ? 2 : 0;  // Flagrun keeps sin/cos of the target angle
          if (l == 0) {
            so[0] = o_z;
            if (off) { so[1] = clip5(sin_t); so[2] = clip5(cos_t); }
            so[1 + off] = o_v0; so[2 + off] = o_v1; so[3 + off] = o_v2; so[4 + off] = o_r; so[5 + off] = o_p;
            so[22 + off] = T.feet[0]; so[23 + off] = T.feet[1]; so[24 + off] = T.feet[2]; so[25 + off] = T.feet[3];
          }
          if (sub == 0) {
            so[6 + off + 4 * k] = clip5(rel1); so[7 + off + 4 * k] = clip5(sp1);
            so[8 + off + 4 * k] = clip5(rel2); so[9 + off + 4 * k] = clip5(sp2);
          }
          if (kind == HRL_ANT_MAZE) {
            int nt = 2;
            if (cfg.sense_target) {  // ant_maze_bullet_env.py:135-178: wtd is the Q1-distorted distance, the pose the true one
              nt = cfg.n_bins;
              const int tb = maze_target_bin(cfg.n_bins, cfg.sensor_span, cfg.sensor_range, cfg.has_box ? 3 : 0, bounds + 16, s.O.x,
                                             s.O.y, yaw, T.tx, T.ty, wtd_new);
              for (int b = l; b < nt; b += LPE) so[26 + b] = (b == tb) ? (float)(1.0 - (double)wtd_new / (double)cfg.sensor_range) : 0.f;
            } else if (l == 0) {  // ant_maze_bullet_env.py:123-133 (true torso xy, not the Q1 mean)
              const float vx = T.tx - s.O.x, vy = T.ty - s.O.y;
              if (cfg.target_encoding == 0) { const float nn = sqrtf(vx * vx + vy * vy); so[26] = vx / nn; so[27] = vy / nn; }
              else { float sa, ca; sincosf(atan2f(vy, vx) - yaw, &sa, &ca); so[26] = sa; so[27] = ca; }
            }
            if (cfg.sense_walls)
              for (int b = l; b < cfg.n_bins; b += LPE)
                so[26 + nt + b] = lidar_ray(b, cfg.n_bins, cfg.sensor_span, cfg.sensor_range, n_lines, bounds, s.O.x, s.O.y, yaw);
          }
          if (kind == HRL_ANT_FLAGRUN && cfg.flag_use_sensor)  // ant_flagrun_env.py:122-130 (body_real_xyz = torso)
            for (int b = l; b < cfg.n_bins; b += LPE)
              so[28 + b] = lidar_ray(b, cfg.n_bins, cfg.sensor_span, cfg.sensor_range, n_lines, bounds, s.O.x, s.O.y, yaw);
        }
      }
      if (todo == 2) {
        // Flagrun reset stage 1 (ant_flagrun_env.py:141-153): calc_state with the STALE target,
        // then next_target(): potential from that stale distance (quirk Q3)
        T.wtd = wtd_new;
        flag_next(cfg, genv, T, s.O.x, s.O.y, 1);
      }
      if (commit) {
        T.wtd = wtd_new;
        if (set_pot) { T.potential = -T.wtd / cfg.dt; set_pot = false; }
      }
      if (first && todo == 1) {
        // WalkerBaseBulletEnv.step [3P-MEM] (SURVEY.md App. A.2) / AntMjEnv.step envs/MjAnt.py:36-97
        fin = mj ? (isfinite(s.q1) && isfinite(s.q2) && isfinite(s.qd1) && isfinite(s.qd2) && isfinite(s.O.x + s.O.y + s.O.z) &&
                    isfinite(s.qx + s.qy + s.qz + s.qw) && isfinite(s.v.x + s.v.y + s.v.z) && isfinite(s.w.x + s.w.y + s.w.z))
                 : (isfinite(o_z) && isfinite(sin_t) && isfinite(cos_t) && isfinite(o_v0) && isfinite(o_v1) && isfinite(o_v2) &&
                    isfinite(o_r) && isfinite(o_p) && isfinite(rel1) && isfinite(sp1) && isfinite(rel2) && isfinite(sp2));
        fin = (gsum(fin ? 0.f : 1.f) == 0.f);
        const int alive = mj ? (s.O.z > 0.26f) : ((o_z + T.initial_z) > 0.26f);
        done = !alive || !fin;
        const float pot_old = T.potential;
        T.potential = -T.wtd / cfg.dt;
        const float progress = T.potential - pot_old;
        const float elec = gsum(fabsf(act1 * sp1) + fabsf(act2 * sp2)) * 0.125f;  // joint_speeds are unclipped
        const float sq = gsum(act1 * act1 + act2 * act2) * 0.125f;
        const float nlim = gsum((fabsf(rel1) > 0.99f ? 1.f : 0.f) + (fabsf(rel2) > 0.99f ? 1.f : 0.f));
        const float electricity = mj ? 0.f : (cfg.electricity_cost * elec + cfg.stall_torque_cost * sq);
        const float inner = (alive ? 1.f : -1.f) + progress + electricity + cfg.joints_at_limit_cost * nlim;
        // quirk Q2: feet flags measured in this step appear in the NEXT observation
#pragma unroll
        for (int j = 0; j < 4; j++) T.feet[j] = (float)__shfl_sync(HRL_FULL_MASK, feet_ground, (lane & ~3) | j);
        float rew = inner, info1 = 0.f;
        int next = 0;
        if (kind == HRL_ANT_MAZE) {
          // ant_maze_bullet_env.py:84-96; the reference's self.t (incremented at :78) is T.t + 1
          rew = inner * cfg.inner_rew_weight;
          const bool last = (T.t + 1 == cfg.maze_max_steps - 1);
          if (T.wtd < cfg.tol && (cfg.done_at_target || last)) { rew += 1.f; done = 1; }
          if (last) done = 1;
          if (cfg.targ_dist_rew && done) rew -= T.wtd;
        } else if (kind == HRL_ANT_MAZE_MJ) {
          rew = inner * cfg.inner_rew_weight;  // ant_maze_mj_env.py:73-77
          if (T.wtd < cfg.tol) { rew += 1.f; done = 1; }
        } else if (kind == HRL_ANT_FLAGRUN) {
          // ant_flagrun_env.py:162-204
          T.since += 1;
          if (T.wtd < cfg.tol) {
            if (!T.rewarded) { rew += cfg.goal_reach_rew; T.rewarded = 1; }
            if (cfg.flag_switch_on_collision) {
              if (flag_next(cfg, genv, T, s.O.x, s.O.y, 0)) { T.since = 0; next = 1; }
              else done = 1;
            }
          }
          if (cfg.flag_timeout > 0 && cfg.flag_timeout <= T.since) {
            if (flag_next(cfg, genv, T, s.O.x, s.O.y, 0)) { T.since = 0; next = 1; }
            else done = 1;
          }
          info1 = (float)T.goals_left;
        }
        T.t++; T.steps_total++;
        float trunc = 0.f;
        if (cfg.max_episode_steps > 0 && T.t >= cfg.max_episode_steps) { trunc = done ? 0.f : 1.f; done = 1; }
        T.ret += rew;
        if (done) { T.ret_sum += T.ret; T.ret = 0.f; }
        if (ROLL && ev_n >= 0) { ev_ret += rew; ev_n = done ? ~(ev_n + 1) : ev_n + 1; }
        if (active && l == 0) {
          if (!ROLL || rew_out) rew_out[e] = rew;
          if (!ROLL || done_out) done_out[e] = (uint8_t)done;
          // info[2]: bit 0 = TimeLimit.truncated, bit 1 = the walk target changed in this step (info['target'] is set)
          if (info_out) reinterpret_cast<float4*>(info_out)[e] = make_float4(inner, info1, trunc + 2.f * (float)next, (float)T.t);
        }
        switched = next;
      }
    }
    // ---------------- terminal obs + reset decision (only after the post-physics compose) ----------------
    int next_todo = 0;
    if (todo == 2) next_todo = 1;
    if (first && todo == 1) {
      if (switched) {  // fresh calc_state with the new target (ant_flagrun_env.py:120,190); a reset waits for it, so
        next_todo = 1; // that the terminal observation is the one the reference returns with done
        pend_reset = done && cfg.auto_reset;
      } else if (done && cfg.auto_reset) next_todo = 3;
    } else if (todo == 1 && pend_reset) { next_todo = 3; pend_reset = false; }
    const unsigned need_mask = __ballot_sync(HRL_FULL_MASK, next_todo == 3);
#ifdef HRL_WARP_TIMES
    wt_passes++; wt_resets += __popc(need_mask) / LPE;
#endif
    if (need_mask && term_out) {
      __syncwarp();
      for (int i = lane; i < EPW * D; i += 32) {
        const int w8 = i / D;
        if (((need_mask >> (LPE * w8)) & 1u) && env0 + w8 < N) term_out[(size_t)env0 * D + i] = sobs[i];
      }
      __syncwarp();
    }
    first = false;
    todo = next_todo;
  }

  if (mode != 1 && obs_out) {
    __syncwarp();
    // coalesced write-back of the staged observation rows (8 consecutive envs = one contiguous span)
    unsigned wmask = 0xffffffffu;
    if (mode == 2) {
      const bool m = mask ? (mask[e] != 0) : true;
      wmask = __ballot_sync(HRL_FULL_MASK, m);
    }
    float* dst = obs_out + (size_t)env0 * D;
    if (env0 + EPW <= N && wmask == 0xffffffffu && ((EPW * D) & 3) == 0 && (((uintptr_t)dst & 15) == 0)) {
      // common case: one contiguous, 16-byte aligned span -> float4 stores, no index arithmetic
      for (int i = lane; i < EPW * D / 4; i += 32) reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(sobs)[i];
    } else {
      for (int i = lane; i < EPW * D; i += 32) {
        const int w8 = i / D;
        if (env0 + w8 < N && ((wmask >> (LPE * w8)) & 1u)) dst[i] = sobs[i];
      }
    }
  }
  if (ROLL) __syncwarp();
  }  // step loop

  // ---- store ----
  if (active) {
    if (l == 0) {
      st.base[e * 4 + 0] = make_float4(s.O.x, s.O.y, s.O.z, T.initial_z);
      st.base[e * 4 + 1] = make_float4(s.qx, s.qy, s.qz, s.qw);
      st.base[e * 4 + 2] = make_float4(s.v.x, s.v.y, s.v.z, T.potential);
      st.base[e * 4 + 3] = make_float4(s.w.x, s.w.y, s.w.z, T.wtd);
      st.miscf[e * 2 + 0] = make_float4(T.tx, T.ty, T.ret, T.ret_sum);
      st.miscf[e * 2 + 1] = make_float4(T.feet[0], T.feet[1], T.feet[2], T.feet[3]);
      st.misci[e * 2 + 0] = make_int4(T.t, T.episode, T.steps_total, T.goals_left);
      st.misci[e * 2 + 1] = make_int4(T.since, T.rewarded, T.gen, 0);
      if (ROLL && ra.ev_ret) { ra.ev_ret[e] = ev_ret; ra.ev_len[e] = ev_n < 0 ? ~ev_n : ev_n; ra.ev_fin[e] = (uint8_t)(ev_n < 0); }
    }
    if (sub == 0) st.leg[e * 4 + k] = make_float4(s.q1, s.q2, s.qd1, s.qd2);
    if (FAMILY == 0) {
      if (IPL == 4) {
        st.items[(e * 4 + l) * 2 + 0] = make_float4(it_x[0], it_y[0], it_x[1], it_y[1]);
        st.items[(e * 4 + l) * 2 + 1] = make_float4(it_x[IPL - 2], it_y[IPL - 2], it_x[IPL - 1], it_y[IPL - 1]);
      } else if (IPL == 2) {
        st.items[e * 8 + l] = make_float4(it_x[0], it_y[0], it_x[IPL - 1], it_y[IPL - 1]);
      } else {
        reinterpret_cast<float2*>(st.items)[e * 16 + l] = make_float2(it_x[0], it_y[0]);
      }
    }
  }
#ifdef HRL_WARP_TIMES
  if (st.wt && lane == 0) {
    unsigned long long* w = st.wt + 4 * (size_t)(blockIdx.x * WPC + warp);
    w[0] = (unsigned long long)(clock64() - wt_t0); w[1] = (unsigned long long)(wt_t1 - wt_t0);
    w[2] = (unsigned long long)wt_trips; w[3] = (unsigned long long)(wt_passes | (wt_resets << 8));
  }
#endif
  if (st.fin_flag) {
    // release at device scope by every writer; the last CTA acquires through the counter and then
    // publishes with a system-scope fence (fences are cumulative; PCIe posted writes stay ordered)
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned prev = atomicAdd(st.fin_count, 1u);
      if (prev == gridDim.x - 1) {  // last CTA: all others fenced before they counted
        __threadfence();
        *st.fin_count = 0;
        __threadfence_system();
        *(volatile unsigned int*)st.fin_flag = st.fin_seq;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// PointGather (point_bot.py, gather_base.py:74-109): 16 lanes per env, lane j owns item j.  The cube
// only translates (north star: "the PointGather point-mass integrator"); its trivial physics is
// evaluated redundantly by the 16 lanes, the per-item work (pickup, respawn, sector bin) is parallel.
// State lives in the same DevState arrays (base rows 0/2, items).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float sum16(float v) {
#pragma unroll
  for (int o = 1; o < 16; o <<= 1) v += __shfl_xor_sync(HRL_FULL_MASK, v, o);
  return v;
}

// One internal step.  Candidate contacts are the 5 fixed surfaces (ground, walls +x -x +y -y) in that order;
// everything is indexed statically so that the solver state stays in registers.
__device__ __forceinline__ void point_substep(V3& pos, V3& vel, V3 force, const SubstepParams& P) {
  const float m = pointbot::MASS, half = pointbot::HALF, im = 1.0f / m;
  const float wx = P.wx - half, wy = P.wy - half;
  const V3 Nn[5] = {mk(0.f, 0.f, 1.f), mk(-1.f, 0.f, 0.f), mk(1.f, 0.f, 0.f), mk(0.f, -1.f, 0.f), mk(0.f, 1.f, 0.f)};
  const float Dd[5] = {pos.z - half - P.gz, wx - pos.x, pos.x + wx, wy - pos.y, pos.y + wy};
  bool on[5];
#pragma unroll
  for (int c = 0; c < 5; c++) on[c] = (c == 0 || P.has_walls) && (Dd[c] < P.margin);
  const V3 f = mk(force.x, force.y, force.z - m * P.g) + (-m * (P.kl + P.kl * norm(vel))) * vel;
  V3 v = vel + (P.h * im) * f;
  v = mk(clampf(v.x, P.vmax), clampf(v.y, P.vmax), clampf(v.z, P.vmax));
  float lamn[5], lama[5], lamb[5], rhsn[5], rhsa[5], rhsb[5];
  V3 T1[5], T2[5];
#pragma unroll
  for (int c = 0; c < 5; c++) {
    const float rel = dot(Nn[c], v);
    float posErr = 0.f, velErr = -rel;
    if (Dd[c] > 0.f) velErr -= Dd[c] * P.inv_h; else posErr = -Dd[c] * P.erp_c * P.inv_h;
    rhsn[c] = (posErr + velErr) * m;
    plane_space(Nn[c], T1[c], T2[c]);
    rhsa[c] = -dot(T1[c], v) * m; rhsb[c] = -dot(T2[c], v) * m;
    lamn[c] = lama[c] = lamb[c] = 0.f;
  }
  V3 dv = mk(0.f, 0.f, 0.f);
  for (int it = 0; it < P.iters; it++) {
#pragma unroll
    for (int c = 0; c < 5; c++) {
      if (!on[c]) continue;
      float dl = rhsn[c] - dot(Nn[c], dv) * m;
      if (lamn[c] + dl < 0.f) dl = -lamn[c];
      lamn[c] += dl; dv = dv + (dl * im) * Nn[c];
    }
#pragma unroll
    for (int c = 0; c < 5; c++) {
      if (!on[c] || !(lamn[c] > 0.f)) continue;
      float sa = lama[c] + rhsa[c] - dot(T1[c], dv) * m, sb = lamb[c] + rhsb[c] - dot(T2[c], dv) * m;
      const float lim = P.mu * lamn[c], len2 = sa * sa + sb * sb;
      if (len2 > lim * lim) { const float sc = lim * rsqrtf(len2); sa *= sc; sb *= sc; }
      const float da = sa - lama[c], db = sb - lamb[c];
      lama[c] = sa; lamb[c] = sb;
      dv = dv + (da * im) * T1[c] + (db * im) * T2[c];
    }
  }
  vel = v + dv;
  pos = pos + P.h * vel;
}

#define HRL_POINT_EPB 8  // envs per 128-thread block
#define HRL_POINT_OBS (8 + 2 * HRL_MAX_BINS)  // widest PointGather observation

// PointGather rollout policy: the 16 lanes of an env split the hidden units, lane j owns units U j .. U j + U - 1
// (U = H / 16: one float4 or float2 of every weight row, the 16 lanes read 256 / 128 contiguous bytes, the 2 envs of a
// warp read the same addresses: broadcast).  Weights as in mlp_policy, with W3[H][2] b3[2].
template <int U>
__device__ __forceinline__ void mlp_layer16(const float* __restrict__ w, const float* __restrict__ b, int n_in, const float* __restrict__ x,
                                            int j, float (&acc)[U]) {
  constexpr int H = 16 * U;
#pragma unroll
  for (int u = 0; u < U; u++) acc[u] = b[U * j + u];
#pragma unroll 4
  for (int i = 0; i < n_in; i++) {
    const float xi = x[i];
    const float* wr = w + i * H + U * j;
    if (U == 4) {
      const float4 wv = *reinterpret_cast<const float4*>(wr);
      acc[0] = fmaf(xi, wv.x, acc[0]); acc[1] = fmaf(xi, wv.y, acc[1]); acc[U - 2] = fmaf(xi, wv.z, acc[U - 2]); acc[U - 1] = fmaf(xi, wv.w, acc[U - 1]);
    } else {
      const float2 wv = *reinterpret_cast<const float2*>(wr);
      acc[0] = fmaf(xi, wv.x, acc[0]); acc[U - 1] = fmaf(xi, wv.y, acc[U - 1]);
    }
  }
#pragma unroll
  for (int u = 0; u < U; u++) acc[u] = tanhf(acc[u]);
}
// w: the packed weights in shared memory; obs: this env's staged observation; hid: 64 floats of this env (shared memory)
template <int U>
__device__ __forceinline__ float2 mlp_policy16(const float* __restrict__ w, int D, const float* __restrict__ obs, float* __restrict__ hid, int j) {
  constexpr int H = 16 * U;
  HRL_CHECK(D <= HRL_POINT_OBS && j >= 0 && j < 16);   // every weight read stays inside the D * H + H + H * H + H + H * 2 + 2 staged floats
  const float* w1 = w, *b1 = w1 + D * H, *w2 = b1 + H, *b2 = w2 + H * H, *w3 = b2 + H, *b3 = w3 + H * 2;
  float h[U];
  mlp_layer16<U>(w1, b1, D, obs, j, h);
#pragma unroll
  for (int u = 0; u < U; u++) {
    HRL_CHECK(U * j + u < 64);
    hid[U * j + u] = h[u];
  }
  __syncwarp();
  mlp_layer16<U>(w2, b2, H, hid, j, h);
  __syncwarp();   // hid is rewritten by the next step's first layer
  float ox = 0.f, oy = 0.f;  // this lane's share of W3 h2, summed over the half-warp
#pragma unroll
  for (int u = 0; u < U; u++) {
    const float2 wv = *reinterpret_cast<const float2*>(w3 + (U * j + u) * 2);
    ox = fmaf(h[u], wv.x, ox); oy = fmaf(h[u], wv.y, oy);
  }
  return make_float2(tanhf(sum16(ox) + b3[0]), tanhf(sum16(oy) + b3[1]));
}
#define HRL_POINT_MLP_MAX_FLOATS (HRL_POINT_OBS * 64 + 64 + 64 * 64 + 64 + 64 * 2 + 2)

// ROLL = 1: the fused rollout of PointGather (see ant_env_kernel): step -1 composes the initial observation, steps
// 0 .. T-1 are full steps whose actions the MLP computes from the observation the previous pass left in sobs; the env
// state stays in registers in between.  Dynamic shared memory: [EPB][64] hidden activations, then the weights.
// ROLL = 2: ROLL = 1 with a normalized policy input (hrl_rollout_mlp_norm); mean[D] and rstd[D] follow the weights.
// ROLL: 4 blocks per SM caps the registers at 128; left to itself ptxas picks 96 and spills the rollout's loop state
template <int ROLL = 0>
__global__ void __launch_bounds__(16 * HRL_POINT_EPB, ROLL ? 4 : 0)
point_env_kernel(const __grid_constant__ hrl_config cfg, DevState st, const float* __restrict__ actions,
                 const uint8_t* __restrict__ mask, float* __restrict__ obs_out_g, float* __restrict__ rew_out_g,
                 uint8_t* __restrict__ done_out_g, float* __restrict__ info_out_g, float* __restrict__ term_out_g, int mode_g,
                 int n_sub, int D, RollArgs ra = RollArgs()) {
  __shared__ unsigned long long sb[HRL_POINT_EPB][2][HRL_MAX_BINS];
  __shared__ float sobs[HRL_POINT_EPB][HRL_POINT_OBS];
  extern __shared__ __align__(16) float smem[];
  const int j = threadIdx.x & 15, eb = threadIdx.x >> 4;
  const int e_raw = blockIdx.x * HRL_POINT_EPB + eb;
  const bool valid = e_raw < cfg.num_envs;
  const int N = cfg.num_envs;
  const int e = valid ? e_raw : cfg.num_envs - 1;  // tail lanes shadow the last env (no stores): every *_sync stays warp-wide
  const uint32_t genv = (uint32_t)(cfg.env_index_offset + e);
  float* hid = smem + eb * 64;
  const float* wsm = smem + HRL_POINT_EPB * 64;
  const float* nstat = wsm + (ROLL == 2 ? D * ra.H + ra.H + ra.H * ra.H + ra.H + ra.H * 2 + 2 : 0);  // ROLL = 2: mean[D], rstd[D]
  if (ROLL) {
    HRL_CHECK(D <= HRL_POINT_OBS && (ra.H == 32 || ra.H == 64));
    const int nw = D * ra.H + ra.H + ra.H * ra.H + ra.H + ra.H * 2 + 2;
    const float* wg = ra.w + (size_t)((int)blockIdx.x * HRL_POINT_EPB / ra.m_envs) * nw;   // this block's member
    for (int i = threadIdx.x; i < nw; i += 16 * HRL_POINT_EPB) const_cast<float*>(wsm)[i] = __ldg(wg + i);
    if (ROLL == 2)
      for (int i = threadIdx.x; i < 2 * D; i += 16 * HRL_POINT_EPB) const_cast<float*>(nstat)[i] = __ldg(i < D ? ra.obs_mean + i : ra.obs_rstd + (i - D));
    __syncthreads();
  }
  const float4 b0 = st.base[e * 4 + 0], b2 = st.base[e * 4 + 2];
  float4 m0 = st.miscf[e * 2 + 0];  // .z running episode return, .w sum of finished returns
  int4 i0 = st.misci[e * 2 + 0];
  V3 pos = mk(b0.x, b0.y, b0.z), vel = mk(b2.x, b2.y, b2.z);
  float initial_z = b0.w;
  const int n_items = cfg.n_food + cfg.n_poison, nb = cfg.n_bins;
  const bool has_item = j < n_items;
  float2 it = reinterpret_cast<const float2*>(st.items)[e * 16 + j];  // item j: food 0..n_food-1, then poison
  float ev_ret = 0.f;  // ROLL: the launch's first episode (see ant_env_kernel)
  int ev_n = 0;
#pragma unroll 1
  for (int step = ROLL ? -1 : 0; step < (ROLL ? ra.T : 1); step++) {
  const int mode = ROLL ? (step < 0 ? 3 : 0) : mode_g;
  float* __restrict__ obs_out = ROLL && obs_out_g ? obs_out_g + (size_t)(step + 1) * N * D : obs_out_g;
  float* __restrict__ rew_out = ROLL && rew_out_g ? rew_out_g + (size_t)max(step, 0) * N : rew_out_g;
  uint8_t* __restrict__ done_out = ROLL && done_out_g ? done_out_g + (size_t)max(step, 0) * N : done_out_g;
  float* __restrict__ info_out = ROLL && info_out_g ? info_out_g + (size_t)max(step, 0) * N * 4 : info_out_g;
  float* __restrict__ term_out = ROLL && term_out_g ? term_out_g + (size_t)max(step, 0) * N * D : term_out_g;
  if (mode <= 1) {
    float ax, ay;
    if (ROLL) {
      const float* x = sobs[eb];
      if (ROLL == 2) {  // normalized input in this env's sensor-bin tile (64 floats), which the observation pass re-initialises
        static_assert(sizeof(sb[0]) >= HRL_POINT_OBS * sizeof(float), "the bin tile must hold a normalized observation");
        float* xn = reinterpret_cast<float*>(sb[eb]);
        for (int i = j; i < D; i += 16) xn[i] = norm_obs(sobs[eb][i], nstat, D, i, ra.obs_clip);
        __syncwarp();
        x = xn;
      }
      const float2 a = ra.H == 64 ? mlp_policy16<4>(wsm, D, x, hid, j) : mlp_policy16<2>(wsm, D, x, hid, j);
      ax = a.x; ay = a.y;
      if (ra.sigma_v || ra.sigma > 0.f) {  // exploration noise: one Box-Muller pair for the two components (as lane 0 of an ant)
        const float s1 = ra.sigma_v ? __ldg(ra.sigma_v) : ra.sigma, s2 = ra.sigma_v ? __ldg(ra.sigma_v + 1) : ra.sigma;
        float u[4];
        rng_u4(ra.seed, genv, STREAM_POLICY, (uint32_t)i0.z, 0u, u);
        const float r0 = sqrtf(-2.f * logf(u[0] + 2.98e-8f));
        float sn, cs;
        sincosf(6.2831853f * u[1], &sn, &cs);
        ax += s1 * r0 * cs; ay += s2 * r0 * sn;
      }
      if (valid && j == 0 && ra.act_out) reinterpret_cast<float2*>(ra.act_out)[(size_t)step * N + e] = make_float2(ax, ay);
    } else {
      ax = actions[e * 2]; ay = actions[e * 2 + 1];
    }
    // point_bot.py:28-31: F = a/|a| * 500 N in the world frame (NaN for a == 0: kept, see gather_base.py:99-101)
    const float nn = sqrtf(ax * ax + ay * ay);
    const V3 F = mk(ax / nn * cfg.torque_scale, ay / nn * cfg.torque_scale, 0.f), Z = mk(0.f, 0.f, 0.f);
    const SubstepParams P = make_params(cfg);
    const int ns = mode == 0 ? cfg.substeps : n_sub;
    for (int i = 0; i < ns; i++) point_substep(pos, vel, (i == 0 || !cfg.torque_first_substep_only) ? F : Z, P);
  }
  bool do_reset = (mode == 2) && (mask ? mask[e] != 0 : true);
  bool work = (mode == 0) || (mode == 3) || do_reset;  // this env still has an observation to produce
  bool stepping = (mode == 0);
  for (int pass = 0; pass < 2; pass++) {
    if (!__any_sync(HRL_FULL_MASK, work)) break;
    if (work && do_reset) {
      i0.x = 0; m0.z = 0.f;
      pos = mk(cfg.start_pos[0], cfg.start_pos[1], cfg.start_pos[2]); vel = mk(0.f, 0.f, 0.f);  // point_bot.py:12,25-26
      initial_z = 1.f;                                                                            // point_bot.py:18
      if (has_item) place_item(cfg, genv, STREAM_ITEM_RESET, (uint32_t)i0.y, j, 0.f, 0.f, it.x, it.y);
      i0.y++;
      do_reset = false;
    }
    float rew_j = 0.f;
    if (work && stepping && has_item) {  // pickup of this lane's item (gather_base.py:84-90, gather_scene.py:95-114)
      const double dx = __dsub_rn((double)it.x, (double)pos.x), dy = __dsub_rn((double)it.y, (double)pos.y);
      const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
      if (d2 < (double)cfg.robot_coll_dist) {
        rew_j = (j < cfg.n_food) ? 1.f : -1.f;
        if (cfg.respawn) place_item(cfg, genv, STREAM_ITEM, (uint32_t)i0.z, j, pos.x, pos.y, it.x, it.y);
        else { it.x = 100.f; it.y = 0.f; }
      }
    }
    const float food_rew = sum16(rew_j);
    // observation: point_bot.py:48-67 (roll = pitch = yaw = 0) + sector sensor gather_base.py:118-168
    for (int b = j; b < 2 * HRL_MAX_BINS; b += 16) sb[eb][b / HRL_MAX_BINS][b % HRL_MAX_BINS] = 0x7ff0000000000000ull;
    __syncwarp();
    if (work && has_item) {
      double d2;
      const int b = gather_item_bin(pos.x, pos.y, 0.f, it.x, it.y, nb, cfg.sensor_range, cfg.sensor_span, &d2);
      HRL_CHECK(b < HRL_MAX_BINS && eb >= 0 && eb < HRL_POINT_EPB);
      if (b >= 0) atomicMin(&sb[eb][j < cfg.n_food ? 0 : 1][b], (unsigned long long)__double_as_longlong(d2));
    }
    __syncwarp();
    // ROLL: sobs of an env without work keeps the observation it emitted last (the policy's next input)
    const bool compose = !ROLL || work;
    float sa, ca;
    sincosf(atan2f(0.f - pos.y, 0.f - pos.x), &sa, &ca);
    const float o8[8] = {pos.z - initial_z, sa, ca, 0.3f * vel.x, 0.3f * vel.y, 0.3f * vel.z, 0.f, 0.f};
    if (compose && j < 8) {
      float v = o8[0];
#pragma unroll
      for (int q = 1; q < 8; q++) v = (j == q) ? o8[q] : v;
      sobs[eb][j] = v;
    }
    if (cfg.use_sensor) {
      for (int b = j; compose && b < 2 * nb; b += 16) {
        const int ty = b / nb, bb = b - ty * nb;
        const unsigned long long bits = sb[eb][ty][bb];
        sobs[eb][8 + b] = bits == 0x7ff0000000000000ull ? 0.f : (float)(1.0 - __longlong_as_double((long long)bits) / (double)cfg.sensor_range);
      }
    } else {
      // use_sensor=False -> get_abs_pos (gather_base.py:170-187): world xy of the min(n_bins, n) nearest food items, then
      // poison items, each sorted by squared distance (stable).  Lane j's rank = number of same-type items that sort
      // before its own; the 16 exact float64 distances go round the half-warp by shuffle.
      const double dx = __dsub_rn((double)it.x, (double)pos.x), dy = __dsub_rn((double)it.y, (double)pos.y);
      const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
      const bool poison = j >= cfg.n_food;
      int rank = 0;
#pragma unroll 1
      for (int o = 0; o < 16; o++) {
        const double od = __shfl_sync(HRL_FULL_MASK, d2, o, 16);
        const bool same = o < n_items && ((o >= cfg.n_food) == poison);
        rank += (same && (od < d2 || (od == d2 && o < j))) ? 1 : 0;
      }
      const int keep_f = min(nb, cfg.n_food), keep_p = min(nb, cfg.n_poison);
      if (compose && has_item && rank < (poison ? keep_p : keep_f)) {
        const int at = 8 + (poison ? 2 * keep_f : 0) + 2 * rank;
        HRL_CHECK(at >= 0 && at + 1 < HRL_POINT_OBS && at + 1 < D);
        sobs[eb][at] = it.x; sobs[eb][at + 1] = it.y;
      }
    }
    __syncwarp();
    bool emit = work && (mode != 1);
    bool again = false;
    if (work && stepping) {
      bool fin = true;
#pragma unroll
      for (int q = 0; q < 8; q++) fin = fin && isfinite(o8[q]);
      int done = !fin;  // PointBot.alive_bonus is always 1 (point_bot.py:73-74)
      i0.x++; i0.z++;
      float trunc = 0.f;
      if (cfg.max_episode_steps > 0 && i0.x >= cfg.max_episode_steps) { trunc = done ? 0.f : 1.f; done = 1; }
      m0.z += food_rew;
      if (done) { m0.w += m0.z; m0.z = 0.f; }
      if (ROLL && ev_n >= 0) { ev_ret += food_rew; ev_n = done ? ~(ev_n + 1) : ev_n + 1; }
      if (valid && j == 0) {
        if (!ROLL || rew_out) rew_out[e] = food_rew;
        if (!ROLL || done_out) done_out[e] = (uint8_t)done;
        if (info_out) reinterpret_cast<float4*>(info_out)[e] = make_float4(food_rew, 0.f, trunc, (float)i0.x);
      }
      if (done && cfg.auto_reset) {
        if (term_out && valid) for (int q = j; q < D; q += 16) term_out[(size_t)e * D + q] = sobs[eb][q];
        do_reset = true; again = true; emit = false;
      }
      stepping = false;
    }
    if (emit && obs_out && valid) for (int q = j; q < D; q += 16) obs_out[(size_t)e * D + q] = sobs[eb][q];
    work = again;
    __syncwarp();
  }
  }  // step loop
  if (valid) {
    if (j == 0) {
      st.base[e * 4 + 0] = make_float4(pos.x, pos.y, pos.z, initial_z);
      st.base[e * 4 + 1] = make_float4(0.f, 0.f, 0.f, 1.f);  // the cube never rotates
      st.base[e * 4 + 2] = make_float4(vel.x, vel.y, vel.z, 0.f);
      st.miscf[e * 2 + 0] = m0;
      st.misci[e * 2 + 0] = i0;
      if (ROLL && ra.ev_ret) { ra.ev_ret[e] = ev_ret; ra.ev_len[e] = ev_n < 0 ? ~ev_n : ev_n; ra.ev_fin[e] = (uint8_t)(ev_n < 0); }
    }
    reinterpret_cast<float2*>(st.items)[e * 16 + j] = it;
  }
}

// ------------------------------------------------------------------------------------------
// state import / export (public layout of include/hrl_b200.h), one thread per env
// ------------------------------------------------------------------------------------------
__global__ void get_state_kernel(int N, DevState st, float* __restrict__ f, int32_t* __restrict__ iv) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  float* o = f + (size_t)e * HRL_STATE_F;
  for (int i = 0; i < HRL_STATE_F; i++) o[i] = 0.f;
  const float4 b0 = st.base[e * 4], b1 = st.base[e * 4 + 1], b2 = st.base[e * 4 + 2], b3 = st.base[e * 4 + 3];
  o[HRL_SF_POS] = b0.x; o[HRL_SF_POS + 1] = b0.y; o[HRL_SF_POS + 2] = b0.z; o[HRL_SF_INITIAL_Z] = b0.w;
  o[HRL_SF_QUAT] = b1.x; o[HRL_SF_QUAT + 1] = b1.y; o[HRL_SF_QUAT + 2] = b1.z; o[HRL_SF_QUAT + 3] = b1.w;
  o[HRL_SF_LINVEL] = b2.x; o[HRL_SF_LINVEL + 1] = b2.y; o[HRL_SF_LINVEL + 2] = b2.z; o[HRL_SF_POTENTIAL] = b2.w;
  o[HRL_SF_ANGVEL] = b3.x; o[HRL_SF_ANGVEL + 1] = b3.y; o[HRL_SF_ANGVEL + 2] = b3.z; o[HRL_SF_WTD] = b3.w;
  for (int k = 0; k < 4; k++) {
    const float4 l = st.leg[e * 4 + k];
    o[HRL_SF_Q + 2 * k] = l.x; o[HRL_SF_Q + 2 * k + 1] = l.y; o[HRL_SF_QD + 2 * k] = l.z; o[HRL_SF_QD + 2 * k + 1] = l.w;
  }
  const float4 m0 = st.miscf[e * 2], m1 = st.miscf[e * 2 + 1];
  o[HRL_SF_TARGET] = m0.x; o[HRL_SF_TARGET + 1] = m0.y; o[HRL_SF_RETURN] = m0.z; o[HRL_SF_RETURN_SUM] = m0.w;
  o[HRL_SF_FEET] = m1.x; o[HRL_SF_FEET + 1] = m1.y; o[HRL_SF_FEET + 2] = m1.z; o[HRL_SF_FEET + 3] = m1.w;
  for (int l = 0; l < 8; l++) {
    const float4 a = st.items[e * 8 + l];
    o[HRL_SF_ITEMS + 4 * l] = a.x; o[HRL_SF_ITEMS + 4 * l + 1] = a.y; o[HRL_SF_ITEMS + 4 * l + 2] = a.z; o[HRL_SF_ITEMS + 4 * l + 3] = a.w;
  }
  const int4 i0 = st.misci[e * 2], i1 = st.misci[e * 2 + 1];
  int32_t* q = iv + (size_t)e * HRL_STATE_I;
  for (int i = 0; i < HRL_STATE_I; i++) q[i] = 0;
  q[HRL_SI_T] = i0.x; q[HRL_SI_EPISODE] = i0.y; q[HRL_SI_STEPS] = i0.z; q[HRL_SI_GOALS_LEFT] = i0.w;
  q[HRL_SI_SINCE] = i1.x; q[HRL_SI_REWARDED] = i1.y; q[HRL_SI_GOAL_GEN] = i1.z;
}

__global__ void set_state_kernel(int N, DevState st, const float* __restrict__ f, const int32_t* __restrict__ iv) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  const float* o = f + (size_t)e * HRL_STATE_F;
  st.base[e * 4] = make_float4(o[HRL_SF_POS], o[HRL_SF_POS + 1], o[HRL_SF_POS + 2], o[HRL_SF_INITIAL_Z]);
  st.base[e * 4 + 1] = make_float4(o[HRL_SF_QUAT], o[HRL_SF_QUAT + 1], o[HRL_SF_QUAT + 2], o[HRL_SF_QUAT + 3]);
  st.base[e * 4 + 2] = make_float4(o[HRL_SF_LINVEL], o[HRL_SF_LINVEL + 1], o[HRL_SF_LINVEL + 2], o[HRL_SF_POTENTIAL]);
  st.base[e * 4 + 3] = make_float4(o[HRL_SF_ANGVEL], o[HRL_SF_ANGVEL + 1], o[HRL_SF_ANGVEL + 2], o[HRL_SF_WTD]);
  for (int k = 0; k < 4; k++)
    st.leg[e * 4 + k] = make_float4(o[HRL_SF_Q + 2 * k], o[HRL_SF_Q + 2 * k + 1], o[HRL_SF_QD + 2 * k], o[HRL_SF_QD + 2 * k + 1]);
  st.miscf[e * 2] = make_float4(o[HRL_SF_TARGET], o[HRL_SF_TARGET + 1], o[HRL_SF_RETURN], o[HRL_SF_RETURN_SUM]);
  st.miscf[e * 2 + 1] = make_float4(o[HRL_SF_FEET], o[HRL_SF_FEET + 1], o[HRL_SF_FEET + 2], o[HRL_SF_FEET + 3]);
  for (int l = 0; l < 8; l++)
    st.items[e * 8 + l] = make_float4(o[HRL_SF_ITEMS + 4 * l], o[HRL_SF_ITEMS + 4 * l + 1], o[HRL_SF_ITEMS + 4 * l + 2], o[HRL_SF_ITEMS + 4 * l + 3]);
  const int32_t* q = iv + (size_t)e * HRL_STATE_I;
  st.misci[e * 2] = make_int4(q[HRL_SI_T], q[HRL_SI_EPISODE], q[HRL_SI_STEPS], q[HRL_SI_GOALS_LEFT]);
  st.misci[e * 2 + 1] = make_int4(q[HRL_SI_SINCE], q[HRL_SI_REWARDED], q[HRL_SI_GOAL_GEN], 0);
}

// ------------------------------------------------------------------------------------------
// stand-alone parity kernels
// ------------------------------------------------------------------------------------------
__global__ void gather_sensor_kernel(int M, int n_bins, float range, float span, const float* __restrict__ xy,
                                     const float* __restrict__ yaw, const float* __restrict__ items,
                                     float* __restrict__ food, float* __restrict__ poison, int32_t* __restrict__ bins) {
  // 16 lanes per case (one per item), 2 cases per warp
  __shared__ unsigned long long sb[8][2][2 * HRL_MAX_BINS];
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const int m = tid >> 4, gi = tid & 15, warp = threadIdx.x >> 5, half = (threadIdx.x >> 4) & 1, lane16 = threadIdx.x & 15;
  for (int i = lane16; i < 2 * HRL_MAX_BINS; i += 16) sb[warp][half][i] = 0x7ff0000000000000ull;
  __syncwarp();
  const bool ok = m < M;
  int b = -1;
  if (ok) {
    double d2;
    b = gather_item_bin(xy[2 * m], xy[2 * m + 1], yaw[m], items[(m * 16 + gi) * 2], items[(m * 16 + gi) * 2 + 1], n_bins, range, span, &d2);
    if (bins) bins[m * 16 + gi] = b;
    HRL_CHECK(b < HRL_MAX_BINS && b < n_bins);
    if (b >= 0) atomicMin(&sb[warp][half][(gi < 8 ? 0 : HRL_MAX_BINS) + b], (unsigned long long)__double_as_longlong(d2));
  }
  __syncwarp();
  if (ok)
    for (int i = lane16; i < 2 * n_bins; i += 16) {
      const int ty = i / n_bins, bb = i - ty * n_bins;
      const unsigned long long bits = sb[warp][half][ty * HRL_MAX_BINS + bb];
      const float v = bits == 0x7ff0000000000000ull ? 0.f : (float)(1.0 - __longlong_as_double((long long)bits) / (double)range);
      (ty ? poison : food)[m * n_bins + bb] = v;
    }
}

__global__ void sense_walls_kernel(int M, int n_bins, float span, float range, int n_lines, const float* __restrict__ bounds,
                                   const float* __restrict__ xy, const float* __restrict__ yaw, float* __restrict__ out) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= M * n_bins) return;
  const int m = tid / n_bins, i = tid - m * n_bins;
  out[tid] = lidar_ray(i, n_bins, span, range, n_lines, bounds, xy[2 * m], xy[2 * m + 1], yaw[m]);
}

// ------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------
static int scene_bounds(const hrl_config* cfg, float* b) {
  // sizeable_enclosed_scene.py:25-34 then maze_scene.py:15-21 (same order as the reference)
  const float x1 = cfg->world_size[0] / 2.f, y1 = cfg->world_size[1] / 2.f, x2 = -x1, y2 = -y1;
  const float w[4][4] = {{x1, y1, x2, y1}, {x1, y1, x1, y2}, {x2, y2, x2, y1}, {x2, y2, x1, y2}};
  memcpy(b, w, sizeof w);
  if (!cfg->has_box) return 4;
  const float bx1 = cfg->box_hi[0], by1 = cfg->box_hi[1], bx2 = cfg->box_lo[0], by2 = cfg->box_lo[1];
  const float bb[3][4] = {{bx1, by1, bx1, by2}, {bx2, by2, bx2, by1}, {bx2, by2, bx1, by2}};
  memcpy(b + 16, bb, sizeof bb);
  return 7;
}

extern "C" {

const char* hrl_last_error(void) { return g_err; }
#define HRL_STR2(x) #x
#define HRL_STR(x) HRL_STR2(x)
const char* hrl_version(void) {
  return "hrl_b200 0.2 (sm_100a; 4 lanes/env; " HRL_STR(HRL_ENVS_PER_WARP) " envs/warp; " HRL_STR(HRL_WARPS_PER_CTA) " warps/CTA; MAXC=" HRL_STR(HRL_MAXC)
#ifdef HRL_BOUNDS
         "; HRL_BOUNDS: device-side index asserts"
#endif
         ")";
}
int64_t hrl_launch_count(void) { return (int64_t)g_launches.load(); }

int hrl_default_config(int32_t kind, int32_t num_envs, hrl_config* c) {
  if (!c) return set_err(HRL_E_INVALID, "null config");
  memset(c, 0, sizeof *c);
  c->env_kind = kind; c->num_envs = num_envs; c->seed = 0; c->max_episode_steps = 2000; c->auto_reset = 1;
  // third-party constants recalled in SURVEY.md App. A.2/A.3 [3P-MEM]
  c->gravity = 9.8f; c->dt = 0.0165f; c->substeps = 4; c->solver_iters = 5;
  c->contact_erp = 0.9f; c->limit_erp = 0.2f; c->lin_damping = 0.04f; c->ang_damping = 0.04f;
  c->friction = 1.5f * 0.8f; c->limit_max_impulse = 100.f; c->max_coord_vel = 100.f; c->contact_margin = 0.02f;
  c->torque_scale = 250.f; c->torque_first_substep_only = 1;
  c->ground_z = 0.005f; c->has_walls = 1; c->has_box = 0;
  // ant_gather_env.py:16-29
  c->n_food = 8; c->n_poison = 8; c->n_bins = 10; c->sensor_range = 20.f; c->sensor_span = (float)HRL_PI_D;
  c->robot_coll_dist = 1.f; c->robot_object_spacing = 2.f; c->dying_cost = -10.f; c->respawn = 1; c->use_sensor = 1;
  // ant_maze_bullet_env.py:23-25
  c->tol = 1.5f; c->done_at_target = 1; c->inner_rew_weight = 0.f; c->target_encoding = 0; c->sense_walls = 1;
  // ant_flagrun_env.py:14-16,157-160
  c->flag_max_targets = 100; c->flag_timeout = 200; c->flag_size = 10.f; c->goal_reach_rew = 5000.f; c->flag_seed = 123;
  c->electricity_cost = -2.0f; c->stall_torque_cost = -0.1f; c->joints_at_limit_cost = -0.1f;
  // non-default kwargs (SURVEY.md 8f item 3): off unless asked for
  c->sense_target = 0; c->maze_max_steps = -1; c->targ_dist_rew = 0;
  c->flag_use_sensor = 0; c->flag_switch_on_collision = 1; c->flag_max_target_dist = 0.f;
  c->item_contacts = 0; c->item_friction = 1.5f * 0.5f; c->item_half = 0.125f; c->item_z = 0.1f;  // assets/food.xml:17-22
  switch (kind) {
    case HRL_ANT_GATHER:
      c->world_size[0] = c->world_size[1] = 15; c->start_pos[2] = 0.75f;
      c->item_contacts = 1;  // the food / poison cubes are real static colliders in the reference (gather_scene.py:66)
      break;
    case HRL_POINT_GATHER:  // point_gather_env.py:8-21, point_bot.py:12,29, player_cube.xml:8
      c->world_size[0] = c->world_size[1] = 15; c->start_pos[2] = 0.5f; c->n_bins = 5;
      c->friction = 0.1f * 0.8f; c->torque_scale = 500.f; break;
    case HRL_ANT_MAZE:
    case HRL_ANT_MAZE_MJ: {  // maze_scene.py:9-21, ant_maze_bullet_env.py:13-14,27; ant_maze_mj_env.py:13-14
      c->world_size[0] = 10; c->world_size[1] = 18; c->has_box = 1;
      c->box_lo[0] = -5; c->box_lo[1] = -2; c->box_lo[2] = 0; c->box_hi[0] = 1; c->box_hi[1] = 2; c->box_hi[2] = 2;
      c->start_pos[0] = -2; c->start_pos[1] = -5; c->start_pos[2] = 0.25f;
      c->sensor_range = 5.f; c->sensor_span = (float)(2 * HRL_PI_D);
      c->n_scene_parts = 3; c->scene_parts_sum[0] = -7; c->scene_parts_sum[1] = 0;  // quirk Q1
      if (kind == HRL_ANT_MAZE) {
        const float t[4][2] = {{2, -3}, {2, 0}, {2, 3}, {-2, 4}};
        c->n_targets = 4; memcpy(c->targets, t, sizeof t);
      } else {
        const float t[5][2] = {{2, -4}, {2, 0}, {2, 4}, {0, 4}, {-2, 4}};
        c->n_targets = 5; memcpy(c->targets, t, sizeof t);
      }
    } break;
    case HRL_ANT_FLAGRUN:  // ant_flagrun_env.py:14-16,62,133-135,142
      c->world_size[0] = c->world_size[1] = 12; c->start_pos[2] = 0.25f; c->tol = 0.5f;
      c->n_scene_parts = 2; c->scene_parts_sum[0] = -6; c->scene_parts_sum[1] = 0;
      c->electricity_cost = 0; c->stall_torque_cost = 0; c->joints_at_limit_cost = 0;
      c->n_bins = 8; c->sensor_span = (float)HRL_PI_D; c->sensor_range = 4.f;  // ant_flagrun_env.py:15 (read when use_sensor)
      break;
    case HRL_ANT_MJ:  // envs/MjAnt.py:31 on the pybulletgym stadium ground
      c->world_size[0] = c->world_size[1] = 50; c->has_walls = 0; c->ground_z = 0.f; c->start_pos[2] = 0.75f; break;
    default: return set_err(HRL_E_INVALID, "unknown env_kind");
  }
  return HRL_OK;
}

static int food_obs_dim(const hrl_config* c) {  // 2 n_bins sector readings, or the xy of the nearest items (use_sensor=False)
  if (c->use_sensor) return 2 * c->n_bins;
  const int kf = c->n_bins < c->n_food ? c->n_bins : c->n_food, kp = c->n_bins < c->n_poison ? c->n_bins : c->n_poison;
  return 2 * kf + 2 * kp;
}
int hrl_obs_dim(const hrl_config* c) {
  if (!c) return -1;
  switch (c->env_kind) {
    case HRL_ANT_GATHER: return 26 + food_obs_dim(c);                    // ant_gather_env.py:54-55,179-196
    case HRL_ANT_MAZE: return 26 + (c->sense_target ? c->n_bins : 2) + (c->sense_walls ? c->n_bins : 0);  // ant_maze_bullet_env.py:54-57
    case HRL_ANT_FLAGRUN: return 28 + (c->flag_use_sensor ? c->n_bins : 0);  // ant_flagrun_env.py:52-54
    case HRL_ANT_MJ: return 29;                                          // MjAnt.py:15
    case HRL_ANT_MAZE_MJ: return 29 + 3 * c->n_bins + 1;                 // ant_maze_mj_env.py:50
    case HRL_POINT_GATHER: return 8 + food_obs_dim(c);                   // gather_base.py:54-55,170-187
  }
  return -1;
}
int hrl_act_dim(const hrl_config* c) { return !c ? -1 : (c->env_kind == HRL_POINT_GATHER ? 2 : 8); }

int hrl_host_layout(const hrl_config* c, size_t* off_rew, size_t* off_info, size_t* off_done, size_t* total) {
  if (!c || hrl_obs_dim(c) < 0 || c->num_envs <= 0) return set_err(HRL_E_INVALID, "bad config for hrl_host_layout");
  const size_t N = (size_t)c->num_envs, D = (size_t)hrl_obs_dim(c);
  const size_t o_rew = (N * D * sizeof(float) + 255) / 256 * 256;
  const size_t o_info = o_rew + (N * sizeof(float) + 255) / 256 * 256;
  const size_t o_done = o_info + N * 4 * sizeof(float);
  if (off_rew) *off_rew = o_rew;
  if (off_info) *off_info = o_info;
  if (off_done) *off_done = o_done;
  if (total) *total = (o_done + N + 255) / 256 * 256;
  return HRL_OK;
}

static int validate(const hrl_config* c) {
  if (!c) return set_err(HRL_E_INVALID, "null config");
  if (c->num_envs <= 0) return set_err(HRL_E_INVALID, "num_envs must be > 0");
  if (hrl_obs_dim(c) < 0) return set_err(HRL_E_INVALID, "unknown env_kind");
  if (hrl_obs_dim(c) > HRL_OBS_STAGE) return set_err(HRL_E_INVALID, "observation wider than 64");
  if (c->n_bins < 1 || c->n_bins > HRL_MAX_BINS) return set_err(HRL_E_INVALID, "n_bins out of range");
  if (c->n_food < 0 || c->n_food > 8 || c->n_poison < 0 || c->n_poison > 8) return set_err(HRL_E_INVALID, "n_food/n_poison out of range");
  // substeps == 0: a step runs the task layer on the current state only (how the parity tests feed the reference's
  // step-level golden vectors through the kernels)
  if (c->substeps < 0 || c->solver_iters < 0) return set_err(HRL_E_INVALID, "bad substeps/solver_iters");
  if (c->n_targets > HRL_MAX_TARGETS || c->flag_max_targets > 127) return set_err(HRL_E_INVALID, "too many targets");
  if (c->env_kind == HRL_POINT_GATHER && (c->item_contacts || !(c->robot_coll_dist > 0.f)))
    return set_err(HRL_E_INVALID, "PointGather cube colliders / contact-based pickup are not built");
  if (c->env_kind == HRL_ANT_GATHER && !(c->robot_coll_dist > 0.f) && !c->item_contacts)
    return set_err(HRL_E_INVALID, "robot_coll_dist <= 0 (contact-based pickup) needs item_contacts = 1");
  if (c->env_kind == HRL_ANT_FLAGRUN && c->flag_max_targets < 1 && !(c->flag_max_target_dist > 0.f))
    return set_err(HRL_E_INVALID, "flagrun needs max_targets > 0 or max_target_dist > 0 (ant_flagrun_env.py:17-18)");
  if (c->env_kind == HRL_ANT_FLAGRUN && c->flag_use_sensor && c->n_bins < 2) return set_err(HRL_E_INVALID, "flagrun sensor needs >= 2 bins");
  if ((c->env_kind == HRL_ANT_MAZE || c->env_kind == HRL_ANT_MAZE_MJ) && c->n_targets < 1) return set_err(HRL_E_INVALID, "maze needs targets");
  return HRL_OK;
}

// Lane mapping used by new handles: HRL_B200_LANES = 4 | 8 | 16 lanes per env (A/B runs); default HRL_DEFAULT_LANES.
#ifndef HRL_DEFAULT_LANES
#define HRL_DEFAULT_LANES 4
#endif
static int default_sub() {
  int lanes = HRL_DEFAULT_LANES;
  if (const char* e = getenv("HRL_B200_LANES")) lanes = atoi(e);
  return lanes == 16 ? 4 : (lanes == 8 ? 2 : 1);
}

int hrl_set_lanes_per_env(hrl_handle* h, int32_t lanes) {
  if (!h || (lanes != 4 && lanes != 8 && lanes != 16)) return set_err(HRL_E_INVALID, "lanes per env must be 4, 8 or 16");
  h->sub = lanes / 4;
  return HRL_OK;
}
int hrl_get_lanes_per_env(const hrl_handle* h) { return h ? 4 * h->sub : -1; }

int hrl_set_compact_rows(hrl_handle* h, int32_t on) {
  if (!h) return set_err(HRL_E_INVALID, "null handle");
  h->compact = on != 0;
  return HRL_OK;
}
// what launch_env runs: the compact rows exist only in the 4-lane Ant kernel
int hrl_get_compact_rows(const hrl_handle* h) {
  return h ? (h->cfg.env_kind != HRL_POINT_GATHER && h->sub == 1 && h->compact) : -1;
}

int hrl_destroy(hrl_handle* h) {
  if (!h) return HRL_OK;
  DeviceGuard guard(h->device);
  cudaFree(h->st.base); cudaFree(h->st.leg); cudaFree(h->st.items); cudaFree(h->st.miscf); cudaFree(h->st.misci);
  cudaFree(h->st.stats); cudaFree(h->d_bounds); cudaFree(h->st.fin_count);
  if (h->h_flag) cudaFreeHost(h->h_flag);
  cudaFree(h->s_act); cudaFree(h->s_obs);  // s_rew / s_info / s_done live inside the s_obs block
  delete h;
  return HRL_OK;
}

int hrl_create(const hrl_config* cfg, int32_t device, hrl_handle** out) {
  if (!out) return set_err(HRL_E_INVALID, "null out");
  *out = nullptr;
  int rc = validate(cfg);
  if (rc) return rc;
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0) return set_err(HRL_E_CUDA, "no CUDA device: this library has no CPU fallback");
  if (device < 0 || device >= ndev) return set_err(HRL_E_INVALID, "bad device index");
  ON_DEVICE(device);
  hrl_handle* h = new hrl_handle();
  memset(h, 0, sizeof *h);
  h->cfg = *cfg; h->device = device; h->N = cfg->num_envs; h->D = hrl_obs_dim(cfg); h->A = hrl_act_dim(cfg);
  const size_t N = (size_t)h->N;
#define ALLOC(p, bytes)                                                   \
  do {                                                                    \
    cudaError_t _e = cudaMalloc((void**)&(p), (bytes));                   \
    if (_e != cudaSuccess) { hrl_destroy(h); return cuda_fail(_e, "cudaMalloc"); } \
    cudaMemset((p), 0, (bytes));                                          \
  } while (0)
  ALLOC(h->st.base, N * 4 * sizeof(float4));
  ALLOC(h->st.leg, N * 4 * sizeof(float4));
  ALLOC(h->st.items, N * 8 * sizeof(float4));
  ALLOC(h->st.miscf, N * 2 * sizeof(float4));
  ALLOC(h->st.misci, N * 2 * sizeof(int4));
  ALLOC(h->st.stats, 4 * sizeof(unsigned long long));
  ALLOC(h->st.fin_count, sizeof(unsigned int));
#ifdef HRL_WARP_TIMES
  ALLOC(h->st.wt, (N + 1) * 4 * sizeof(unsigned long long));
#endif
  if (cudaHostAlloc((void**)&h->h_flag, 64, cudaHostAllocMapped) != cudaSuccess) { cudaGetLastError(); h->h_flag = nullptr; }
  else *h->h_flag = 0;
  ALLOC(h->d_bounds, 32 * sizeof(float));  // 7 x 4 bound lines (+ pad: the kernels fetch them with one 32-lane load)
  ALLOC(h->s_act, N * h->A * sizeof(float));
  {
    size_t off_rew, off_info, off_done, total;
    hrl_host_layout(cfg, &off_rew, &off_info, &off_done, &total);
    ALLOC(h->s_obs, total);
    h->s_rew = (float*)((char*)h->s_obs + off_rew);
    h->s_info = (float*)((char*)h->s_obs + off_info);
    h->s_done = (uint8_t*)h->s_obs + off_done;
    h->s_out_bytes = total;
  }
#undef ALLOC
  // late failures release the handle; *out is assigned last
#define CKH(call)                                                               \
  do {                                                                          \
    cudaError_t _e = (call);                                                    \
    if (_e != cudaSuccess) { hrl_destroy(h); return cuda_fail(_e, #call); }     \
  } while (0)
  float b[32];
  memset(b, 0, sizeof b);
  h->n_lines = scene_bounds(cfg, b);
  CKH(cudaMemcpy(h->d_bounds, b, sizeof b, cudaMemcpyHostToDevice));
  // opt in to the dynamic shared memory the ant kernels need; they live in shared memory and registers (hardly any
  // L1 traffic): take the whole carve-out
#define OPT_IN(FAM, SUB)                                                                                                      \
  CKH(cudaFuncSetAttribute(ant_env_kernel<FAM, SUB>, cudaFuncAttributeMaxDynamicSharedMemorySize,                             \
                           HRL_WARPS_PER_CTA * Map<SUB>::SMEM_FLOATS * (int)sizeof(float)));                                  \
  CKH(cudaFuncSetAttribute(ant_env_kernel<FAM, SUB>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared))
  OPT_IN(0, 0); OPT_IN(1, 0); OPT_IN(0, 1); OPT_IN(1, 1); OPT_IN(0, 2); OPT_IN(1, 2); OPT_IN(0, 4); OPT_IN(1, 4);
#undef OPT_IN
  // the fused-rollout instantiations: 2 warps per CTA + the policy weights (<= 35 KB) in shared memory, 2 CTAs per SM
  const int roll_smem = (HRL_ROLL_WARPS * Map<1>::SMEM_FLOATS + HRL_MLP_MAX_FLOATS) * (int)sizeof(float);
  CKH(cudaFuncSetAttribute(ant_env_kernel<0, 1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, roll_smem));
  CKH(cudaFuncSetAttribute(ant_env_kernel<1, 1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, roll_smem));
  CKH(cudaFuncSetAttribute(ant_env_kernel<0, 1, 1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CKH(cudaFuncSetAttribute(ant_env_kernel<1, 1, 1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  // normalized policy input: the observation mean and rstd (2 x obs_dim <= 2 x HRL_OBS_STAGE floats) behind the weights
  const int norm_smem = roll_smem + 2 * HRL_OBS_STAGE * (int)sizeof(float);
  CKH(cudaFuncSetAttribute(ant_env_kernel<0, 1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, norm_smem));
  CKH(cudaFuncSetAttribute(ant_env_kernel<1, 1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, norm_smem));
  CKH(cudaFuncSetAttribute(ant_env_kernel<0, 1, 2>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CKH(cudaFuncSetAttribute(ant_env_kernel<1, 1, 2>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  h->sub = default_sub();
  {
    // CTAs (= warps of 8 envs) per wave: 6 per SM with the 14-wide rows (37.5 KB), 7 with the compact ones (30.1 KB, ~7 %
    // more solver instructions).  Compact pays when it saves a whole wave: e.g. 16 384 envs = 2048 CTAs = 3 waves vs 2.
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
    const int ctas = (h->N + HRL_EPW - 1) / HRL_EPW, w6 = (ctas + 6 * n_sm - 1) / (6 * n_sm), w7 = (ctas + 7 * n_sm - 1) / (7 * n_sm);
    h->compact = w7 < w6;
    if (const char* e = getenv("HRL_B200_COMPACT")) h->compact = atoi(e) != 0;
  }
  // like the reference, reset() must be called before the first step(); an un-reset env has a
  // zero quaternion, produces a non-finite observation and is ended by the NaN guard
  CKH(cudaDeviceSynchronize());
#undef CKH
  *out = h;
  return HRL_OK;
}

static int launch_env(hrl_handle* h, int mode, int n_sub, const float* act, const uint8_t* mask, float* obs, float* rew,
                      uint8_t* done, float* info, float* term, cudaStream_t s, bool signal = false) {
  ON_DEVICE(h->device);
  DevState st = h->st;
  st.fin_flag = nullptr;
  if (signal && h->h_flag && h->cfg.env_kind != HRL_POINT_GATHER) {
    void* dflag = nullptr;
    if (cudaHostGetDevicePointer(&dflag, h->h_flag, 0) == cudaSuccess) { st.fin_flag = (unsigned int*)dflag; st.fin_seq = ++h->seq; }
    else cudaGetLastError();
  }
  if (h->cfg.env_kind == HRL_POINT_GATHER) {
    const int B = 16 * HRL_POINT_EPB, G = (h->N + HRL_POINT_EPB - 1) / HRL_POINT_EPB;
    point_env_kernel<0><<<G, B, 0, s>>>(h->cfg, h->st, act, mask, obs, rew, done, info, term, mode, n_sub, h->D);
  } else {
    const int T = 32 * HRL_WARPS_PER_CTA;
#define LAUNCH(FAM, SUB)                                                                                                     \
  do {                                                                                                                       \
    const int EPC = Map<SUB>::EPW * HRL_WARPS_PER_CTA, G = (h->N + EPC - 1) / EPC;                                           \
    const size_t smem = (size_t)HRL_WARPS_PER_CTA * Map<SUB>::SMEM_FLOATS * sizeof(float);                                   \
    ant_env_kernel<FAM, SUB><<<G, T, smem, s>>>(h->cfg, st, h->d_bounds, h->n_lines, act, mask, obs, rew, done, info, term,  \
                                                mode, n_sub, h->D);                                                          \
  } while (0)
    const bool gather = h->cfg.env_kind == HRL_ANT_GATHER;
    if (h->sub == 4) { if (gather) LAUNCH(0, 4); else LAUNCH(1, 4); }
    else if (h->sub == 2) { if (gather) LAUNCH(0, 2); else LAUNCH(1, 2); }
    else if (h->compact) { if (gather) LAUNCH(0, 0); else LAUNCH(1, 0); }
    else { if (gather) LAUNCH(0, 1); else LAUNCH(1, 1); }
#undef LAUNCH
  }
  g_launches++;
  CK(cudaGetLastError());
  if (st.fin_flag) {
    // poll the completion word (written after a system-scope fence by the last CTA); look at the
    // stream now and then so that a failed launch cannot hang the caller
    volatile unsigned int* f = h->h_flag;
    for (unsigned spins = 1; *f != st.fin_seq; spins++) {
      if ((spins & 0x3fff) == 0) {
        cudaError_t q = cudaStreamQuery(s);
        if (q == cudaErrorNotReady) continue;
        if (q != cudaSuccess) return cuda_fail(q, "env kernel");
        break;  // stream drained: results are visible
      }
#if defined(__x86_64__) || defined(__i386__)
      __builtin_ia32_pause();
#endif
    }
    std::atomic_thread_fence(std::memory_order_acquire);
  }
  return HRL_OK;
}

int hrl_reset(hrl_handle* h, const uint8_t* d_mask, float* d_obs, void* stream) {
  if (!h) return set_err(HRL_E_INVALID, "null handle");
  return launch_env(h, 2, 0, nullptr, d_mask, d_obs, nullptr, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

int hrl_step(hrl_handle* h, const float* d_actions, float* d_obs, float* d_rew, uint8_t* d_done, float* d_info,
             float* d_terminal_obs, void* stream) {
  if (!h || !d_actions || !d_obs || !d_rew || !d_done) return set_err(HRL_E_INVALID, "null argument to hrl_step");
  return launch_env(h, 0, 0, d_actions, nullptr, d_obs, d_rew, d_done, d_info, d_terminal_obs, (cudaStream_t)stream);
}

/* non-NULL when `p` is pinned host memory the device can address directly (UVA): the device alias.
 * Pinned buffers are long-lived in a stepping loop, so positive answers are cached per handle. */
static void* mapped_alias(hrl_handle* h, const void* p, bool cache = true) {
  if (cache)
    for (int i = 0; i < h->alias_n; i++)
      if (h->alias_key[i] == p) return h->alias_val[i];
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  // pinned host memory: its device alias; device memory (a caller may keep `info` on the device): the pointer itself
  void* d = (a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeDevice) ? a.devicePointer : nullptr;
  if (d && cache) {
    if (h->alias_n == 12) h->alias_n = 0;  // tiny ring: evict everything
    h->alias_key[h->alias_n] = p; h->alias_val[h->alias_n] = d; h->alias_n++;
  }
  return d;
}

int hrl_set_host_mode(hrl_handle* h, int32_t mode) {
  if (!h || mode < HRL_HOST_AUTO || mode > HRL_HOST_ZEROCOPY) return set_err(HRL_E_INVALID, "bad argument to hrl_set_host_mode");
  h->host_mode = mode;
  h->alias_n = 0;  // also forgets the cached pinned-buffer aliases (call this after freeing such a buffer)
  return HRL_OK;
}

int hrl_step_host(hrl_handle* h, const float* h_actions, float* h_obs, float* h_rew, uint8_t* h_done, float* h_info,
                  void* stream) {
  if (!h || !h_actions || !h_obs || !h_rew || !h_done) return set_err(HRL_E_INVALID, "null argument to hrl_step_host");
  cudaStream_t s = (cudaStream_t)stream;
  ON_DEVICE(h->device);
  const size_t N = (size_t)h->N;
  // inputs: pinned actions are read by the kernel in place; anything else is copied H2D first
  const float* d_act = nullptr;
  // (action arrays come and go with the caller: asked afresh every step, never cached)
  if (h->host_mode != HRL_HOST_COPY) d_act = (const float*)mapped_alias(h, h_actions, false);
  if (!d_act) {
    CK(cudaMemcpyAsync(h->s_act, h_actions, N * h->A * sizeof(float), cudaMemcpyHostToDevice, s));
    d_act = h->s_act;
  }
  if (h->host_mode != HRL_HOST_COPY) {
    // zero-copy outputs: the kernel writes its results to pinned host memory over PCIe while it computes, so the
    // transfer overlaps the step instead of following it; completion = a word the last CTA publishes
    float* o = (float*)mapped_alias(h, h_obs);
    float* r = (float*)mapped_alias(h, h_rew);
    uint8_t* d = (uint8_t*)mapped_alias(h, h_done);
    float* i = h_info ? (float*)mapped_alias(h, h_info) : nullptr;
    if (o && r && d && (i || !h_info)) {
      const bool poll = h->h_flag && h->cfg.env_kind != HRL_POINT_GATHER;
      int rc = launch_env(h, 0, 0, d_act, nullptr, o, r, d, i, nullptr, s, poll);
      if (rc) return rc;
      if (!poll) CK(cudaStreamSynchronize(s));
      return HRL_OK;
    }
    if (h->host_mode == HRL_HOST_ZEROCOPY) return set_err(HRL_E_INVALID, "zero-copy host mode needs pinned (page-locked) buffers");
  }
  int rc = launch_env(h, 0, 0, d_act, nullptr, h->s_obs, h->s_rew, h->s_done, h->s_info, nullptr, s);
  if (rc) return rc;
  size_t off_rew, off_info, off_done, total;
  hrl_host_layout(&h->cfg, &off_rew, &off_info, &off_done, &total);
  const bool info_on_device = h_info && mapped_alias(h, h_info) == (void*)h_info;   // device pointer: no copy wanted
  if (info_on_device) {
    CK(cudaMemcpyAsync(h_info, h->s_info, N * 4 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    h_info = nullptr;
  }
  if (h_info && (char*)h_rew == (char*)h_obs + off_rew && (char*)h_info == (char*)h_obs + off_info &&
      (char*)h_done == (char*)h_obs + off_done) {
    CK(cudaMemcpyAsync(h_obs, h->s_obs, off_done + N, cudaMemcpyDeviceToHost, s));  // packed layout: one copy
  } else {
    CK(cudaMemcpyAsync(h_obs, h->s_obs, N * h->D * sizeof(float), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(h_rew, h->s_rew, N * sizeof(float), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(h_done, h->s_done, N, cudaMemcpyDeviceToHost, s));
    if (h_info) CK(cudaMemcpyAsync(h_info, h->s_info, N * 4 * sizeof(float), cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  return HRL_OK;
}

// AntFlagrunBulletEnv.next_target() as a public call (ant_flagrun_env.py:112-120; the step calls it by itself on
// reach / timeout): pops the next goal of the masked envs, resets `_rewarded`, restarts the potential from the stale
// walk_target_dist (quirk Q3).  Envs whose goal list is empty keep their target (the reference raises IndexError).
__global__ void flag_next_kernel(const __grid_constant__ hrl_config cfg, DevState st, const uint8_t* __restrict__ mask) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= cfg.num_envs || (mask && !mask[e])) return;
  const float4 b0 = st.base[e * 4 + 0], b2 = st.base[e * 4 + 2], b3 = st.base[e * 4 + 3];
  float4 m0 = st.miscf[e * 2 + 0];
  int4 i0 = st.misci[e * 2 + 0], i1 = st.misci[e * 2 + 1];
  TaskRegs T;
  T.initial_z = b0.w; T.potential = b2.w; T.wtd = b3.w; T.tx = m0.x; T.ty = m0.y; T.ret = m0.z; T.ret_sum = m0.w;
  T.t = i0.x; T.episode = i0.y; T.steps_total = i0.z; T.goals_left = i0.w; T.since = i1.x; T.rewarded = i1.y; T.gen = i1.z;
  if (!flag_next(cfg, (uint32_t)(cfg.env_index_offset + e), T, b0.x, b0.y, 0)) return;
  st.base[e * 4 + 2] = make_float4(b2.x, b2.y, b2.z, T.potential);
  st.miscf[e * 2 + 0] = make_float4(T.tx, T.ty, m0.z, m0.w);
  st.misci[e * 2 + 0] = make_int4(i0.x, i0.y, i0.z, T.goals_left);
  st.misci[e * 2 + 1] = make_int4(i1.x, T.rewarded, i1.z, i1.w);  // steps_since_goal_change is the step's business (:190,201), not next_target's
}

int hrl_flagrun_next_target(hrl_handle* h, const uint8_t* d_mask, void* stream) {
  if (!h) return set_err(HRL_E_INVALID, "null handle");
  if (h->cfg.env_kind != HRL_ANT_FLAGRUN) return set_err(HRL_E_INVALID, "hrl_flagrun_next_target: not an AntFlagrun handle");
  ON_DEVICE(h->device);
  flag_next_kernel<<<(h->N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->cfg, h->st, d_mask);
  g_launches++;
  CK(cudaGetLastError());
  return HRL_OK;
}

/* Fused rollout: T env steps in ONE launch with an in-kernel MLP policy (see mlp_policy / mlp_policy16); with the
 * observation statistics, the ROLL = 2 instantiations feed the policy the normalized observation (norm_obs).  The one
 * launch path of hrl_rollout_mlp* (P = 1, per-step buffers) and hrl_evaluate_mlp (P members, per-env results): the
 * callers check their own buffers, the policy arguments are checked here. */
static int launch_rollout(hrl_handle* h, const char* fn, int32_t T, int32_t P, const float* d_weights, int32_t hidden, float sigma,
                          const float* d_sigma, uint64_t noise_seed, const float* d_obs_mean, const float* d_obs_rstd, float obs_clip,
                          float* d_obs, float* d_act, float* d_rew, uint8_t* d_done, float* d_info, float* d_terminal_obs,
                          float* d_ret, int32_t* d_len, uint8_t* d_finished, void* stream) {
  if (!d_weights) return set_err(HRL_E_INVALID, fn, "d_weights is NULL");
  if (hidden != 32 && hidden != 64) return set_err(HRL_E_INVALID, fn, "hidden width must be 32 or 64");
  if (!(sigma >= 0.f)) return set_err(HRL_E_INVALID, fn, "sigma must be >= 0");
  if (!d_obs_mean != !d_obs_rstd) return set_err(HRL_E_INVALID, fn, "d_obs_mean and d_obs_rstd must both be given or both be NULL");
  const bool norm = d_obs_mean != nullptr;
  if (norm && !(obs_clip > 0.f && isfinite(obs_clip))) return set_err(HRL_E_INVALID, fn, "obs_clip must be finite and > 0");
  ON_DEVICE(h->device);
  DevState st = h->st;
  st.fin_flag = nullptr;
  RollArgs ra;
  ra.T = T; ra.H = hidden; ra.w = d_weights; ra.sigma = sigma; ra.sigma_v = d_sigma; ra.seed = noise_seed; ra.act_out = d_act;
  ra.obs_mean = d_obs_mean; ra.obs_rstd = d_obs_rstd; ra.obs_clip = obs_clip;
  ra.m_envs = h->N / P; ra.ev_ret = d_ret; ra.ev_len = d_len; ra.ev_fin = d_finished;
  const int nw = h->D * hidden + hidden + hidden * hidden + hidden + hidden * h->A + h->A + (norm ? 2 * h->D : 0);
  cudaStream_t s = (cudaStream_t)stream;
  if (h->cfg.env_kind == HRL_POINT_GATHER) {
    const int G = (h->N + HRL_POINT_EPB - 1) / HRL_POINT_EPB;
    const size_t smem = ((size_t)HRL_POINT_EPB * 64 + nw) * sizeof(float);
    if (norm)
      point_env_kernel<2><<<G, 16 * HRL_POINT_EPB, smem, s>>>(h->cfg, st, nullptr, nullptr, d_obs, d_rew, d_done, d_info, d_terminal_obs, 0, 0,
                                                              h->D, ra);
    else
      point_env_kernel<1><<<G, 16 * HRL_POINT_EPB, smem, s>>>(h->cfg, st, nullptr, nullptr, d_obs, d_rew, d_done, d_info, d_terminal_obs, 0, 0,
                                                              h->D, ra);
  } else {
    const int Tn = 32 * HRL_ROLL_WARPS, EPC = Map<1>::EPW * HRL_ROLL_WARPS, G = (h->N + EPC - 1) / EPC;
    const size_t smem = ((size_t)HRL_ROLL_WARPS * Map<1>::SMEM_FLOATS + nw) * sizeof(float);
#define ROLL_LAUNCH(FAM, R)                                                                                                 \
  ant_env_kernel<FAM, 1, R><<<G, Tn, smem, s>>>(h->cfg, st, h->d_bounds, h->n_lines, nullptr, nullptr, d_obs, d_rew, d_done, d_info, \
                                                d_terminal_obs, 0, 0, h->D, ra)
    if (h->cfg.env_kind == HRL_ANT_GATHER) {
      if (norm) ROLL_LAUNCH(0, 2); else ROLL_LAUNCH(0, 1);
    } else {
      if (norm) ROLL_LAUNCH(1, 2); else ROLL_LAUNCH(1, 1);
    }
#undef ROLL_LAUNCH
  }
  g_launches++;
  CK(cudaGetLastError());
  return HRL_OK;
}

int hrl_rollout_mlp_norm(hrl_handle* h, int32_t T, const float* d_weights, int32_t hidden, float sigma, const float* d_sigma,
                         uint64_t noise_seed, const float* d_obs_mean, const float* d_obs_rstd, float obs_clip, float* d_obs,
                         float* d_act, float* d_rew, uint8_t* d_done, float* d_info, float* d_terminal_obs, void* stream) {
  if (!h || T < 1 || !d_weights || !d_obs || !d_act || !d_rew || !d_done) return set_err(HRL_E_INVALID, "bad argument to hrl_rollout_mlp");
  return launch_rollout(h, "hrl_rollout_mlp_norm", T, 1, d_weights, hidden, sigma, d_sigma, noise_seed, d_obs_mean, d_obs_rstd, obs_clip,
                        d_obs, d_act, d_rew, d_done, d_info, d_terminal_obs, nullptr, nullptr, nullptr, stream);
}

int hrl_evaluate_mlp(hrl_handle* h, int32_t T, int32_t P, const float* d_weights, int32_t hidden, float sigma, const float* d_sigma,
                     uint64_t noise_seed, const float* d_obs_mean, const float* d_obs_rstd, float obs_clip, float* d_ret,
                     int32_t* d_len, uint8_t* d_finished, void* stream) {
  static const char* fn = "hrl_evaluate_mlp";
  if (!h) return set_err(HRL_E_INVALID, fn, "null handle");
  if (T < 1) return set_err(HRL_E_INVALID, fn, "T must be >= 1");
  if (P < 1) return set_err(HRL_E_INVALID, fn, "the member count P must be >= 1");
  if (!d_ret || !d_len || !d_finished) return set_err(HRL_E_INVALID, fn, "d_ret, d_len and d_finished must all be given");
  if (P > 1) {
    // a CTA stages ONE member's weights: it must not straddle two members
    const int epc = h->cfg.env_kind == HRL_POINT_GATHER ? HRL_POINT_EPB : Map<1>::EPW * HRL_ROLL_WARPS;
    char msg[200];
    if (h->N % P) {
      snprintf(msg, sizeof msg, "num_envs %d is not a multiple of the member count %d", h->N, P);
      return set_err(HRL_E_INVALID, fn, msg);
    }
    if ((h->N / P) % epc) {
      snprintf(msg, sizeof msg, "envs per member (num_envs / P = %d) must be a multiple of %d for this env family when P > 1", h->N / P, epc);
      return set_err(HRL_E_INVALID, fn, msg);
    }
  }
  return launch_rollout(h, fn, T, P, d_weights, hidden, sigma, d_sigma, noise_seed, d_obs_mean, d_obs_rstd, obs_clip, nullptr, nullptr,
                        nullptr, nullptr, nullptr, nullptr, d_ret, d_len, d_finished, stream);
}

int hrl_rollout_mlp_ex(hrl_handle* h, int32_t T, const float* d_weights, int32_t hidden, float sigma, const float* d_sigma,
                       uint64_t noise_seed, float* d_obs, float* d_act, float* d_rew, uint8_t* d_done, float* d_info,
                       float* d_terminal_obs, void* stream) {
  return hrl_rollout_mlp_norm(h, T, d_weights, hidden, sigma, d_sigma, noise_seed, nullptr, nullptr, 0.f, d_obs, d_act, d_rew, d_done,
                              d_info, d_terminal_obs, stream);
}

int hrl_rollout_mlp(hrl_handle* h, int32_t T, const float* d_weights, int32_t hidden, float sigma, uint64_t noise_seed, float* d_obs,
                    float* d_act, float* d_rew, uint8_t* d_done, void* stream) {
  return hrl_rollout_mlp_ex(h, T, d_weights, hidden, sigma, nullptr, noise_seed, d_obs, d_act, d_rew, d_done, nullptr, nullptr, stream);
}

int hrl_observe(hrl_handle* h, float* d_obs, void* stream) {
  if (!h || !d_obs) return set_err(HRL_E_INVALID, "null argument to hrl_observe");
  return launch_env(h, 3, 0, nullptr, nullptr, d_obs, nullptr, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

int hrl_substeps(hrl_handle* h, const float* d_actions, int32_t n_sub, void* stream) {
  if (!h || !d_actions || n_sub < 0) return set_err(HRL_E_INVALID, "bad argument to hrl_substeps");
  return launch_env(h, 1, n_sub, d_actions, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

int hrl_get_state(hrl_handle* h, float* d_f, int32_t* d_i, void* stream) {
  if (!h || !d_f || !d_i) return set_err(HRL_E_INVALID, "null argument to hrl_get_state");
  ON_DEVICE(h->device);
  get_state_kernel<<<(h->N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->N, h->st, d_f, d_i);
  g_launches++;
  CK(cudaGetLastError());
  return HRL_OK;
}
int hrl_set_state(hrl_handle* h, const float* d_f, const int32_t* d_i, void* stream) {
  if (!h || !d_f || !d_i) return set_err(HRL_E_INVALID, "null argument to hrl_set_state");
  ON_DEVICE(h->device);
  set_state_kernel<<<(h->N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->N, h->st, d_f, d_i);
  g_launches++;
  CK(cudaGetLastError());
  return HRL_OK;
}

int hrl_gather_sensor(int32_t M, int32_t n_bins, float sensor_range, float sensor_span, const float* d_xy,
                      const float* d_yaw, const float* d_items, float* d_food, float* d_poison, int32_t* d_bins,
                      void* stream) {
  if (M < 0 || n_bins < 1 || n_bins > HRL_MAX_BINS || !d_xy || !d_yaw || !d_items || !d_food || !d_poison)
    return set_err(HRL_E_INVALID, "bad argument to hrl_gather_sensor");
  if (M == 0) return HRL_OK;
  const int T = 256, G = (M * 16 + T - 1) / T;
  gather_sensor_kernel<<<G, T, 0, (cudaStream_t)stream>>>(M, n_bins, sensor_range, sensor_span, d_xy, d_yaw, d_items, d_food, d_poison, d_bins);
  g_launches++;
  CK(cudaGetLastError());
  return HRL_OK;
}

int hrl_sense_walls(int32_t M, int32_t n_bins, float span, float range, int32_t n_lines, const float* d_bounds,
                    const float* d_xy, const float* d_yaw, float* d_out, void* stream) {
  if (M < 0 || n_bins < 1 || n_bins > HRL_MAX_BINS || n_lines < 0 || !d_bounds || !d_xy || !d_yaw || !d_out)
    return set_err(HRL_E_INVALID, "bad argument to hrl_sense_walls");
  if (M == 0) return HRL_OK;
  const int T = 128, G = (M * n_bins + T - 1) / T;
  sense_walls_kernel<<<G, T, 0, (cudaStream_t)stream>>>(M, n_bins, span, range, n_lines, d_bounds, d_xy, d_yaw, d_out);
  g_launches++;
  CK(cudaGetLastError());
  return HRL_OK;
}

/* GAE(lambda) over a rollout buffer (gae_kernel, hrl_gae.cuh); runs on the current device. */
int hrl_gae(int32_t T, int32_t N, float gamma, float lam, const float* d_rew, const uint8_t* d_done, const float* d_info,
            const float* d_values, const float* d_terminal_values, float* d_adv, float* d_ret, void* stream) {
  if (T < 1 || N < 1 || !d_rew || !d_done || !d_values || !d_adv) return set_err(HRL_E_INVALID, "bad argument to hrl_gae");
  if (!(gamma >= 0.f && gamma <= 1.f) || !(lam >= 0.f && lam <= 1.f))
    return set_err(HRL_E_INVALID, "hrl_gae: gamma and lam must lie in [0, 1]");
  if (!d_info != !d_terminal_values)
    return set_err(HRL_E_INVALID, "hrl_gae: d_info and d_terminal_values must both be given or both be NULL");
  int dev = 0, sms = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int W = gae_warps(T, N, sms), L = (T + W - 1) / W;
  gae_kernel<<<(N + 31) / 32, 32 * W, 0, (cudaStream_t)stream>>>(T, N, L, gamma, gamma * lam, d_rew, d_done, d_info, d_values,
                                                                 d_terminal_values, d_adv, d_ret);
  g_launches++;
  CK(cudaGetLastError());
  return HRL_OK;
}

// CTAs of the one-cluster normalization kernels (hrl_normalize.cuh) on the current device: 16 (a non-portable cluster
// size) where the device can co-schedule them, else the portable 8.  Cached per device.
static int norm_cluster_size(int dev) {
  static std::atomic<int> cache[64];
  if (dev >= 0 && dev < 64 && cache[dev].load()) return cache[dev].load();
  int best = 8;
  const void* kernels[2] = {(const void*)obs_moments_kernel, (const void*)return_moments_kernel};
  bool ok16 = true;
  for (const void* k : kernels) {
    ok16 = ok16 && cudaFuncSetAttribute(k, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(16); cfg.blockDim = dim3(HRL_NORM_THREADS);
    cudaLaunchAttribute a;
    a.id = cudaLaunchAttributeClusterDimension;
    a.val.clusterDim.x = 16; a.val.clusterDim.y = 1; a.val.clusterDim.z = 1;
    cfg.attrs = &a; cfg.numAttrs = 1;
    int n = 0;
    ok16 = ok16 && cudaOccupancyMaxActiveClusters(&n, k, &cfg) == cudaSuccess && n >= 1;
  }
  cudaGetLastError();  // a refused query is an answer, not an error of the next launch
  if (ok16) best = 16;
  if (dev >= 0 && dev < 64) cache[dev].store(best);
  return best;
}

extern "C++" {  // a template cannot have C linkage
template <typename... Exp, typename... Act>
static cudaError_t launch_cluster(void (*kernel)(Exp...), int C, cudaStream_t s, Act&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(C); cfg.blockDim = dim3(HRL_NORM_THREADS); cfg.dynamicSmemBytes = 0; cfg.stream = s;
  cudaLaunchAttribute a;
  a.id = cudaLaunchAttributeClusterDimension;
  a.val.clusterDim.x = C; a.val.clusterDim.y = 1; a.val.clusterDim.z = 1;
  cfg.attrs = &a; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Act>(args)...);
}
}

/* Running observation statistics (obs_moments_kernel, hrl_normalize.cuh); runs on the current device. */
int hrl_obs_moments(int32_t M, int32_t D, const float* d_x, double* d_moments, float eps, float* d_mean_f, float* d_rstd_f,
                    void* stream) {
  if (M < 1 || D < 1 || D > HRL_NORM_MAX_D || !d_x || !d_moments || !d_mean_f || !d_rstd_f)
    return set_err(HRL_E_INVALID, "bad argument to hrl_obs_moments");
  if (!(eps > 0.f)) return set_err(HRL_E_INVALID, "hrl_obs_moments: eps must be > 0");
  int dev = 0;
  CK(cudaGetDevice(&dev));
  const int C = norm_cluster_size(dev);
  CK(launch_cluster(obs_moments_kernel, C, (cudaStream_t)stream, (int)M, (int)D, d_x, d_moments, eps, d_mean_f, d_rstd_f));
  g_launches++;
  return HRL_OK;
}

/* Return-based reward scaling (return_scan_kernel, return_moments_kernel, reward_apply_kernel); current device. */
int hrl_reward_scale(int32_t T, int32_t N, float gamma, float clip, float eps, const float* d_rew, const uint8_t* d_done,
                     double* d_returns, double* d_ret_moments, double* d_work, float* d_out, void* stream) {
  if (T < 1 || N < 1 || !d_rew || !d_done || !d_returns || !d_ret_moments || !d_work || !d_out)
    return set_err(HRL_E_INVALID, "bad argument to hrl_reward_scale");
  if (!(gamma >= 0.f && gamma <= 1.f)) return set_err(HRL_E_INVALID, "hrl_reward_scale: gamma must lie in [0, 1]");
  if (!(clip > 0.f) || !(eps > 0.f)) return set_err(HRL_E_INVALID, "hrl_reward_scale: clip and eps must be > 0");
  int dev = 0, sms = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int C = norm_cluster_size(dev);
  cudaStream_t s = (cudaStream_t)stream;
  return_scan_kernel<<<(N + 255) / 256, 256, 0, s>>>(T, N, (double)gamma, d_rew, d_done, d_returns, d_out);
  g_launches++;
  CK(cudaGetLastError());
  CK(launch_cluster(return_moments_kernel, C, s, (int)T, (int)N, eps, (const float*)d_out, d_ret_moments, d_work));
  g_launches++;
  const int gx = (N + 255) / 256, gy = (int)std::min<long long>(T, std::max<long long>(1, 8LL * sms / gx));
  reward_apply_kernel<<<dim3(gx, gy), 256, 0, s>>>(T, N, clip, d_rew, d_work, d_out);
  g_launches++;
  CK(cudaGetLastError());
  return HRL_OK;
}

// Measurement aid: everything enqueued on `stream` after this call waits on the device until the 32-bit word at
// d_flag (pinned host memory the device can address, or device memory) equals `expect`, or `timeout_ns` elapses.
// bench.py queues a whole batch of (L2 flush, event, step, event) behind one gate and then opens it, so that the
// per-step event pairs never contain a host-side launch gap.
__global__ void gate_kernel(const volatile unsigned int* flag, unsigned int expect, unsigned long long timeout_ns) {
  unsigned long long t0, t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  while (*flag != expect) {
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    if (t - t0 > timeout_ns) break;
    __nanosleep(500);
  }
}
int hrl_stream_gate(const uint32_t* d_flag, uint32_t expect, uint64_t timeout_ns, void* stream) {
  if (!d_flag) return set_err(HRL_E_INVALID, "null flag for hrl_stream_gate");
  gate_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(d_flag, expect, (unsigned long long)timeout_ns);
  g_launches++;
  CK(cudaGetLastError());
  return HRL_OK;
}

#ifdef HRL_DEBUG_CONTACTS
int hrl_debug_contacts(float* d_buf) {  // debugging build: where the kernels dump the candidate lists (NULL: off)
  CK(cudaMemcpyToSymbol(g_dbg_contacts, &d_buf, sizeof d_buf));
  return HRL_OK;
}
#endif
#ifdef HRL_WARP_TIMES
/* profiling build (tools/warp_times.py): per-warp records of the LAST ant-kernel launch, 4 x u64 per warp */
int hrl_debug_warp_times(hrl_handle* h, unsigned long long* out, int n_warps) {
  if (!h || !out) return set_err(HRL_E_INVALID, "null argument");
  ON_DEVICE(h->device);
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out, h->st.wt, (size_t)n_warps * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return HRL_OK;
}
#endif

/* instrumentation for the FLOP model (bench.py roofline): contacts, limit rows, env-substeps */
int hrl_get_stats(hrl_handle* h, unsigned long long out[4], int reset) {
  if (!h || !out) return set_err(HRL_E_INVALID, "null argument to hrl_get_stats");
  ON_DEVICE(h->device);
  CK(cudaMemcpy(out, h->st.stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  if (reset) CK(cudaMemset(h->st.stats, 0, 4 * sizeof(unsigned long long)));
  return HRL_OK;
}

}  // extern "C"
