// sm_100a kernels + C ABI of the TriFinger MDP hot path (see include/leibniz_b200.h).
//
// Two launches per env step, both env-major and HBM-bound (no tensor cores: the path is
// elementwise, ~2 FLOP/B):
//   pre_physics_kernel   ordered mask compaction (decoupled look-back) + reset / goal-reset
//                        sampling and scatter + action store + action->torque; tile slabs by TMA bulk copy
//   post_physics_kernel  obs/states fill + scale_transform, six reward terms, termination,
//                        step counters / timeouts / dones, episode statistics; one lane per output column
// Reference paths are relative to /root/reference/leibnizgym/.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>

#include "lg_device.cuh"
#include "lg_post.cuh"
#include "lg_pre.cuh"

namespace lg {

// ---- batched primitives -------------------------------------------------------------------------
__global__ void quat_mul_kernel(const float* a, const float* b, float* out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 qa = reinterpret_cast<const float4*>(a)[i], qb = reinterpret_cast<const float4*>(b)[i];
  const Quat r = quat_mul(Quat{qa.x, qa.y, qa.z, qa.w}, Quat{qb.x, qb.y, qb.z, qb.w});
  reinterpret_cast<float4*>(out)[i] = make_float4(r.x, r.y, r.z, r.w);
}
__global__ void quat_diff_kernel(const float* a, const float* b, float* out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 qa = reinterpret_cast<const float4*>(a)[i], qb = reinterpret_cast<const float4*>(b)[i];
  out[i] = quat_diff_rad(Quat{qa.x, qa.y, qa.z, qa.w}, Quat{qb.x, qb.y, qb.z, qb.w});
}
template <int OP>
__global__ void rowwise_kernel(const float* x, const float* lo, const float* hi, float* out, int64_t total, int dims) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % dims);
  const float l = lo[c], h = hi[c], v = x[i];
  if (OP == 0) out[i] = scale_transform(v, (l + h) * 0.5f, h - l);
  else if (OP == 1) out[i] = unscale_transform(v, l, h);
  else out[i] = saturate(v, l, h);
}
__global__ void lgsk_kernel(const float* x, float scale, float* out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = lgsk(x[i], scale);
}
__global__ void keypoints_kernel(const float* pose, float size, float* out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 8) return;
  const int64_t e = i >> 3;
  const int k = (int)(i & 7);
  const float* p = pose + e * 7;
  const float h = size * 0.5f;
  const float vx = (k & 1) ? h : -h, vy = (k & 2) ? h : -h, vz = (k & 4) ? h : -h;
  float rx, ry, rz;
  quat_rotate(Quat{p[3], p[4], p[5], p[6]}, vx, vy, vz, rx, ry, rz);
  out[i * 3] = p[0] + rx; out[i * 3 + 1] = p[1] + ry; out[i * 3 + 2] = p[2] + rz;
}

// Stand-in for the simulator's rigid-body integration of the (gravity-free, collision-free) goal body of the
// moving-goal task: semi-implicit Euler over dt on root rows [n, 13] = pos 3 | quat xyzw 4 | lin vel 3 | ang vel 3,
//   p += v dt;   q <- normalize(exp(w dt / 2) (x) q)   (world-frame angular velocity, quaternion exponential).
__global__ void integrate_rows_kernel(float* rows, int64_t row_stride, float dt, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float* r = rows + i * row_stride;
  const float wx = r[10], wy = r[11], wz = r[12];
  r[0] = r[0] + r[7] * dt; r[1] = r[1] + r[8] * dt; r[2] = r[2] + r[9] * dt;
  const float w = norm3(wx, wy, wz);
  if (!(w > 0.0f)) return;   // not turning: the orientation stays bit-identical
  const float half = 0.5f * w * dt;
  const float k = w > 1e-12f ? __fdiv_rn(sinf(half), w) : 0.5f * dt;   // sin(half)/w -> dt/2 as w -> 0
  const Quat dq{wx * k, wy * k, wz * k, cosf(half)};
  Quat q = quat_mul(dq, Quat{r[3], r[4], r[5], r[6]});
  const float nrm = sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w);
  const float inv = __frcp_rn(fmaxf(nrm, 1e-12f));
  r[3] = q.x * inv; r[4] = q.y * inv; r[5] = q.z * inv; r[6] = q.w * inv;
}

// exhaustive check of div_by_const's contract for one (span, rcp): all 2^32 numerators.
// out[0] = in-window numerators that are not bit-identical to IEEE division (must be 0);
// out[1] = worst ulp distance for 0 < |x| < 2^-100 (must be <= 1); out[2] = huge/inf numerators not flagged.
__global__ void selftest_division_kernel(float span, float rcp, unsigned long long* out) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  unsigned long long bad = 0, unflagged = 0;
  unsigned int worst = 0;
  for (uint64_t bits = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; bits < (1ull << 32); bits += stride) {
    const float x = __uint_as_float((uint32_t)bits);
    float amax = 0.0f;
    const float a = div_by_const(x, span, rcp, amax), b = __fdiv_rn(x, span);
    const float ax = fabsf(x);
    if (x != x) continue;                                   // nan in, nan out on both paths
    if (!(ax < kDivSafeMax)) { if (amax < kDivSafeMax) ++unflagged; continue; }
    if (ax == 0.0f) { if (a != 0.0f) ++bad; continue; }
    if (ax >= 7.8886091e-31f /* 2^-100 */) { if (__float_as_uint(a) != __float_as_uint(b)) ++bad; continue; }
    const int d = abs((int)(__float_as_uint(a) & 0x7fffffffu) - (int)(__float_as_uint(b) & 0x7fffffffu));
    worst = max(worst, (unsigned int)d);
  }
  if (bad) atomicAdd(out, bad);
  if (worst) atomicMax(out + 1, (unsigned long long)worst);
  if (unflagged) atomicAdd(out + 2, unflagged);
}

}  // namespace lg

// =========================================================================================
// C ABI
// =========================================================================================
namespace {
thread_local std::string g_error;
int fail(int code, const std::string& msg) { g_error = msg; return code; }
// What this thread launched last (lg_pre_physics_chained chains itself to a directly preceding lg_post_physics only).
thread_local struct { void* stream; bool post; } g_prev = {nullptr, false};
int check_launch(const char* what) {
  g_prev.post = false;
  const cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(LG_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(err));
  return LG_OK;
}
bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

bool env_flag(const char* name) { const char* v = std::getenv(name); return v && v[0] && v[0] != '0'; }
int env_int(const char* name, int dflt) { const char* v = std::getenv(name); return v ? std::atoi(v) : dflt; }

int sm_count() {
  static const int n = [] {
    int dev = 0, v = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v > 0 ? v : 148;
  }();
  return n;
}

// Programmatic dependent launch: bit 1 = the post-physics kernel after whatever precedes it, bit 0 = the pre-physics
// kernel after a post-physics kernel, when the caller vouches for its inputs (lg_pre_physics_chained).  LG_PDL=0 /
// LG_NO_PDL=1 switch both off, LG_PDL=2 the second.  lg_pre_physics itself is always launched in stream order.
int pdl_mode() { static const int m = env_flag("LG_NO_PDL") ? 0 : (env_int("LG_PDL", 3) & 3); return m; }

// Launch with programmatic stream serialisation (PDL) unless LG_NO_PDL is set.
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(bool pdl, void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Envs per CTA of the post-physics kernel: 32 when the grid needs several waves anyway, otherwise the
// smallest tile that still fits one wave (4 CTAs per SM) so that all SMs carry the same load.
int pick_tile_envs(int64_t n) {
  static const int forced = env_int("LG_TILE_ENVS", 0);
  if (forced == 32 || forced == 28 || forced == 24 || forced == 16) return forced;
  const int64_t capacity = (int64_t)sm_count() * 4;
  if ((n + 31) / 32 > capacity) return 32;
  const int cands[] = {16, 24, 28, 32};
  for (int e : cands)
    if ((n + e - 1) / e <= capacity) return e;
  return 32;
}

int validate(const LgParams* P, const LgSimState* S, const LgBuffers* B, bool need_states) {
  if (!P || !S || !B) return fail(LG_ERR_BAD_ARG, "null LgParams / LgSimState / LgBuffers");
  if (P->num_envs <= 0) return fail(LG_ERR_BAD_ARG, "num_envs must be positive");
  if (P->num_envs >= (1 << 23)) return fail(LG_ERR_BAD_ARG, "num_envs per shard must be < 2^23");
  if (P->action_dim != 9 && P->action_dim != 18) return fail(LG_ERR_BAD_ARG, "action_dim must be 9 or 18");
  if (!S->dof_state || !S->root_state || !S->rigid_body) return fail(LG_ERR_BAD_ARG, "null simulator tensor");
  if (!B->obs || !B->action || !B->reward || !B->reset || !B->goal_reset || !B->successes || !B->steps_count ||
      !B->goal_pose || !B->goal_movement || !B->history || !B->control)
    return fail(LG_ERR_BAD_ARG, "null env buffer");
  if (need_states && P->asymmetric_obs && (!B->states || !S->dof_force || !S->ft_sensors))
    return fail(LG_ERR_BAD_ARG, "asymmetric_obs needs states, dof_force and ft_sensors");
  const void* al[] = {S->dof_state, S->dof_force, S->ft_sensors, B->obs, B->states, B->obs_clipped, B->states_clipped,
                      B->action, B->goal_pose, B->history, B->applied_torque};
  for (const void* p : al)
    if (p && !aligned16(p)) return fail(LG_ERR_BAD_ARG, "tensor base pointers must be 16-byte aligned");
  const int episode_ptrs = (B->episode_return != nullptr) + (B->last_episode_return != nullptr) +
                           (B->last_episode_length != nullptr) + (B->last_episode_success != nullptr) + (B->episode_stats != nullptr);
  if (episode_ptrs != 0 && episode_ptrs != 5)
    return fail(LG_ERR_BAD_ARG, "episode_return, last_episode_return, last_episode_length, last_episode_success and "
                                "episode_stats go together");
  const int term_ptrs = (B->episode_term_return != nullptr) + (B->last_episode_term_return != nullptr) +
                        (B->episode_term_stats != nullptr);
  if (term_ptrs != 0 && term_ptrs != 3)
    return fail(LG_ERR_BAD_ARG, "episode_term_return, last_episode_term_return and episode_term_stats go together");
  if (term_ptrs && !episode_ptrs)
    return fail(LG_ERR_BAD_ARG, "episode_term_return needs the episode statistics buffers (episode_return, "
                                "last_episode_return, last_episode_length, last_episode_success, episode_stats)");
  if (term_ptrs && (!aligned16(B->episode_term_return) || !aligned16(B->last_episode_term_return)))
    return fail(LG_ERR_BAD_ARG, "episode_term_return and last_episode_term_return must be 16-byte aligned");
  // per-episode DR offsets: sigmas only on observation columns, the mask marking exactly the nonzero ones
  uint64_t mask = 0;
  for (int c = 0; c < 64; ++c) {
    const float sg = P->dr_bias_sigma[c];
    if (sg != 0.0f && (c >= 32 + P->action_dim || !std::isfinite(sg) || sg < 0.0f))
      return fail(LG_ERR_BAD_ARG, "dr_bias_sigma: finite, >= 0, and only on the obs_dim observation columns");
    if (sg != 0.0f) mask |= 1ull << c;
  }
  if (mask != P->dr_bias_mask) return fail(LG_ERR_BAD_ARG, "dr_bias_mask must mark exactly the columns with dr_bias_sigma != 0");
  if ((mask || P->dr_action_bias_sigma != 0.0f) && !P->dr_activate)
    return fail(LG_ERR_BAD_ARG, "dr_bias_sigma / dr_action_bias_sigma != 0 need dr_activate");
  if (mask && !B->obs_bias) return fail(LG_ERR_BAD_ARG, "dr_bias_sigma != 0 needs LgBuffers.obs_bias");
  const float asg = P->dr_action_bias_sigma;
  if (asg != 0.0f && (!std::isfinite(asg) || asg < 0.0f))
    return fail(LG_ERR_BAD_ARG, "dr_action_bias_sigma must be finite and >= 0");
  if (asg != 0.0f && !B->action_bias) return fail(LG_ERR_BAD_ARG, "dr_action_bias_sigma != 0 needs LgBuffers.action_bias");
  return LG_OK;
}

template <bool REWARD>
int launch_post(const LgParams* P, const LgSimState* S, const LgBuffers* B, double sched, cudaStream_t st) {
  if (int rc = validate(P, S, B, true)) return rc;
  if (REWARD && !B->step_stats) return fail(LG_ERR_BAD_ARG, "null statistics buffer");
  if (P->normalize_obs && !B->scale_table) return fail(LG_ERR_BAD_ARG, "null scale_table");
  if (REWARD && !P->fuse_bookkeeping) {
    // stand-alone _post_step: nobody zeroed the accumulators (lg_pre_physics does in the fused sequence)
    if (cudaMemsetAsync(B->step_stats, 0, LG_NUM_STATS * sizeof(double), st) != cudaSuccess) return check_launch("memset");
    if (B->episode_stats && cudaMemsetAsync(B->episode_stats, 0, LG_NUM_EPISODE_STATS * sizeof(double), st) != cudaSuccess)
      return check_launch("memset");
    if (B->episode_term_stats &&
        cudaMemsetAsync(B->episode_term_stats, 0, LG_NUM_EPISODE_TERMS * sizeof(double), st) != cudaSuccess)
      return check_launch("memset");
  }
  const bool asym = P->asymmetric_obs != 0;
  const bool clip = B->obs_clipped != nullptr;
  if (clip && asym && !B->states_clipped) return fail(LG_ERR_BAD_ARG, "obs_clipped and states_clipped go together");
  LgCoef cf;
  std::memset(&cf, 0, sizeof(cf));
  if (REWARD && P->use_device_clock) {
    if (!B->reward_coef) return fail(LG_ERR_BAD_ARG, "use_device_clock needs reward_coef");
  } else {
    lg::compute_coefs(*P, sched, cf.v);
  }
  const int E = P->action_dim == 9 ? pick_tile_envs(P->num_envs) : 32;
  const unsigned grid = (unsigned)((P->num_envs + E - 1) / E);
  cudaError_t err;
  // rarely-used paths (DR noise, keypoint term, moving goal, bf16 copies, episode statistics) live in their own
  // instantiation: switched off they cost nothing
  const bool ext = P->dr_activate || P->goal_rotation || ((P->term_active_mask >> LG_TERM_KEYPOINT) & 1) || B->obs_bf16 ||
                   B->states_bf16 || B->episode_return;
#define LG_X(AD, AS, CL, EE, EX) launch_pdl(pdl_mode() & 2, lg::post_physics_kernel<AD, AS, REWARD, CL, EE, EX>, grid, lg::kPostThreads, 0, st, *P, *S, *B, cf)
#ifdef LG_FAST_BUILD
  if (ext || clip || P->action_dim != 9) return fail(LG_ERR_UNSUPPORTED, "LG_FAST_BUILD: instantiation not built");
  if (asym) err = E == 28 ? LG_X(9, true, false, 28, false) : LG_X(9, true, false, 32, false);
  else err = E == 28 ? LG_X(9, false, false, 28, false) : LG_X(9, false, false, 32, false);
#else
#define LG_K(AD, AS, CL, EE) (ext ? LG_X(AD, AS, CL, EE, true) : LG_X(AD, AS, CL, EE, false))
#define LG_E(AD, AS, CL) (E == 16 ? LG_K(AD, AS, CL, 16) : E == 24 ? LG_K(AD, AS, CL, 24) : E == 28 ? LG_K(AD, AS, CL, 28) : LG_K(AD, AS, CL, 32))
  if (P->action_dim == 9) {
    if (asym) err = clip ? LG_E(9, true, true) : LG_E(9, true, false);
    else err = clip ? LG_E(9, false, true) : LG_E(9, false, false);
  } else {
    if (asym) err = clip ? LG_K(18, true, true, 32) : LG_K(18, true, false, 32);
    else err = clip ? LG_K(18, false, true, 32) : LG_K(18, false, false, 32);
  }
#endif
#ifndef LG_FAST_BUILD
#undef LG_E
#undef LG_K
#endif
#undef LG_X
  if (err != cudaSuccess) return fail(LG_ERR_CUDA, std::string("post_physics_kernel: ") + cudaGetErrorString(err));
  const int rc = check_launch("post_physics_kernel");
  if (rc == LG_OK && REWARD) { g_prev.stream = (void*)st; g_prev.post = true; }
  return rc;
}
}  // namespace

extern "C" {

int lg_version(void) { return LG_VERSION; }
int lg_set_l2_fetch_granularity(int bytes) {
  if (bytes != 32 && bytes != 64 && bytes != 128) return fail(LG_ERR_BAD_ARG, "granularity must be 32, 64 or 128");
  if (cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)bytes) != cudaSuccess) return check_launch("cudaDeviceSetLimit");
  return LG_OK;
}
const char* lg_last_error(void) { return g_error.c_str(); }
size_t lg_struct_size(int which) {
  switch (which) {
    case 0: return sizeof(LgParams);
    case 1: return sizeof(LgSimState);
    case 2: return sizeof(LgBuffers);
    case 3: return sizeof(LgControl);
    case 4: return sizeof(LgRewardTerm);
    case 5: return sizeof(LgHostStep);
    case 6: return sizeof(LgTorchRng);
    default: return 0;
  }
}
int64_t lg_scan_tiles(int64_t n) { return (n + lg::kPreTile - 1) / lg::kPreTile; }
int64_t lg_pre_resident_tiles(void) {
  // the instantiation grids beyond one wave use (see pre_physics_kernel: MINB = 4)
  int per_sm9 = 0, per_sm18 = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm9, lg::pre_physics_kernel<9, false, 4, true>, lg::kPreThreads, 0);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm18, lg::pre_physics_kernel<18, false, 4, true>, lg::kPreThreads, 0);
  const int per_sm = per_sm9 < per_sm18 ? per_sm9 : per_sm18;
  cudaGetLastError();   // no device: report one CTA per SM of the default count rather than an error
  return (int64_t)(per_sm > 0 ? per_sm : 1) * sm_count();
}

int lg_post_physics(const LgParams* P, const LgSimState* S, const LgBuffers* B, double sched_step, void* stream) {
  return launch_post<true>(P, S, B, sched_step, (cudaStream_t)stream);
}
int lg_fill_observations(const LgParams* P, const LgSimState* S, const LgBuffers* B, void* stream) {
  return launch_post<false>(P, S, B, 0.0, (cudaStream_t)stream);
}
int lg_init_history(const LgParams* P, const LgSimState* S, const LgBuffers* B, void* stream) {
  if (int rc = validate(P, S, B, false)) return rc;
  const int64_t total = P->num_envs * LG_HISTORY_COLS;
  lg::init_history_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(*P, *S, *B);
  return check_launch("init_history_kernel");
}

namespace {
int check_torch_rng(const LgParams* P, const LgBuffers* B) {
  if (!B->torch_rng) return fail(LG_ERR_BAD_ARG, "rng_stream LG_RNG_TORCH needs LgBuffers.torch_rng");
  if (P->inject_draws) return fail(LG_ERR_BAD_ARG, "rng_stream LG_RNG_TORCH draws torch's stream: injected draws are not read");
  if (P->sm_count <= 0 || P->threads_per_sm < 256) return fail(LG_ERR_BAD_ARG, "rng_stream LG_RNG_TORCH needs sm_count and threads_per_sm");
  if (P->env_offset != 0 || P->global_num_envs != P->num_envs)
    return fail(LG_ERR_BAD_ARG, "rng_stream LG_RNG_TORCH draws the stream of one process over all envs: no sharding");
  return LG_OK;
}
int launch_pre(const LgParams* P, const LgSimState* S, const LgBuffers* B, const float* action_in, void* stream,
               bool chained, bool exclusive_sm) {
  if (int rc = validate(P, S, B, false)) return rc;
  if (!action_in) return fail(LG_ERR_BAD_ARG, "null action_in");
  if (!B->scan_status || !B->reset_ids || !B->goal_reset_ids || !B->counts)
    return fail(LG_ERR_BAD_ARG, "null compaction buffer");
  if (P->inject_draws && !(B->inject_reset_u || B->inject_goal_u || B->inject_reset_n || B->inject_goal_n))
    return fail(LG_ERR_BAD_ARG, "inject_draws set without injected arrays");
  const int tiles = (int)lg_scan_tiles(P->num_envs);
  if (!aligned16(action_in)) return fail(LG_ERR_BAD_ARG, "action_in must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const bool torch_rng = P->rng_stream == LG_RNG_TORCH;
  if (torch_rng) {
    if (int rc = check_torch_rng(P, B)) return rc;
    // list lengths and base offset first, in a launch of their own: no CTA of the pass below may wait for another
    // one's total (ticket grids are not co-resident)
    const int64_t want = (P->num_envs + 16 * lg::kCountThreads - 1) / (16 * lg::kCountThreads);
    const unsigned grid = (unsigned)(want < sm_count() ? (want > 0 ? want : 1) : sm_count());
    lg::torch_count_kernel<<<grid, lg::kCountThreads, 0, st>>>(B->reset, B->goal_reset, B->force_reset, B->force_goal_reset,
                                                               P->num_envs, *P, B->torch_rng);
    if (int rc = check_launch("torch_count_kernel")) return rc;
    chained = false;   // the pass reads what the counting launch wrote: plain stream order
  }
  // The look-back spins on predecessor tiles, so every tile a CTA can wait for must be running: while the whole grid
  // is co-resident (lg_pre_resident_tiles) tiles are block indices; larger grids take their tiles by ticket, in
  // dispatch order.  (The post pass's CTAs cannot crowd this kernel out: they are only launched once every CTA of
  // this grid has started.)  LG_PRE_TICKET=1 forces the ticket path (tests).
  static const int64_t resident_ctas = lg_pre_resident_tiles();
  static const bool force_ticket = env_flag("LG_PRE_TICKET");
  const bool ticket = force_ticket || tiles > resident_ctas;
cudaError_t err;
  // grids that are co-resident at 3 CTAs per SM (<= 85 registers) run the latency-tuned instantiation, larger ones
  // the 64-register one; both thresholds come from the occupancy of the instantiation that is launched
  static const int64_t resident_small = [] {
    int a = 0, b = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, lg::pre_physics_kernel<9, false, 3, true>, lg::kPreThreads, 0);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, lg::pre_physics_kernel<18, false, 3, true>, lg::kPreThreads, 0);
    const int per_sm = a < b ? a : b;
    return (int64_t)(per_sm > 0 ? per_sm : 1) * sm_count();
  }();
  const bool small = tiles <= resident_small;
  // Grids of 32 .. kDirectMaxTiles tiles, all running at once (one CTA per SM), count the flagged envs in front of each
  // tile directly from the flag bytes instead of chaining the tiles by look-back (count_flagged_before, lg_pre.cuh):
  // 16 384 envs 11.00 -> 10.58 us/step.  Below 32 tiles the look-back chain is short and wins (1024 envs: 6.49 against
  // 6.67 us/step).  Needs the flag arrays 16-byte aligned.  LG_PRE_DIRECT=0 keeps the look-back (tests, A/B).
  static const bool no_direct = env_int("LG_PRE_DIRECT", 1) == 0;
  const bool direct = !ticket && small && !no_direct && tiles >= 32 && tiles <= lg::kDirectMaxTiles && tiles <= sm_count() &&
                      aligned16(B->reset) && aligned16(B->goal_reset) && aligned16(B->force_reset) &&
                      aligned16(B->force_goal_reset);
  const lg::PreHot hot = {action_in, S->dof_state, B->applied_torque, P->num_envs, tiles, 0};
  // chained launch (lg_pre_physics_chained): optionally one CTA per SM, by 100 KB of unused dynamic shared memory
  const bool pdl = chained && (pdl_mode() & 1) != 0;
  const size_t dyn = (pdl && direct && exclusive_sm) ? 100 * 1024 : 0;
  if (dyn) {
    static const cudaError_t opt_in = [] {
      cudaError_t a = cudaFuncSetAttribute(lg::pre_physics_kernel<9, false, 3, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
      cudaError_t b = cudaFuncSetAttribute(lg::pre_physics_kernel<18, false, 3, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
      return a != cudaSuccess ? a : b;
    }();
    if (opt_in != cudaSuccess) return fail(LG_ERR_CUDA, std::string("pre_physics_kernel shared memory opt-in: ") + cudaGetErrorString(opt_in));
  }
#define LG_PRE(AD, TK, MB, SP, DR) err = torch_rng \
    ? launch_pdl(false, lg::pre_physics_kernel<AD, TK, MB, SP, DR, true>, (unsigned)tiles, SP ? lg::kPreThreads : lg::kScanThreads, 0, st, hot, *P, *S, *B) \
    : launch_pdl(pdl, lg::pre_physics_kernel<AD, TK, MB, SP, DR>, (unsigned)tiles, SP ? lg::kPreThreads : lg::kScanThreads, DR ? dyn : 0, st, hot, *P, *S, *B)
  if (P->action_dim == 9) {
    if (ticket) LG_PRE(9, true, 6, false, false); else if (direct) LG_PRE(9, false, 3, true, true);
    else if (small) LG_PRE(9, false, 3, true, false); else LG_PRE(9, false, 4, true, false);
  } else {
    if (ticket) LG_PRE(18, true, 6, false, false); else if (direct) LG_PRE(18, false, 3, true, true);
    else if (small) LG_PRE(18, false, 3, true, false); else LG_PRE(18, false, 4, true, false);
  }
#undef LG_PRE
  if (err != cudaSuccess) return fail(LG_ERR_CUDA, std::string("pre_physics_kernel: ") + cudaGetErrorString(err));
  if (int rc = check_launch("pre_physics_kernel")) return rc;
  if (!B->obs_bias && !B->action_bias) return LG_OK;
  // extension: the per-episode DR offsets of the envs this pass reset (lg_pre.cuh, draw_bias_kernel): a warp per env
  const int64_t want = (P->num_envs * 32 + lg::kDrawBiasThreads - 1) / lg::kDrawBiasThreads;
  const unsigned grid = (unsigned)(want < 8 * sm_count() ? want : 8 * sm_count());
  err = launch_pdl(pdl_mode() & 2, lg::draw_bias_kernel, grid, lg::kDrawBiasThreads, 0, st, *P, *B);
  if (err != cudaSuccess) return fail(LG_ERR_CUDA, std::string("draw_bias_kernel: ") + cudaGetErrorString(err));
  return check_launch("draw_bias_kernel");
}
}  // namespace

int lg_pre_physics(const LgParams* P, const LgSimState* S, const LgBuffers* B, const float* action_in, void* stream) {
  return launch_pre(P, S, B, action_in, stream, false, false);
}
int lg_pre_physics_chained(const LgParams* P, const LgSimState* S, const LgBuffers* B, const float* action_in,
                           int exclusive_sm, void* stream) {
  const bool after_post = g_prev.post && g_prev.stream == stream;
  return launch_pre(P, S, B, action_in, stream, after_post, exclusive_sm != 0);
}

int lg_compact(const uint8_t* mask, int64_t n, int64_t* ids_out, int32_t* count_out, uint64_t* status,
               LgControl* control, void* stream) {
  if (!mask || !ids_out || !count_out || !status || !control) return fail(LG_ERR_BAD_ARG, "null argument");
  if (n < 0 || n >= (1 << 23)) return fail(LG_ERR_BAD_ARG, "n out of range");
  if (n == 0) { cudaMemsetAsync(count_out, 0, 2 * sizeof(int32_t), (cudaStream_t)stream); return check_launch("memset"); }
  const int tiles = (int)lg_scan_tiles(n);
  lg::compact_kernel<<<tiles, lg::kScanThreads, 0, (cudaStream_t)stream>>>(mask, n, ids_out, count_out, status, control, tiles);
  return check_launch("compact_kernel");
}

static int reset_list(const LgParams* P, const LgSimState* S, const LgBuffers* B, const int64_t* ids, int64_t k,
                      int goal_only, void* stream) {
  if (int rc = validate(P, S, B, false)) return rc;
  if (k < 0 || (k > 0 && !ids)) return fail(LG_ERR_BAD_ARG, "bad id list");
  if (k == 0) return LG_OK;   // the reference makes no call for an empty list: nothing is drawn
  if (P->rng_stream == LG_RNG_TORCH) {
    if (int rc = check_torch_rng(P, B)) return rc;
    lg::reset_ids_kernel<true><<<(unsigned)((k + 127) / 128), 128, 0, (cudaStream_t)stream>>>(*P, *S, *B, ids, k, goal_only);
    if (int rc = check_launch("reset_ids_kernel")) return rc;
    lg::torch_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(B->torch_rng, lg::torch_plan(*P, (uint32_t)k, goal_only != 0).total());
    if (int rc = check_launch("torch_advance_kernel")) return rc;
    // the DR offsets come from the own stream, keyed by the epoch, also here: each call must draw new ones
    if (!B->obs_bias && !B->action_bias) return LG_OK;
    lg::bump_epoch_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(B->control);
    return check_launch("bump_epoch_kernel");
  }
  lg::reset_ids_kernel<<<(unsigned)((k + 127) / 128), 128, 0, (cudaStream_t)stream>>>(*P, *S, *B, ids, k, goal_only);
  if (int rc = check_launch("reset_ids_kernel")) return rc;
  lg::bump_epoch_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(B->control);
  return check_launch("bump_epoch_kernel");
}
int lg_reset_envs(const LgParams* P, const LgSimState* S, const LgBuffers* B, const int64_t* ids, int64_t k, void* stream) {
  return reset_list(P, S, B, ids, k, 0, stream);
}
int lg_goal_reset_envs(const LgParams* P, const LgSimState* S, const LgBuffers* B, const int64_t* ids, int64_t k, void* stream) {
  return reset_list(P, S, B, ids, k, 1, stream);
}

int lg_torch_philox(uint64_t seed, uint64_t offset, int64_t n, int normal, float* out, void* stream) {
  if (n < 0 || n >= (1ll << 31) || (n > 0 && !out) || (offset & 3u)) return fail(LG_ERR_BAD_ARG, "bad argument");
  if (n == 0) return LG_OK;
  int dev = 0, tps = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&tps, cudaDevAttrMaxThreadsPerMultiProcessor, dev) != cudaSuccess)
    return check_launch("lg_torch_philox");
  const uint32_t gmax = (uint32_t)sm_count() * ((uint32_t)tps / 256u);
  lg::torch_philox_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(seed, offset, (uint32_t)n, gmax, normal, out);
  return check_launch("torch_philox_kernel");
}
uint64_t lg_torch_philox_advance(int64_t n, int32_t sm_count, int32_t threads_per_sm) {
  if (n <= 0 || sm_count <= 0 || threads_per_sm < 256) return 0;
  // 64-bit form of lg::torch_advance (the kernels' sizes fit 32 bits; this host function takes any n)
  const uint64_t gmax = (uint64_t)sm_count * (uint64_t)(threads_per_sm / 256), g = ((uint64_t)n + 255) / 256;
  const uint64_t T = 256 * (g < gmax ? g : gmax);
  return 4 * (((uint64_t)n - 1) / (4 * T) + 1);
}

int lg_pre_step(const LgParams* P, const LgSimState* S, const LgBuffers* B, void* stream) {
  if (int rc = validate(P, S, B, false)) return rc;
  if (!B->applied_torque) return fail(LG_ERR_BAD_ARG, "null applied_torque");
  lg::pre_step_kernel<<<(unsigned)((P->num_envs + 127) / 128), 128, 0, (cudaStream_t)stream>>>(*P, *S, *B);
  return check_launch("pre_step_kernel");
}

#define LG_GRID(n) (unsigned)(((n) + 255) / 256), 256, 0, (cudaStream_t)stream
int lg_quat_mul(const float* a, const float* b, float* out, int64_t n, void* stream) {
  if (!a || !b || !out || n < 0) return fail(LG_ERR_BAD_ARG, "bad argument");
  if (!aligned16(a) || !aligned16(b) || !aligned16(out)) return fail(LG_ERR_BAD_ARG, "quaternion arrays must be 16-byte aligned");
  if (n) lg::quat_mul_kernel<<<LG_GRID(n)>>>(a, b, out, n);
  return check_launch("quat_mul_kernel");
}
int lg_quat_diff_rad(const float* a, const float* b, float* out, int64_t n, void* stream) {
  if (!a || !b || !out || n < 0) return fail(LG_ERR_BAD_ARG, "bad argument");
  if (!aligned16(a) || !aligned16(b)) return fail(LG_ERR_BAD_ARG, "quaternion arrays must be 16-byte aligned");
  if (n) lg::quat_diff_kernel<<<LG_GRID(n)>>>(a, b, out, n);
  return check_launch("quat_diff_kernel");
}
static int rowwise(int op, const float* x, const float* lo, const float* hi, float* out, int64_t n, int32_t dims, void* stream) {
  if (!x || !lo || !hi || !out || n < 0 || dims <= 0) return fail(LG_ERR_BAD_ARG, "bad argument");
  const int64_t total = n * dims;
  if (total == 0) return LG_OK;
  if (op == 0) lg::rowwise_kernel<0><<<LG_GRID(total)>>>(x, lo, hi, out, total, dims);
  else if (op == 1) lg::rowwise_kernel<1><<<LG_GRID(total)>>>(x, lo, hi, out, total, dims);
  else lg::rowwise_kernel<2><<<LG_GRID(total)>>>(x, lo, hi, out, total, dims);
  return check_launch("rowwise_kernel");
}
int lg_scale_transform(const float* x, const float* lo, const float* hi, float* out, int64_t n, int32_t d, void* s) { return rowwise(0, x, lo, hi, out, n, d, s); }
int lg_unscale_transform(const float* x, const float* lo, const float* hi, float* out, int64_t n, int32_t d, void* s) { return rowwise(1, x, lo, hi, out, n, d, s); }
int lg_saturate(const float* x, const float* lo, const float* hi, float* out, int64_t n, int32_t d, void* s) { return rowwise(2, x, lo, hi, out, n, d, s); }
int lg_lgsk_kernel(const float* x, float scale, float* out, int64_t n, void* stream) {
  if (!x || !out || n < 0) return fail(LG_ERR_BAD_ARG, "bad argument");
  if (n) lg::lgsk_kernel<<<LG_GRID(n)>>>(x, scale, out, n);
  return check_launch("lgsk_kernel");
}
int lg_cube_keypoints(const float* pose, float cube_size, float* out, int64_t n, void* stream) {
  if (!pose || !out || n < 0) return fail(LG_ERR_BAD_ARG, "bad argument");
  if (n) lg::keypoints_kernel<<<LG_GRID(n * 8)>>>(pose, cube_size, out, n);
  return check_launch("keypoints_kernel");
}

int lg_integrate_goal(const LgParams* P, const LgSimState* S, float dt, void* stream) {
  if (!P || !S || !S->root_state || P->num_envs < 0) return fail(LG_ERR_BAD_ARG, "bad argument");
  const int64_t n = P->num_envs;
  if (n) lg::integrate_rows_kernel<<<LG_GRID(n)>>>(S->root_state + (size_t)P->goal_slot * 13, (int64_t)P->actors_per_env * 13, dt, n);
  return check_launch("integrate_rows_kernel");
}

int lg_selftest_division(float span, float rcp, unsigned long long* mismatches_dev, void* stream) {
  if (!mismatches_dev) return fail(LG_ERR_BAD_ARG, "null argument");
  lg::selftest_division_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(span, rcp, mismatches_dev);
  return check_launch("selftest_division_kernel");
}

int lg_upload_sim_state(const LgParams* P, const LgSimState* S, const LgHostStep* H, void* stream) {
  if (!P || !S || !H || !H->dof_state_host || !H->root_state_host || !H->rigid_body_host)
    return fail(LG_ERR_BAD_ARG, "null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t N = P->num_envs;
  const cudaMemcpyKind k = cudaMemcpyHostToDevice;
  cudaMemcpyAsync(S->dof_state, H->dof_state_host, sizeof(float) * N * 18, k, st);
  // Of root_state and rigid_body only the rows the path reads: the object actor's row and the three fingertip
  // bodies, each one strided 2-D copy of 52-byte rows.  Measured on a B200 (PCIe 5 x16, scripts/pcie_probe.cu,
  // 16384 envs): object rows 39 us against 65 us for the whole tensor; the three fingertip copies 143 us against
  // 199 us for the run of bodies 6..16 and 311 us for the whole tensor.
  const size_t row = sizeof(float) * 13;
  cudaMemcpy2DAsync(S->root_state + (size_t)P->object_slot * 13, row * P->actors_per_env,
                    H->root_state_host + (size_t)P->object_slot * 13, row * P->actors_per_env, row, (size_t)N, k, st);
  if (P->goal_rotation)  // moving goal: the pose the simulator integrated for the goal body is read back (:1279-1284)
    cudaMemcpy2DAsync(S->root_state + (size_t)P->goal_slot * 13, row * P->actors_per_env,
                      H->root_state_host + (size_t)P->goal_slot * 13, row * P->actors_per_env, sizeof(float) * 7, (size_t)N, k, st);
  const size_t pitch = row * P->bodies_per_env;
  for (int i = 0; i < 3; ++i) {
    const size_t off = (size_t)P->fingertip_body[i] * 13;
    cudaMemcpy2DAsync(const_cast<float*>(S->rigid_body) + off, pitch, H->rigid_body_host + off, pitch, row, (size_t)N, k, st);
  }
  if (P->asymmetric_obs) {
    if (!H->dof_force_host || !H->ft_sensors_host) return fail(LG_ERR_BAD_ARG, "null host buffer (asymmetric)");
    cudaMemcpyAsync(const_cast<float*>(S->dof_force), H->dof_force_host, sizeof(float) * N * 9, k, st);
    cudaMemcpyAsync(const_cast<float*>(S->ft_sensors), H->ft_sensors_host, sizeof(float) * N * 18, k, st);
  }
  return check_launch("lg_upload_sim_state");
}

int lg_step_host_pipelined(const LgParams* P, const LgSimState* S, const LgBuffers* B, const LgHostStep* H,
                           double sched_step, int chunks, void* stream_main, void* stream_up, void* stream_down) {
  if (int rc = validate(P, S, B, true)) return rc;
  if (!H || !H->dof_state_host || !H->root_state_host || !H->rigid_body_host || !H->action_host || !H->action_staging ||
      !H->reward_host || (!H->obs_host && !(P->asymmetric_obs && H->states_host && !P->dr_activate)))
    return fail(LG_ERR_BAD_ARG, "null host buffer");
  if (chunks < 1 || chunks > 16) return fail(LG_ERR_BAD_ARG, "chunks must be in 1..16");
  if (chunks == 1) return lg_step_host(P, S, B, H, sched_step, stream_main);   // nothing to overlap: one stream, no events
  if (P->asymmetric_obs && (!H->dof_force_host || !H->ft_sensors_host || !H->states_host))
    return fail(LG_ERR_BAD_ARG, "null host buffer (asymmetric)");
  cudaStream_t main = (cudaStream_t)stream_main, up = (cudaStream_t)stream_up, down = (cudaStream_t)stream_down;
  // events are created once per host thread and reused (timing disabled: cheapest kind)
  struct Pool { cudaEvent_t pre, done, up[16], post[16]; bool ok = false; };
  static thread_local Pool pool;
  if (!pool.ok) {
    const unsigned f = cudaEventDisableTiming;
    cudaEventCreateWithFlags(&pool.pre, f); cudaEventCreateWithFlags(&pool.done, f);
    for (int i = 0; i < 16; ++i) { cudaEventCreateWithFlags(&pool.up[i], f); cudaEventCreateWithFlags(&pool.post[i], f); }
    pool.ok = true;
  }
  const int64_t N = P->num_envs;
  const int A = P->action_dim, od = 32 + A, sd = P->asymmetric_obs ? od + 72 : 0;
  const float* obs_src = B->obs_clipped ? B->obs_clipped : B->obs;
  const float* st_src = B->states_clipped ? B->states_clipped : B->states;
  // the action arrives first; resets / torque consume it together with the previous state
  cudaMemcpyAsync(H->action_staging, H->action_host, sizeof(float) * N * A, cudaMemcpyHostToDevice, main);
  if (int rc = lg_pre_physics(P, S, B, H->action_staging, stream_main)) return rc;
  cudaEventRecord(pool.pre, main);
  cudaStreamWaitEvent(up, pool.pre, 0);
  int64_t lo = 0;
  for (int c = 0; c < chunks; ++c) {
    int64_t hi = c == chunks - 1 ? N : ((N * (c + 1) / chunks + 16) / 32) * 32;
    if (hi > N) hi = N;
    if (hi <= lo) continue;
    LgParams pc = *P;
    pc.num_envs = hi - lo; pc.env_offset = P->env_offset + lo; pc.stats_num_envs = N; pc.fuse_bookkeeping = 1;
    LgSimState sc = *S;
    sc.dof_state += lo * 18; sc.root_state += lo * 13 * P->actors_per_env; sc.rigid_body += lo * 13 * P->bodies_per_env;
    if (sc.dof_force) sc.dof_force += lo * 9;
    if (sc.ft_sensors) sc.ft_sensors += lo * 18;
    LgHostStep hc = *H;
    hc.dof_state_host += lo * 18; hc.root_state_host += lo * 13 * P->actors_per_env;
    hc.rigid_body_host += lo * 13 * P->bodies_per_env;
    if (hc.dof_force_host) hc.dof_force_host += lo * 9;
    if (hc.ft_sensors_host) hc.ft_sensors_host += lo * 18;
    LgBuffers bc = *B;
    bc.obs += lo * od; if (bc.states) bc.states += lo * sd;
    if (bc.obs_clipped) bc.obs_clipped += lo * od;
    if (bc.states_clipped) bc.states_clipped += lo * sd;
    bc.action += lo * A; bc.reward += lo; bc.reset += lo; bc.goal_reset += lo; bc.successes += lo;
    if (bc.dones) bc.dones += lo;
    bc.steps_count += lo; bc.goal_pose += lo * 7; bc.goal_movement += lo * 6; bc.history += lo * LG_HISTORY_COLS;
    if (bc.applied_torque) bc.applied_torque += lo * 9;
    bc.term_rewards = nullptr;
    if (bc.episode_return) {
      bc.episode_return += lo; bc.last_episode_return += lo; bc.last_episode_length += lo; bc.last_episode_success += lo;
    }
    if (bc.episode_term_return) {
      bc.episode_term_return += lo * LG_NUM_EPISODE_TERMS; bc.last_episode_term_return += lo * LG_NUM_EPISODE_TERMS;
    }
    if (bc.obs_bias) bc.obs_bias += lo * od;
    if (bc.action_bias) bc.action_bias += lo * A;
    if (int rc = lg_upload_sim_state(&pc, &sc, &hc, stream_up)) return rc;
    cudaEventRecord(pool.up[c], up);
    cudaStreamWaitEvent(main, pool.up[c], 0);
    if (int rc = lg_post_physics(&pc, &sc, &bc, sched_step, stream_main)) return rc;
    cudaEventRecord(pool.post[c], main);
    cudaStreamWaitEvent(down, pool.post[c], 0);
    if (H->obs_host) cudaMemcpyAsync(H->obs_host + lo * od, obs_src + lo * od, sizeof(float) * (hi - lo) * od, cudaMemcpyDeviceToHost, down);
    if (sd) cudaMemcpyAsync(H->states_host + lo * sd, st_src + lo * sd, sizeof(float) * (hi - lo) * sd, cudaMemcpyDeviceToHost, down);
    cudaMemcpyAsync(H->reward_host + lo, B->reward + lo, sizeof(float) * (hi - lo), cudaMemcpyDeviceToHost, down);
    if (H->dones_host && B->dones) cudaMemcpyAsync(H->dones_host + lo, B->dones + lo, (size_t)(hi - lo), cudaMemcpyDeviceToHost, down);
    lo = hi;
  }
  cudaEventRecord(pool.done, down);
  cudaStreamWaitEvent(main, pool.done, 0);
  return check_launch("lg_step_host_pipelined");
}

#ifdef LG_TRACE
// development only: copies the phase stamps of kernel `which` (0 post, 1 pre) to host memory
int lg_trace_read(int which, unsigned long long* dst, int ctas) {
  if (which < 0 || which > 1 || ctas > lg::kTraceMaxCtas) return fail(LG_ERR_BAD_ARG, "bad trace request");
  const size_t bytes = sizeof(unsigned long long) * 2 * lg::kTraceSlots * (size_t)ctas;
  if (cudaMemcpyFromSymbol(dst, lg::g_trace, bytes, sizeof(unsigned long long) * 2 * lg::kTraceSlots * lg::kTraceMaxCtas * which) != cudaSuccess)
    return check_launch("lg_trace_read");
  return LG_OK;
}
#endif

int lg_step_host(const LgParams* P, const LgSimState* S, const LgBuffers* B, const LgHostStep* H, double sched_step, void* stream) {
  if (int rc = validate(P, S, B, true)) return rc;
  if (!H || !H->dof_state_host || !H->root_state_host || !H->rigid_body_host || !H->action_host || !H->action_staging ||
      !H->reward_host || (!H->obs_host && !(P->asymmetric_obs && H->states_host && !P->dr_activate)))
    return fail(LG_ERR_BAD_ARG, "null host buffer");
  if (P->asymmetric_obs && (!H->dof_force_host || !H->ft_sensors_host || !H->states_host))
    return fail(LG_ERR_BAD_ARG, "null host buffer (asymmetric)");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t N = P->num_envs;
  const int obs_dim = 32 + P->action_dim, state_dim = obs_dim + 72;
  // the action arrives first: the pre-physics pass (resets, torque) consumes it together with last step's state
  cudaMemcpyAsync(H->action_staging, H->action_host, sizeof(float) * N * P->action_dim, cudaMemcpyHostToDevice, st);
  if (int rc = lg_pre_physics(P, S, B, H->action_staging, stream)) return rc;
  // "physics": the simulator's new state lands in the device tensors (only the rows the path reads)
  if (int rc = lg_upload_sim_state(P, S, H, stream)) return rc;
  if (int rc = lg_post_physics(P, S, B, sched_step, stream)) return rc;
  const float* obs_src = B->obs_clipped ? B->obs_clipped : B->obs;
  if (H->obs_host) cudaMemcpyAsync(H->obs_host, obs_src, sizeof(float) * N * obs_dim, cudaMemcpyDeviceToHost, st);
  if (P->asymmetric_obs) {
    const float* st_src = B->states_clipped ? B->states_clipped : B->states;
    cudaMemcpyAsync(H->states_host, st_src, sizeof(float) * N * state_dim, cudaMemcpyDeviceToHost, st);
  }
  cudaMemcpyAsync(H->reward_host, B->reward, sizeof(float) * N, cudaMemcpyDeviceToHost, st);
  if (H->dones_host && B->dones) cudaMemcpyAsync(H->dones_host, B->dones, N, cudaMemcpyDeviceToHost, st);
  return check_launch("lg_step_host");
}

}  // extern "C"
