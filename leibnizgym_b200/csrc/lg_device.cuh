// Device-side building blocks of the TriFinger MDP hot path (sm_100a).
//
// Numerics contract: the translation unit is compiled with -fmad=false, IEEE division and
// square root and without fast-math, so every fp32 operation below rounds exactly once, in
// the order written — the order of the reference's ATen ops.  The only fused multiply-adds
// are the explicit __fmaf_rn calls in norm3(), which reproduce the contraction inside
// ATen's CPU 2-norm reduction (measured against torch 2.11; see DESIGN.md "numerics"), and
// the one in torch_normal(), which reproduces the contraction in torch's CUDA Box-Muller.
//
// All reference paths are relative to /root/reference/leibnizgym/.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "leibniz_b200.h"

namespace lg {

// Development-only phase tracing (-DLG_TRACE, scripts/trace_step.py): lane 0 of selected warps stamps %globaltimer
// and the SM clock at named points of the two step kernels; never compiled into the shipped library.
#ifdef LG_TRACE
constexpr int kTraceSlots = 32, kTraceMaxCtas = 8192;
__device__ unsigned long long g_trace[2][kTraceMaxCtas][2 * kTraceSlots];
__device__ __forceinline__ void trace_point(int kernel, int slot) {
  unsigned long long t, c;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  asm volatile("mov.u64 %0, %%clock64;" : "=l"(c));
  if (blockIdx.x < kTraceMaxCtas) { g_trace[kernel][blockIdx.x][slot] = t; g_trace[kernel][blockIdx.x][kTraceSlots + slot] = c; }
}
#define LG_TP(kernel, slot, cond) do { if (cond) trace_point(kernel, slot); } while (0)
#else
#define LG_TP(kernel, slot, cond) do { } while (0)
#endif

constexpr float kTwoPi = 6.283185307179586f;  // fp32(2 * np.pi), envs/trifinger/sample.py:29, :82

// ---------------------------------------------------------------------------------------
// memory helpers
// ---------------------------------------------------------------------------------------
// streaming 128-bit load: read-only path, no L1 allocation (every input byte is used once).  Only for tensors the
// calling kernel never writes (simulator rows in the post-physics pass).
__device__ __forceinline__ float4 ld_stream4(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
// the same without the read-only path: for rows the SAME kernel rewrites later (the history entry), where
// ld.global.nc would be outside the PTX contract (.nc data must not change during the kernel)
__device__ __forceinline__ float4 ld_hist4(const float4* p) {
  float4 v;
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
// 32-bit load of a column element: no L1 allocation (every input byte is used once), 64-byte L2 fetches (the gathered
// 52-byte rows cost 25 % fewer DRAM sectors than with the default granularity).  Not the read-only `.nc` path: the
// goal-pose column is rewritten by the same kernel in the moving-goal path, and `.nc` data must not change while
// the kernel runs.
__device__ __forceinline__ float ld_stream1(const float* p) {
  float v;
#ifdef LG_NC_LOADS
  asm volatile("ld.global.nc.L1::no_allocate.L2::64B.f32 %0, [%1];" : "=f"(v) : "l"(p));
#else
  asm volatile("ld.global.L1::no_allocate.L2::64B.f32 %0, [%1];" : "=f"(v) : "l"(p));
#endif
  return v;
}
__device__ __forceinline__ uint64_t ld_volatile_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ---------------------------------------------------------------------------------------
// math primitives (utils/torch_utils.py)
// ---------------------------------------------------------------------------------------
// torch.norm(v, p=2, dim=-1) of a 3-vector: ATen accumulates acc = fma(x, x, acc) then sqrt
__device__ __forceinline__ float norm3(float x, float y, float z) {
  float acc = x * x;
  acc = __fmaf_rn(y, y, acc);
  acc = __fmaf_rn(z, z, acc);
  return sqrtf(acc);
}

struct Quat { float x, y, z, w; };  // xyzw, real part last (torch_utils.py:83-113)

// quat_mul, the reference's 8-multiplication form, same operation order (torch_utils.py:101-109)
__device__ __forceinline__ Quat quat_mul(const Quat a, const Quat b) {
  const float ww = (a.z + a.x) * (b.x + b.y);
  const float yy = (a.w - a.y) * (b.w + b.z);
  const float zz = (a.w + a.y) * (b.w - b.z);
  const float xx = (ww + yy) + zz;
  const float qq = 0.5f * (xx + (a.z - a.x) * (b.x - b.y));
  Quat r;
  r.w = (qq - ww) + (a.z - a.y) * (b.y - b.z);
  r.x = (qq - xx) + (a.x + a.w) * (b.x + b.w);
  r.y = (qq - yy) + (a.w - a.x) * (b.y + b.z);
  r.z = (qq - zz) + (a.z + a.y) * (b.w - b.x);
  return r;
}

__device__ __forceinline__ Quat quat_conjugate(const Quat a) {  // torch_utils.py:116-128
  return Quat{-a.x, -a.y, -a.z, a.w};
}

// |(a (x) conj b)_xyz| clamped to <= 1: the quantity the reference feeds to asin (torch_utils.py:145-149)
__device__ __forceinline__ float quat_diff_sine(const Quat a, const Quat b) {
  const Quat m = quat_mul(a, quat_conjugate(b));
  const float n = norm3(m.x, m.y, m.z);
  return n > 1.0f ? 1.0f : n;  // torch.clamp(max=1.0); NaN stays NaN
}

__device__ __forceinline__ float quat_diff_rad(const Quat a, const Quat b) {  // torch_utils.py:131-150
  return 2.0f * asinf(quat_diff_sine(a, b));
}

// extension: the 8 cube corners (+-s/2)^3 rotated by the pose quaternion and translated
__device__ __forceinline__ void quat_rotate(const Quat q, float vx, float vy, float vz, float& ox, float& oy, float& oz) {
  // v' = v + 2 w (q_v x v) + 2 q_v x (q_v x v)
  const float tx = 2.0f * (q.y * vz - q.z * vy), ty = 2.0f * (q.z * vx - q.x * vz), tz = 2.0f * (q.x * vy - q.y * vx);
  ox = vx + q.w * tx + (q.y * tz - q.z * ty);
  oy = vy + q.w * ty + (q.z * tx - q.x * tz);
  oz = vz + q.w * tz + (q.x * ty - q.y * tx);
}

// 2 * (x - centre) / span with centre = (lo + hi) * 0.5, span = hi - lo (torch_utils.py:33-36)
__device__ __forceinline__ float scale_transform(float x, float centre, float span) {
  return __fdiv_rn(2.0f * (x - centre), span);
}
// x * (hi - lo) * 0.5 + centre (torch_utils.py:54-57)
__device__ __forceinline__ float unscale_transform(float x, float lo, float hi) {
  const float centre = (lo + hi) * 0.5f;
  return (x * (hi - lo)) * 0.5f + centre;
}
// torch.min / torch.max / torch.clamp propagate NaN; fminf / fmaxf would return the other operand and turn a diverged
// value into a legal-looking bound.  min.NaN / max.NaN compile to one FMNMX.NAN each (fminf / fmaxf: one FMNMX) and
// give the same bits for every non-NaN input.
__device__ __forceinline__ float min_nan(float a, float b) {
  float r;
  asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float max_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float saturate(float x, float lo, float hi) {  // torch_utils.py:60-75: max(min(x, hi), lo)
  return max_nan(min_nan(x, hi), lo);
}
// torch.clamp(x, lo, hi) (wrappers/vec_task.py:147, :162, :167)
__device__ __forceinline__ float clamp_nan(float x, float lo, float hi) { return min_nan(max_nan(x, lo), hi); }

// 1 / (e^{s x} + 2 + e^{-s x}) (envs/trifinger/rewards.py:20-34); generalised eps for the extension
__device__ __forceinline__ float lgsk(float x, float scale, float eps = 2.0f) {
  const float s = x * scale;
  const float den = (expf(s) + eps) + expf(-s);
  return __frcp_rn(den);
}

// ---------------------------------------------------------------------------------------
// Philox4x32-10 counter RNG (own key schedule; SURVEY.md §D option B)
// ---------------------------------------------------------------------------------------
struct U4 { uint32_t x, y, z, w; };

__device__ __forceinline__ U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = U4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

// [0, 1) with 24 random bits, the resolution of torch's CPU float uniform
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-8f; }

// sin and cos of x in [0, 2 pi] (all sampler angles are), ~1 ulp, without the libdevice calls' large-argument
// slow path: the reset code is executed by a handful of warps per SM, so its latency is its instruction count.
// Quadrant reduction with a 3-term split of pi/2 whose products with k <= 4 are exact, cephes minimax kernels.
__device__ __forceinline__ void sincos_2pi(float x, float& s, float& c) {
  const float kf = rintf(x * 0.636619772367581343f);
  float r = x - kf * 1.5703125f;
  r = r - kf * 4.837512969970703125e-4f;
  r = r - kf * 7.54978995489188216e-8f;
  const float z = r * r;
  const float sp = ((-1.9515295891e-4f * z + 8.3321608736e-3f) * z - 1.6666654611e-1f) * z * r + r;
  const float cp = ((2.443315711809948e-5f * z - 1.388731625493765e-3f) * z + 4.166664568298827e-2f) * z * z - 0.5f * z + 1.0f;
  const int k = (int)kf & 3;
  s = (k == 0) ? sp : (k == 1) ? cp : (k == 2) ? -sp : -cp;
  c = (k == 0) ? cp : (k == 1) ? -sp : (k == 2) ? -cp : sp;
}

// Box-Muller pair from two 32-bit words
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& n0, float& n1) {
  const float u1 = (float)((a >> 8) + 1u) * 5.9604644775390625e-8f;  // (0, 1]
  const float r = sqrtf(-2.0f * logf(u1));
  float sn, cs;
  sincos_2pi(kTwoPi * u01(b), sn, cs);
  n0 = r * cs;
  n1 = r * sn;
}

enum DrawPurpose : uint32_t { kPurposeReset = 0x52455345u, kPurposeGoal = 0x474f414cu, kPurposeNoise = 0x4e4f4953u,
                              kPurposeBias = 0x42494153u };

// Random numbers of ONE env for ONE reset call.  Either Philox keyed by
// (seed, global env id, purpose, epoch) or rows of injected arrays (test hook).
struct DrawSource {
  const float* inj_u;  // row pointer into [k,24] or nullptr
  const float* inj_n;  // row pointer into [k,8]  or nullptr
  uint32_t k0, k1, env_lo, env_hi_purpose, epoch_lo;

  __device__ __forceinline__ U4 block(uint32_t b) const {
    return philox4x32_10(U4{env_lo, env_hi_purpose, b, epoch_lo}, k0, k1);
  }
  // canonical uniform columns 4b .. 4b+3 (include/leibniz_b200.h: LG_INJECT_U_COLS) with ONE Philox evaluation
  __device__ __forceinline__ void uniform4(int b, float out[4]) const {
    if (inj_u) {
      const float* p = inj_u + 4 * b;
      out[0] = p[0]; out[1] = p[1]; out[2] = p[2]; out[3] = p[3];
      return;
    }
    const U4 r = block((uint32_t)b);
    out[0] = u01(r.x); out[1] = u01(r.y); out[2] = u01(r.z); out[3] = u01(r.w);
  }
  // four normals: cols 0..3 (first = true) or 4..7
  __device__ __forceinline__ void normal4(bool first, float out[4]) const {
    if (inj_n) {
      const float* p = inj_n + (first ? 0 : 4);
      out[0] = p[0]; out[1] = p[1]; out[2] = p[2]; out[3] = p[3];
      return;
    }
    const U4 r = block(first ? 8u : 9u);
    box_muller(r.x, r.y, out[0], out[1]);
    box_muller(r.z, r.w, out[2], out[3]);
  }
};

__device__ __forceinline__ DrawSource make_draws(const LgParams& P, uint64_t epoch, int64_t env_local,
                                                 uint32_t purpose, const float* inj_u, const float* inj_n,
                                                 int64_t rank) {
  DrawSource d;
  const uint64_t genv = (uint64_t)(P.env_offset + env_local);
  d.k0 = (uint32_t)P.seed;
  d.k1 = (uint32_t)(P.seed >> 32) ^ (uint32_t)(epoch >> 32);
  d.env_lo = (uint32_t)genv;
  d.env_hi_purpose = (uint32_t)(genv >> 32) ^ purpose;
  d.epoch_lo = (uint32_t)epoch;
  d.inj_u = (P.inject_draws && inj_u) ? inj_u + rank * LG_INJECT_U_COLS : nullptr;
  d.inj_n = (P.inject_draws && inj_n) ? inj_n + rank * LG_INJECT_N_COLS : nullptr;
  return d;
}

// ---------------------------------------------------------------------------------------
// torch's CUDA Philox stream (LG_RNG_TORCH; SURVEY.md §D option A)
// ---------------------------------------------------------------------------------------
// torch.rand / torch.randn of n fp32 elements (ATen/native/cuda/DistributionTemplates.h): a grid-stride kernel of
// g = min(SMs x threads_per_sm / 256, ceil(n / 256)) blocks of 256 threads; thread t runs curand_init(seed, t, offset)
// and draws one Philox4x32-10 block per round, whose four words feed elements t + T (4 r + lane), T = 256 g.
// `gmax` = SMs x (threads_per_sm / 256).  All sizes fit 32 bits: n < 18 x 2^23.
__host__ __device__ __forceinline__ uint32_t torch_threads(uint32_t n, uint32_t gmax) {
  const uint32_t g = (n + 255u) / 256u;
  return 256u * (g < gmax ? g : gmax);
}
// how far one call of n elements advances the generator's offset (calc_execution_policy)
__host__ __device__ __forceinline__ uint32_t torch_advance(uint32_t n, uint32_t gmax) {
  return n == 0 ? 0u : 4u * ((n - 1u) / (4u * torch_threads(n, gmax)) + 1u);
}
// the Philox block element j of such a call comes from, and its lane: curand_init puts the key = seed, the
// subsequence (thread) in the high counter words and offset / 4 + round in the low ones (curand_philox4x32_x.h)
__device__ __forceinline__ U4 torch_block(uint64_t seed, uint64_t offset, uint32_t n, uint32_t gmax, uint32_t j, int& lane) {
  const uint32_t T = torch_threads(n, gmax), q = j / T;
  lane = (int)(q & 3u);
  const uint64_t c = (offset >> 2) + (q >> 2);
  return philox4x32_10(U4{(uint32_t)c, (uint32_t)(c >> 32), j - q * T, 0u}, (uint32_t)seed, (uint32_t)(seed >> 32));
}
constexpr float kTwoPow32Inv = 2.3283064365386963e-10f;         // CURAND_2POW32_INV = 2^-32
constexpr float kTwoPow32Inv2Pi = kTwoPow32Inv * 6.2831855f;       // CURAND_2POW32_INV_2PI (exact product)
__device__ __forceinline__ uint32_t u4_lane(const U4 w, int lane) {
  return lane == 0 ? w.x : lane == 1 ? w.y : lane == 2 ? w.z : w.w;
}
// curand_uniform (x 2^-32 + 2^-33, in (0, 1]), then uniform_kernel's `v * 1 + 0` and `v == 1 ? 0 : v`
__device__ __forceinline__ float torch_uniform(uint32_t x) {
  const float v = (float)x * kTwoPow32Inv + kTwoPow32Inv * 0.5f;
  return v == 1.0f ? 0.0f : v;
}
// curand_normal4: _curand_box_muller on words (0, 1) and (2, 3), lane 0 / 2 = s sin v, lane 1 / 3 = s cos v.  torch's
// kernels are compiled with contraction on: v = y (2 pi 2^-32) + pi 2^-32 is one FFMA there (u's product is exact,
// logf's code does not depend on contraction, __sincosf is MUFU.SIN / MUFU.COS).
__device__ __forceinline__ float torch_normal(const U4 w, int lane) {
  const uint32_t a = lane < 2 ? w.x : w.z, b = lane < 2 ? w.y : w.w;
  const float u = (float)a * kTwoPow32Inv + kTwoPow32Inv * 0.5f;
  const float v = __fmaf_rn((float)b, kTwoPow32Inv2Pi, kTwoPow32Inv2Pi * 0.5f);
  const float s = sqrtf(-2.0f * logf(u));
  float sn, cs;
  __sincosf(v, &sn, &cs);
  return (lane & 1) ? cs * s : sn * s;
}

// The reference's calls of one _reset_impl (goal_only = false) or _goal_reset_impl (true) for a list of k envs, in
// its order (SURVEY.md §A.5, oracle/trifinger_oracle.py), and the canonical columns each one fills:
//   rand(k, 18) -> u0..17 (robot, random reset) | rand(k) x 3 -> u18, u19, u20 (object, random reset)
//   goal: rand(k) -> u21, u22 (difficulties -1, 1, 3, 4, 5), u23 (-1, 3, 4, 5); randn(k, 4) -> n0..3 (4, 5, 6);
//         rotation: randn(k, 3) -> n4..6, randn(k, 1) -> n7
// Column c of a call of width w is element rank x w + c of it.
struct TorchPlan {
  uint32_t k, gmax;
  bool robot, object, goal_uv, goal_w, goal_n, rot;
  __host__ __device__ uint32_t adv(uint32_t w) const { return torch_advance(k * w, gmax); }
  __host__ __device__ uint32_t goal_base() const { return (robot ? adv(18) : 0u) + (object ? 3u * adv(1) : 0u); }
  __host__ __device__ uint32_t goal_uniforms() const { return (goal_uv ? 2u : 0u) + (goal_w ? 1u : 0u); }
  __host__ __device__ uint32_t total() const {   // the whole list's advance
    return k == 0 ? 0u : goal_base() + goal_uniforms() * adv(1) + (goal_n ? adv(4) : 0u) + (rot ? adv(3) + adv(1) : 0u);
  }
};
__host__ __device__ __forceinline__ TorchPlan torch_plan(const LgParams& P, uint32_t k, bool goal_only) {
  TorchPlan p;
  const int d = P.task_difficulty;
  p.k = k;
  p.gmax = (uint32_t)P.sm_count * ((uint32_t)P.threads_per_sm / 256u);
  p.robot = !goal_only && P.robot_reset == LG_RESET_RANDOM;
  p.object = !goal_only && P.object_reset == LG_RESET_RANDOM;
  p.goal_uv = d == -1 || d == 1 || d == 3 || d == 4 || d == 5;
  p.goal_w = d == -1 || d == 3 || d == 4 || d == 5;
  p.goal_n = d == 4 || d == 5 || d == 6;
  p.rot = P.goal_rotation != 0;
  return p;
}

// DrawSource of the torch stream: the same interface, the canonical columns of ONE env (its rank in the list) drawn
// where the reference's calls would have put them.  One Philox evaluation per column (against one per four columns
// in the own stream); columns that no call fills read 0 and are never used by the samplers.
struct TorchDraws {
  uint64_t seed, base;   // base: the offset of the list's first call
  TorchPlan p;
  uint32_t rank;
  __device__ float uniform_col(int c) const {
    uint64_t o = base;
    uint32_t n = p.k, e = rank;
    if (c < 18) {
      if (!p.robot) return 0.0f;
      n = 18u * p.k; e = rank * 18u + (uint32_t)c;
    } else if (c < 21) {
      if (!p.object) return 0.0f;
      o += (p.robot ? p.adv(18) : 0u) + (uint32_t)(c - 18) * p.adv(1);
    } else {
      if (c < 23 ? !p.goal_uv : !p.goal_w) return 0.0f;
      o += p.goal_base() + (uint32_t)(c - 21) * p.adv(1);
    }
    int lane;
    const U4 w = torch_block(seed, o, n, p.gmax, e, lane);
    return torch_uniform(u4_lane(w, lane));
  }
  __device__ float normal_col(int c) const {
    uint64_t o = base + p.goal_base() + p.goal_uniforms() * p.adv(1);
    uint32_t n, e;
    if (c < 4) {
      if (!p.goal_n) return 0.0f;
      n = 4u * p.k; e = rank * 4u + (uint32_t)c;
    } else {
      if (!p.rot) return 0.0f;
      if (p.goal_n) o += p.adv(4);
      if (c < 7) { n = 3u * p.k; e = rank * 3u + (uint32_t)(c - 4); }
      else { o += p.adv(3); n = p.k; e = rank; }
    }
    int lane;
    const U4 w = torch_block(seed, o, n, p.gmax, e, lane);
    return torch_normal(w, lane);
  }
  __device__ void uniform4(int b, float out[4]) const {
#pragma unroll 1
    for (int q = 0; q < 4; ++q) out[q] = uniform_col(4 * b + q);
  }
  __device__ void normal4(bool first, float out[4]) const {
#pragma unroll 1
    for (int q = 0; q < 4; ++q) out[q] = normal_col((first ? 0 : 4) + q);
  }
};

__device__ __forceinline__ TorchDraws make_torch_draws(const LgParams& P, uint64_t seed, uint64_t base, uint32_t k,
                                                       bool goal_only, int64_t rank) {
  TorchDraws d;
  d.seed = seed; d.base = base;
  d.p = torch_plan(P, k, goal_only);
  d.rank = (uint32_t)rank;
  return d;
}

// ---------------------------------------------------------------------------------------
// samplers (envs/trifinger/sample.py)
// ---------------------------------------------------------------------------------------
// random_xy: r = sqrt(u0) * R, theta = 2 pi u1 (sample.py:22-34)
__device__ __forceinline__ void sample_disc(float u0, float u1, float radius_max, float& x, float& y) {
  float r = sqrtf(u0);
  r = r * radius_max;
  float sn, cs;
  sincos_2pi(kTwoPi * u1, sn, cs);
  x = r * cs;
  y = r * sn;
}
// random_yaw_orientation -> quaternion_from_euler_xyz(0, 0, 2 pi u) (sample.py:77-84, torch_utils.py:153-180)
__device__ __forceinline__ Quat sample_yaw(float u) {
  float sn, cs;
  sincos_2pi((kTwoPi * u) * 0.5f, sn, cs);
  return Quat{0.0f, 0.0f, sn, cs};
}
// random_orientation: normalize(randn(4), eps=1e-12) (sample.py:55-65); ATen's 2-norm over a
// contiguous 4-vector accumulates without contraction
__device__ __forceinline__ Quat sample_orientation(const float n[4]) {
  const float ss = ((n[0] * n[0] + n[1] * n[1]) + n[2] * n[2]) + n[3] * n[3];
  const float den = fmaxf(sqrtf(ss), 1e-12f);
  return Quat{__fdiv_rn(n[0], den), __fdiv_rn(n[1], den), __fdiv_rn(n[2], den), __fdiv_rn(n[3], den)};
}

// __sample_object_goal_poses (envs/trifinger/trifinger_env.py:1194-1265; draw order SURVEY.md §A.5), in two halves
// that share nothing — position (uniform columns 21..23) and orientation + angular velocity (the normals) — so that
// the fused kernel can run them on different warps: together they are the longest dependent chain of a reset.
__device__ __forceinline__ void sample_goal_position(const LgParams& P, const float ug[3], float pos[3]) {
  const int d = P.task_difficulty;
  float x = 0.0f, y = 0.0f, z;
  const float half = (float)P.cube_half_size;
  if (d == -1 || d == 1 || d == 3 || d == 4 || d == 5)
    sample_disc(ug[0], ug[1], (float)P.max_com_distance, x, y);
  if (d == -1 || d == 1) {
    z = half;
  } else if (d == 3) {
    z = (float)(P.cube_max_height - P.cube_half_size) * ug[2] + half;
  } else if (d == 4 || d == 5) {
    z = (float)(P.cube_max_height - P.cube_radius_3d) * ug[2] + (float)P.cube_radius_3d;
  } else {  // 2, 6: fixed position in the air
    z = (float)(P.cube_half_size + 0.05);
  }
  pos[0] = x; pos[1] = y; pos[2] = z;
}
template <class D>
__device__ __forceinline__ void sample_goal_orientation(const LgParams& P, const D dr, float yaw_u, float quat[4],
                                                        float angvel[3]) {
  const int d = P.task_difficulty;
  Quat q{0.0f, 0.0f, 0.0f, 1.0f};
  if (d == -1) q = sample_yaw(yaw_u);
  if (d == 4 || d == 5 || d == 6) {
    float n[4];
    dr.normal4(true, n);
    q = sample_orientation(n);
  }
  angvel[0] = angvel[1] = angvel[2] = 0.0f;
  if (P.goal_rotation) {  // random_angular_vel (sample.py:67-75)
    float n[4];
    dr.normal4(false, n);
    const float len = norm3(n[0], n[1], n[2]);
    const float mag = n[3] * (float)P.goal_rate_magnitude;
    angvel[0] = mag * __fdiv_rn(n[0], len);
    angvel[1] = mag * __fdiv_rn(n[1], len);
    angvel[2] = mag * __fdiv_rn(n[2], len);
  }
  quat[0] = q.x; quat[1] = q.y; quat[2] = q.z; quat[3] = q.w;
}

// Write the sampled goal into the goal buffers and the goal actor's root row (trifinger_env.py:1248-1265):
// `half` 0 = position (+ the row's linear velocity), 1 = orientation and angular velocity, 2 = both.
// D: DrawSource (own stream, injected columns) or TorchDraws.
template <class D>
__device__ __noinline__ void apply_goal_sample(const LgParams& P, const LgSimState& S, const LgBuffers& B,
                                               int64_t e, const D dr, int half = 2) {
  float* gp = B.goal_pose + e * 7;
  float* gm = B.goal_movement + e * 6;
  float* row = S.root_state + ((int64_t)P.actors_per_env * e + P.goal_slot) * 13;
  // goal columns 21..23 live in uniform block 5; the yaw of difficulty -1 is its last column
  float u5[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  if (half != 1 || P.task_difficulty == -1) dr.uniform4(5, u5);
  if (half != 1) {
    float pos[3];
    sample_goal_position(P, u5 + 1, pos);
#pragma unroll
    for (int c = 0; c < 3; ++c) { gp[c] = pos[c]; row[c] = pos[c]; row[7 + c] = gm[c]; }
  }
  if (half != 0) {
    float quat[4], angvel[3];
    sample_goal_orientation(P, dr, u5[3], quat, angvel);
#pragma unroll
    for (int c = 0; c < 4; ++c) { gp[3 + c] = quat[c]; row[3 + c] = quat[c]; }
#pragma unroll
    for (int c = 0; c < 3; ++c) { gm[3 + c] = angvel[c]; row[10 + c] = angvel[c]; }
  }
}

// extension (no reference code): the episode of env e (steps_count `steps` > 0) ends.  Its running return, length and
// success become its record and the return is zeroed; with per-term returns, so does the running row (32 contiguous
// bytes, two 128-bit pieces).  Out of line: the reset sub-task keeps its registers.
__device__ __noinline__ void end_episode(const LgBuffers& B, int64_t e, int64_t steps) {
  B.last_episode_return[e] = B.episode_return[e];
  B.last_episode_length[e] = steps;
  B.last_episode_success[e] = B.successes[e];
  B.episode_return[e] = 0.0f;
  if (B.episode_term_return) {
    float4* run = reinterpret_cast<float4*>(B.episode_term_return + e * LG_NUM_EPISODE_TERMS);
    float4* rec = reinterpret_cast<float4*>(B.last_episode_term_return + e * LG_NUM_EPISODE_TERMS);
    const float4 a = run[0], b = run[1];
    rec[0] = a; rec[1] = b;
    run[0] = run[1] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// extension (no reference code): the per-episode domain-randomisation offsets of env e, redrawn by its reset.  Always
// this build's Philox stream keyed by (seed, global env id, kPurposeBias, `epoch` = that of the reset's own draws),
// whatever stream or injected arrays the reset itself reads.  Philox block b < kBiasActionBlock holds obs columns
// 4b .. 4b+3 and is drawn only when one of them has sigma != 0; block kBiasActionBlock + b holds action columns
// 4b .. 4b+3.  Columns with sigma = 0 are stored as +0.0 (sigma x n would be -0.0 for n < 0).  draw_bias_block writes
// what block `b` covers (nothing for a block beyond the row); draw_bias all of them.
constexpr int kBiasActionBlock = 16;   // beyond the widest observation (50 columns: blocks 0 .. 12)
__device__ __forceinline__ void draw_bias_block(const LgParams& P, const LgBuffers& B, int64_t e, uint64_t epoch, int b) {
  const bool act = b >= kBiasActionBlock;
  const int width = act ? P.action_dim : 32 + P.action_dim, c0 = 4 * (act ? b - kBiasActionBlock : b);
  float* row = act ? B.action_bias : B.obs_bias;
  if (!row || c0 >= width) return;
  row += e * width;
  const unsigned m = act ? (P.dr_action_bias_sigma != 0.0f ? 15u : 0u) : (unsigned)(P.dr_bias_mask >> c0) & 15u;
  float n[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  if (m) {
    const U4 r = make_draws(P, epoch, e, kPurposeBias, nullptr, nullptr, 0).block((uint32_t)b);
    box_muller(r.x, r.y, n[0], n[1]);
    box_muller(r.z, r.w, n[2], n[3]);
  }
#pragma unroll
  for (int q = 0; q < 4; ++q)
    if (c0 + q < width)
      row[c0 + q] = ((m >> q) & 1u) ? (act ? P.dr_action_bias_sigma : P.dr_bias_sigma[c0 + q]) * n[q] : 0.0f;
}
// Out of line: the hook kernels keep their registers.
__device__ __noinline__ void draw_bias(const LgParams& P, const LgBuffers& B, int64_t e, uint64_t epoch) {
#pragma unroll 1
  for (int b = 0; b < kBiasActionBlock + (LG_MAX_ACTION_DIM + 3) / 4; ++b) draw_bias_block(P, B, e, epoch, b);
}

// _reset_impl for ONE env (trifinger_env.py:373-411, :1101-1192) cut into TEN independent sub-tasks, so that the
// fused kernel can run them on different warps (uniform control flow inside a warp) instead of one long serial
// chain per resetting env.  The draws are counter-based (or injected by column), so every sub-task fetches exactly
// the columns it needs; the arithmetic per output is unchanged.  Index lists are written by the caller.
//   0..4  robot joint state, uniform block b = canonical columns 4b..4b+3 (pos 0..8 | vel 9..17)     :1119-1144
//   5, 8  object position / orientation -> root row + history entry                                    :1164-1192
//   6, 9  goal position / orientation + movement (skipped when a goal reset of the same env follows)   :408-411
//   7     episode bookkeeping                                                                           :382-387
// The four long ones (5, 8, 6, 9: a Philox block each, then sqrt / sincos, or Box-Muller and a normalisation) are halves
// of what used to be two sub-tasks: the goal pose alone was a chain of ~550 instructions per resetting env.
// The zeroing of fingertip history entry 1 (:1146-1147) is a dead write in the reference (SURVEY.md §C2) and has
// no counterpart here.
constexpr int kResetSubtasks = 10;
// `dof_mirror`: optional second destination of the env's new joint-state row (the fused kernel's shared-memory copy,
// from which the torque is computed right afterwards).
// Out of line on purpose: the fused kernel reaches it from several call sites behind a block-uniform branch that most
// tiles never take; one copy keeps the kernel's hot path (no resets) small enough to sit in the instruction cache.
template <class D>
__device__ __noinline__ void reset_subtask(const LgParams& P, const LgSimState& S, const LgBuffers& B, int64_t e,
                                           int sub, const D dr, bool goal_reset_follows,
                                           float* dof_mirror = nullptr, bool clear_flag = true) {
  if (sub < 5) {
    if (P.robot_reset == LG_RESET_NONE) return;
    float* dof = S.dof_state + e * 18;
    float un[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    const bool random = P.robot_reset == LG_RESET_RANDOM;
    if (random) dr.uniform4(sub, un);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int i = 4 * sub + q;            // canonical column: joint position i (< 9) or velocity i - 9
      if (i < 18) {
        const bool is_vel = i >= 9;
        const int j = is_vel ? i - 9 : i;
        float x = is_vel ? P.dof_default_vel[j] : P.dof_default_pos[j];
        if (random) {
          const float n = 2.0f * un[q] - 1.0f;
          x = x + (float)(is_vel ? P.dof_vel_stddev : P.dof_pos_stddev) * n;
        }
        dof[2 * j + (is_vel ? 1 : 0)] = x;
        if (dof_mirror) dof_mirror[2 * j + (is_vel ? 1 : 0)] = x;
      }
    }
  } else if (sub == 5 || sub == 8) {
    // history entry 0 gets (pose, 0 velocity); its pose part is what the next post-physics pass reads as
    // "previous object pose" (SURVEY.md §C2).  5: position (+ zero velocities), 8: orientation.
    if (P.object_reset == LG_RESET_NONE) return;
    float* h = B.history + e * LG_HISTORY_COLS + 9;
    float* row = S.root_state + ((int64_t)P.actors_per_env * e + P.object_slot) * 13;
    if (sub == 5) {
      float x = 0.0f, y = 0.0f;
      const float z = (float)P.cube_half_size;
      if (P.object_reset == LG_RESET_RANDOM) {
        float ub4[4];
        dr.uniform4(4, ub4);                     // columns 18, 19 (disc radius, angle) are lanes 2, 3
        sample_disc(ub4[2], ub4[3], (float)P.max_com_distance, x, y);
      }
      h[0] = x; h[1] = y; h[2] = z;
      row[0] = x; row[1] = y; row[2] = z;
#pragma unroll
      for (int c = 7; c < 13; ++c) row[c] = 0.0f;
    } else {
      Quat q{0.0f, 0.0f, 0.0f, 1.0f};
      if (P.object_reset == LG_RESET_RANDOM) {
        float ub5[4];
        dr.uniform4(5, ub5);                     // column 20 (object yaw)
        q = sample_yaw(ub5[0]);
      }
      h[3] = q.x; h[4] = q.y; h[5] = q.z; h[6] = q.w;
      row[3] = q.x; row[4] = q.y; row[5] = q.z; row[6] = q.w;
    }
  } else if (sub == 6 || sub == 9) {
    // 6: goal position, 9: goal orientation + angular velocity
    if (!goal_reset_follows) apply_goal_sample(P, S, B, e, dr, sub == 6 ? 0 : 1);
  } else {
    // extension (no reference code): the episode ends here.  Every reset route comes through this sub-task, before the
    // counters are zeroed; steps_count == 0 means nothing happened since the previous reset and its record stays.
    if (B.episode_return) {
      const int64_t steps = B.steps_count[e];
      if (steps > 0) end_episode(B, e, steps);
    }
    if (clear_flag) B.reset[e] = 0;   // (the fused kernel's direct-prefix variant clears its tile's flags itself, later)
    B.steps_count[e] = 0;
    B.successes[e] = 0;
    float* act = B.action + e * P.action_dim;
    for (int c = 0; c < P.action_dim; ++c) act[c] = 0.0f;
  }
}

// all of it for one env, in the reference's order (hooks on explicit id lists)
template <class D>
__device__ __forceinline__ void reset_one_env(const LgParams& P, const LgSimState& S, const LgBuffers& B,
                                              int64_t e, const D dr) {
  reset_subtask(P, S, B, e, 7, dr, false);
  for (int sub = 0; sub < kResetSubtasks; ++sub)
    if (sub != 7) reset_subtask(P, S, B, e, sub, dr, false);
}

// _pre_step for ONE env (trifinger_env.py:442-498): action -> applied joint torque
__device__ __forceinline__ void torque_one_env(const LgParams& P, const float* __restrict__ act,
                                               const float* __restrict__ dof, float* __restrict__ out) {
#pragma unroll
  for (int j = 0; j < 9; ++j) {
    const float pos = dof[2 * j], vel = dof[2 * j + 1];
    float a = act[j];
    if (P.normalize_action) a = unscale_transform(a, P.action_low[j], P.action_high[j]);
    float tq;
    if (P.command_mode == LG_CMD_TORQUE) {
      tq = a;
    } else if (P.command_mode == LG_CMD_POSITION) {
      tq = P.kp[j] * (a - pos);
      tq = tq - P.kd[j] * vel;
    } else {
      float k = act[9 + j];
      if (P.normalize_action) k = unscale_transform(k, P.action_low[9 + j], P.action_high[9 + j]);
      tq = k * (a - pos);
      tq = tq - P.kd[j] * vel;
    }
    tq = saturate(tq, P.torque_low[j], P.torque_high[j]);
    if (P.apply_safety_damping) {
      tq = tq - P.safety_kd[j] * vel;
      tq = saturate(tq, P.torque_low[j], P.torque_high[j]);
    }
    out[j] = tq;
  }
}

}  // namespace lg
