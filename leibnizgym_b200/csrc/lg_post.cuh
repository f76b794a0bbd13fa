// post-physics pass of the TriFinger MDP hot path (sm_100a): obs/states fill + scale_transform, six reward terms,
// termination, step counters / timeouts / dones, episode statistics — one lane per output column.
// Included by lg_kernels.cu (single translation unit).  Reference paths are relative to /root/reference/leibnizgym/.
#pragma once

#include <cuda_bf16.h>

#include <type_traits>

#include "lg_device.cuh"

namespace lg {


// Programmatic dependent launch (PDL): a kernel launched with programmatic stream serialisation may
// begin (CTA scheduling, parameter fetch, address set-up) before its predecessor has finished;
// griddepcontrol.wait then blocks until the predecessor's grid has completed and its writes are
// visible.  Two ~2 us launches per step make this worth ~1/4 of the step time at 16k envs.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- TMA bulk copies (cp.async.bulk, SASS UBLKCP): one thread moves a whole contiguous tile slab -------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}"
      :: "r"(smem_u32(bar)), "r"(phase) : "memory");
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_store(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               :: "l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_store_commit_and_wait() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void fence_async_proxy() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// ---- per-thread asynchronous 16- and 4-byte copies (cp.async, SASS LDGSTS): global -> shared without a register -----
__device__ __forceinline__ void async_copy16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void async_copy4(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void async_copy_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void async_copy_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// =========================================================================================
// post-physics: one CTA = one tile of E envs, 4 threads per env
// =========================================================================================
constexpr int kPostThreads = 256;

template <int A, bool ASYM>
struct Layout {
  static constexpr int OBS = 32 + A;              // q 9 | qdot 9 | object pose 7 | goal pose 7 | action A
  static constexpr int STATE = OBS + 72;          // + object vel 6 | fingertips 39 | torque 9 | wrench 18
  static constexpr int ROW = ASYM ? STATE : OBS;  // floats per env in the staged tile
  static constexpr int OFF_OBJ = 18, OFF_GOAL = 25, OFF_ACT = 32;
  static constexpr int OFF_OBJVEL = OBS, OFF_TIPS = OBS + 6, OFF_TORQUE = OBS + 45, OFF_FT = OBS + 54;
};

// coefficient slots computed once per CTA (python-float arithmetic of the reward modules)
enum Coef { C_REACH = 0, C_MOVE, C_DIST, C_ROT_SCALE, C_ROT_SCHED, C_ROT_W, C_DELTA_RAMP, C_DELTA_W,
            C_OBJMOVE, C_DT, C_DT_RCP, C_POS_TOL, C_ROT_TOL, C_BONUS, C_KP_W, C_KP_SCALE, C_KP_EPS, C_NOISE_EPOCH,
            C_COUNT };

__host__ __device__ inline double sched_gate(const LgRewardTerm& t, double T) {  // rewards.py:56-60
  if (t.sched_start != t.sched_end) return (t.sched_start <= T && T <= t.sched_end) ? 1.0 : 0.0;
  return 1.0;
}
__host__ __device__ inline double sched_ramp(const LgRewardTerm& t, double T) {  // rewards.py:14-17, :169-172
  if (t.sched_start != t.sched_end) {
    const double v = (T - t.sched_start) / (t.sched_end - t.sched_start);
    return v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v);
  }
  return 1.0;
}
// The reward modules' Python-float arithmetic for env_steps_count = T.  Same code on host and device
// (IEEE double in both places), so the two clock modes produce identical coefficients.
__host__ __device__ inline void compute_coefs(const LgParams& P, double T, float* c) {
  const LgRewardTerm* t = P.terms;
  c[C_REACH] = (float)(t[0].weight * sched_gate(t[0], T));             // rewards.py:235
  c[C_MOVE] = (float)t[1].weight;                                       // rewards.py:263
  c[C_DIST] = (float)((t[2].weight * P.dt) * sched_gate(t[2], T));     // rewards.py:63
  c[C_ROT_SCALE] = (float)t[3].scale;                                   // rewards.py:137
  c[C_ROT_SCHED] = (float)(sched_gate(t[3], T) * P.dt);
  c[C_ROT_W] = (float)t[3].weight;                                      // rewards.py:139
  c[C_DELTA_RAMP] = (float)sched_ramp(t[4], T);                         // rewards.py:182
  c[C_DELTA_W] = (float)t[4].weight;                                    // rewards.py:184
  c[C_OBJMOVE] = (float)t[5].weight;                                    // rewards.py:91
  c[C_DT] = (float)P.dt;
  c[C_DT_RCP] = 1.0f / (float)P.dt;                                     // IEEE division: correctly rounded
  c[C_POS_TOL] = (float)P.position_tolerance;
  c[C_ROT_TOL] = (float)P.orientation_tolerance;
  c[C_BONUS] = (float)P.success_bonus;
  c[C_KP_W] = (float)(t[6].weight * P.dt);
  c[C_KP_SCALE] = (float)t[6].scale;
  c[C_KP_EPS] = (float)t[6].eps;
  // step identifier of the domain-randomisation noise stream: env_steps_count itself (bit pattern, not a value)
  union { uint32_t u; float f; } bits;
  bits.u = (uint32_t)(unsigned long long)T;
  c[C_NOISE_EPOCH] = bits.f;
}
static_assert(C_COUNT <= LG_NUM_COEF, "LgCoef too small");

// Fast division by a per-column constant: q = x*r, q' = fma(fma(-q, span, x), r, q) with r = fp32(1/span)
// correctly rounded (Markstein).  Contract, verified exhaustively by lg_selftest_division over all 2^32
// numerators for every span the env uses:
//   * 2^-100 <= |x| < 2^100 : bit-identical to IEEE x / span;
//   * x = +-0                : 0 (a negative zero comes out as +0);
//   * 0 < |x| < 2^-100       : within 1 ulp (the residual may be subnormal);
//   * |x| >= 2^100, inf      : flagged through `amax`; the caller redoes the column with __fdiv_rn.
__device__ __forceinline__ float div_by_const(float num, float span, float rcp, float& amax) {
  const float q = num * rcp;
  const float r = __fmaf_rn(-q, span, num);
  amax = fmaxf(amax, fabsf(num));
  return __fmaf_rn(r, rcp, q);
}
constexpr float kDivSafeMax = 1.2676506e30f;  // 2^100

// bfloat16 bits of a float, round-to-nearest-even (what torch's .to(torch.bfloat16) does)
__device__ __forceinline__ uint16_t to_bf16(float x) { return __bfloat16_as_ushort(__float2bfloat16_rn(x)); }

// One lane = one OUTPUT column of the tile ("role"), walking over the envs of its part of the tile.
// The role fixes, per lane and once per launch: the source pointer and row stride, the output column
// with its scale constants, and where (if anywhere) the raw value is staged for the reward math.
// The per-element code is then identical for every lane — no divergence although the lanes of a warp
// read from seven different tensors — and free of index arithmetic:
//     load   v[k] = src[k * stride]                       (all loads of the tile in flight at once)
//     emit   states[k][dcol] = obs[k][dcol] = scale(v[k])  (compile-time row offsets)
// Role order = output column order of the states row, except that the nine fingertip POSITION columns
// come right after the observation columns: the lanes that feed obs, the reward staging and the next
// history entry are then all in the first two warps of a part, and the other warps skip that code.
template <int A, bool ASYM, int E>
struct Roles {
  static constexpr int OBS = 32 + A;
  static constexpr int R_TIPPOS = OBS;                  // 9 roles
  static constexpr int R_TIPREST = R_TIPPOS + 9;        // 30 roles (asymmetric only)
  static constexpr int R_OBJVEL = R_TIPREST + 30;       // 6
  static constexpr int R_FT = R_OBJVEL + 6;             // 18
  static constexpr int R_TQ = R_FT + 18;                // 9
  static constexpr int R_END = ASYM ? R_TQ + 9 : R_TIPREST;
  static constexpr int LANES = R_END <= 64 ? 64 : 128;  // role lanes per tile part
  static constexpr int PARTS = kPostThreads / LANES;    // the tile's envs are split over the parts
  static constexpr int EP = E / PARTS;                  // envs per lane
  static_assert(E % PARTS == 0 && E <= 32, "tile must split evenly; the reward math uses one lane per env");
  static constexpr int FRONT = R_TIPREST;               // roles < FRONT may feed obs / staging / history
  static constexpr int FRONT_WARPS = (FRONT + 31) / 32; // warps of a part that hold such roles
  // warps that meet at the staging barrier: the four reward warps and the front warps of every part
  static constexpr int STAGE_WARPS = LANES == 128 ? 4 + (PARTS - 1) * FRONT_WARPS : kPostThreads / 32;
  static_assert(R_END <= LANES, "more output columns than role lanes");
};

// What a role lane needs to know, independent of the tile: where its column comes from, where it goes, and whether
// the raw value is staged for the reward math / kept as next step's history.
struct RoleInfo {
  int src_id;        // 0 dof_state, 1 root_state, 2 goal_pose, 3 action, 4 rigid_body, 5 ft_sensors, 6 dof_force
  int src_off;       // float offset of (env 0, column) inside that tensor
  int stride;        // source row stride in floats
  int dcol;          // output column (scaled): states[:, dcol], obs[:, dcol] if dcol < OBS; -1: none
  int stage_id;      // 0 none, 1 object pose, 2 goal pose, 3 fingertip positions
  int stage_off;     // column inside that staging array
  int stage_stride;  // staging row stride
  int hist_col;      // column of the NEXT history entry this lane provides, or -1
};

template <int A, bool ASYM>
__device__ __forceinline__ RoleInfo role_info(const LgParams& P, int role) {
  using L = Layout<A, ASYM>;
  using R = Roles<A, ASYM, 32>;   // the role ranges do not depend on the tile size
  RoleInfo r;
  r.stage_id = 0; r.stage_off = 0; r.stage_stride = 0; r.hist_col = -1;
  const int body_stride = P.bodies_per_env * 13, actor_stride = P.actors_per_env * 13;
  auto tip_off = [&](int tip, int c) {
    const int body = tip == 0 ? P.fingertip_body[0] : tip == 1 ? P.fingertip_body[1] : P.fingertip_body[2];
    return body * 13 + c;
  };
  if (role < 18) {                                         // dof_state (pos, vel) interleaved  trifinger_env.py:1003-1007
    r.src_id = 0; r.src_off = role; r.stride = 18;
    r.dcol = (role & 1) * 9 + (role >> 1);
  } else if (role < 25) {                                  // object pose (root row of actor 4e+2)  :975, :1011
    const int c = role - 18;
    r.src_id = 1; r.src_off = P.object_slot * 13 + c; r.stride = actor_stride;
    r.dcol = L::OFF_OBJ + c;
    r.stage_id = 1; r.stage_off = c; r.stage_stride = 7; r.hist_col = 9 + c;
  } else if (role < 32) {                                  // goal pose buffer                  :1015
    const int c = role - 25;
    r.src_id = 2; r.src_off = c; r.stride = 7;
    r.dcol = L::OFF_GOAL + c;
    r.stage_id = 2; r.stage_off = c; r.stage_stride = 7;
  } else if (role < R::OBS) {                              // last action                       :1019
    const int c = role - 32;
    r.src_id = 3; r.src_off = c; r.stride = A;
    r.dcol = L::OFF_ACT + c;
  } else if (role < R::R_TIPREST) {                        // fingertip positions (bodies 6/11/16)  :974, :1040
    const int j = role - R::R_TIPPOS, tip = j / 3, c = j - tip * 3;
    r.src_id = 4; r.src_off = tip_off(tip, c); r.stride = body_stride;
    r.dcol = ASYM ? L::OFF_TIPS + tip * 13 + c : -1;
    r.stage_id = 3; r.stage_off = j; r.stage_stride = 9; r.hist_col = j;
  } else if (role < R::R_OBJVEL) {                         // fingertip orientation + velocity
    const int j = role - R::R_TIPREST, tip = j / 10, c = 3 + (j - tip * 10);
    r.src_id = 4; r.src_off = tip_off(tip, c); r.stride = body_stride;
    r.dcol = L::OFF_TIPS + tip * 13 + c;
  } else if (role < R::R_FT) {                             // object velocity                   :1035
    const int c = role - R::R_OBJVEL;
    r.src_id = 1; r.src_off = P.object_slot * 13 + 7 + c; r.stride = actor_stride;
    r.dcol = L::OFF_OBJVEL + c;
  } else if (role < R::R_TQ) {                             // fingertip wrenches                :1051
    const int c = role - R::R_FT;
    r.src_id = 5; r.src_off = c; r.stride = 18;
    r.dcol = L::OFF_FT + c;
  } else {                                                 // dof torque                        :1047
    const int c = role - R::R_TQ;
    r.src_id = 6; r.src_off = c; r.stride = 9;
    r.dcol = L::OFF_TORQUE + c;
  }
  return r;
}

// Statistics in fixed point (see reward_combine): scale 2^30, values must stay below 2^28 so that 32 of them fit int64.
constexpr float kStatFixScale = 1073741824.0f, kStatFixMax = 268435456.0f;
// What a statistics lane multiplies its integer sum by: lane s of the combine warp owns slot s.  Reward-term, reward and success
// entries are means over this shard (trifinger_env.py:554, :1098), the rest are counts (:1067, :1076).  Evaluated in
// the kernel prologue (an fp64 division is a chain of ~10 dependent fp64 operations, each ~0.1-0.2 us for a lone warp
// on this part).  When the env count is a power of two the factor is one too and only its exponent is kept: the
// integer sum then becomes a double by integer instructions alone (i64_times_pow2).
struct StatScale { double factor; int shift; bool pow2; };
__device__ __forceinline__ StatScale stat_lane_scale(const LgParams& P, int slot) {
  const long long n = P.stats_num_envs > 0 ? P.stats_num_envs : P.num_envs;
  const bool float_mean = slot < LG_STAT_POSITION_GOAL || slot == LG_STAT_REWARD;
  const bool mean = float_mean || slot == LG_STAT_SUCCESSES;
  StatScale sc;
  sc.pow2 = (n & (n - 1)) == 0;
  sc.shift = (float_mean ? -30 : 0) - (mean ? 63 - __clzll(n) : 0);
  sc.factor = (mean ? 1.0 / (double)n : 1.0) * (float_mean ? 1.0 / 1073741824.0 : 1.0);
  return sc;
}
// v * 2^shift as a double, by integer instructions (round to nearest even beyond 53 bits; no overflow / underflow
// for the shifts used here)
__device__ __forceinline__ double i64_times_pow2(long long v, int shift) {
  if (v == 0) return 0.0;
  const unsigned long long a = v < 0 ? 0ull - (unsigned long long)v : (unsigned long long)v;
  const int lz = __clzll((long long)a);
  const unsigned long long m = a << lz;                         // leading one at bit 63
  unsigned long long mant = m >> 11;                            // 53 bits, leading one included
  const unsigned rem = (unsigned)m & 0x7ffu;
  mant += (rem > 0x400u || (rem == 0x400u && (mant & 1ull))) ? 1ull : 0ull;
  // a carry out of the mantissa lands in the exponent field, which is what rounding up to a power of two means
  unsigned long long bits = ((unsigned long long)(1023 + 63 - lz + shift) << 52) + (mant - (1ull << 52));
  if (v < 0) bits |= 1ull << 63;
  return __longlong_as_double((long long)bits);
}
__device__ __noinline__ double i64_times_factor(long long v, double factor) { return (double)v * factor; }
// exact sum of a 64-bit integer (|x| < 2^58) over the warp's lanes: three limbs through the warp-reduce unit
// (REDUX), independent of each other, instead of five dependent shuffle + add rounds
__device__ __forceinline__ long long warp_sum_i64(long long x) {
  const unsigned l0 = (unsigned)x & 0x1fffffu, l1 = (unsigned)(x >> 21) & 0x1fffffu;
  const int l2 = (int)(x >> 42);
  const unsigned s0 = __reduce_add_sync(0xffffffffu, l0), s1 = __reduce_add_sync(0xffffffffu, l1);
  const int s2 = __reduce_add_sync(0xffffffffu, l2);
  return (long long)s0 + ((long long)s1 << 21) + ((long long)s2 << 42);
}
// Cold path of the statistics: fp64 butterflies over the lanes, for values outside the fixed-point window.  The terms
// come by value: an array argument would pin the caller's copy to local memory.
__device__ __noinline__ double stat_sums_fp64(float t0, float t1, float t2, float t3, float t4, float t5, float t6,
                                              float reward, unsigned active, int lane) {
  const float x[8] = {t0, t1, t2, t3, t4, t5, t6, reward};
  double mine = 0.0;
  for (int k = 0; k <= 7; ++k) {
    if (k < 7 && !((active >> k) & 1)) continue;
    double acc = (double)x[k];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == (k < 7 ? LG_STAT_TERM0 + k : LG_STAT_REWARD)) mine = acc;
  }
  return mine;
}
// The same for one value per lane (episode returns outside the fixed-point window); every lane gets the sum.
__device__ __noinline__ double warp_sum_fp64(float x) {
  double acc = (double)x;
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return acc;
}

// Per-term returns of the fresh records (env e, or -1: none on this lane) folded into episode_term_stats: lane
// `tslot` keeps slot tslot, by the same means as the episode returns (2^-30 fixed point, fp64 butterflies for
// |x| >= 2^28, inf and NaN; one decision for the warp).  Called by the combine warp when it holds fresh records; out
// of line, so that the warp's common path keeps its registers.
__device__ __noinline__ void episode_term_fold(const LgBuffers& B, int64_t e, int tslot) {
  float4 ra = make_float4(0.f, 0.f, 0.f, 0.f), rb = ra;
  if (e >= 0) {
    const float4* rec = reinterpret_cast<const float4*>(B.last_episode_term_return + e * LG_NUM_EPISODE_TERMS);
    ra = rec[0]; rb = rec[1];
  }
  const float x[LG_NUM_EPISODE_TERMS] = {ra.x, ra.y, ra.z, ra.w, rb.x, rb.y, rb.z, rb.w};
  bool fits = true;
#pragma unroll
  for (int k = 0; k < LG_NUM_EPISODE_TERMS; ++k) fits = fits && fabsf(x[k]) < kStatFixMax;
  double sum = 0.0;
  if (__all_sync(0xffffffffu, fits)) {
    long long fixed = 0;
#pragma unroll
    for (int k = 0; k < LG_NUM_EPISODE_TERMS; ++k) {
      const long long t = warp_sum_i64(__float2ll_rn(x[k] * kStatFixScale));
      if (tslot == k) fixed = t;
    }
    sum = i64_times_pow2(fixed, -30);
  } else {
#pragma unroll
    for (int k = 0; k < LG_NUM_EPISODE_TERMS; ++k) {   // cold
      const double t = warp_sum_fp64(x[k]);
      if (tslot == k) sum = t;
    }
  }
  if (tslot >= 0 && tslot < LG_NUM_EPISODE_TERMS) atomicAdd(B.episode_term_stats + tslot, sum);
}

constexpr int kCombineWarp = 3;   // the reward warp with the shortest sub-task (previous angle) also combines

// ======== reward warps: lane = env, warp = sub-task (uniform control flow inside a warp) ================
// Called by the four reward warps (threads 0..127) of a post-physics CTA once the tile's object pose, goal pose,
// fingertip positions and previous history entry are staged in shared memory (raw, unscaled); E <= 32 envs per tile.
//   warp 0: finger_reach_object_rate | warp 1: finger_move_penalty, object_dist, object_move | warp 2: current angle,
//   object_rot | warp 3: previous angle.  The results wait in `s_part` for reward_combine.
template <int E, bool EXT>
__device__ __forceinline__ void reward_subtasks(const LgParams& P, int nvalid,
                                                const float* s_obj, const float* s_goal, const float* s_tips,
                                                const float* s_hist, const float* s_coef, float* s_part) {
  constexpr int HS = LG_HISTORY_COLS + 1;
  const int tid = threadIdx.x;
  const int rw = tid >> 5, renv = tid & 31;
  // ======== reward warps: lane = env, warp = sub-task (uniform control flow inside a warp) ================
  {
    const int env = renv;
    const bool live = renv < nvalid;
    const float* obj = s_obj + env * 7;
    const float* goal = s_goal + env * 7;
    const float* tips = s_tips + env * 9;
    const float* hist = s_hist + env * HS;
    if (live) {
      const float gx = goal[0], gy = goal[1], gz = goal[2];
      if (rw == 0) {
        // finger_reach_object_rate (rewards.py:219-235): sum_i (|tip_i - obj| - |tip_i' - obj'|)
        const float ox = obj[0], oy = obj[1], oz = obj[2];
        const float px = hist[9], py = hist[10], pz = hist[11];
        float acc = 0.0f;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const float cur = norm3(tips[3 * i] - ox, tips[3 * i + 1] - oy, tips[3 * i + 2] - oz);
          const float prev = norm3(hist[3 * i] - px, hist[3 * i + 1] - py, hist[3 * i + 2] - pz);
          acc = acc + (cur - prev);
        }
        s_part[(0) * E + env] = s_coef[C_REACH] * acc;
      } else if (rw == 1) {
        // finger_move_penalty (rewards.py:261-263): sum_9 ((tip - tip') / dt)^2
        const float dt = s_coef[C_DT], dt_rcp = s_coef[C_DT_RCP];
        float acc = 0.0f, dmax = 0.0f;
#pragma unroll
        for (int k = 0; k < 9; ++k) {
          const float d = div_by_const(tips[k] - hist[k], dt, dt_rcp, dmax);
          acc = acc + d * d;
        }
        if (!(dmax < kDivSafeMax)) {  // cold
          acc = 0.0f;
          for (int k = 0; k < 9; ++k) {
            const float d = __fdiv_rn(tips[k] - hist[k], dt);
            acc = acc + d * d;
          }
        }
        s_part[(1) * E + env] = s_coef[C_MOVE] * acc;
        // object_dist (rewards.py:62-63) and object_move (rewards.py:88-91)
        const float d = norm3(obj[0] - gx, obj[1] - gy, obj[2] - gz);
        const float dprev = norm3(hist[9] - gx, hist[10] - gy, hist[11] - gz);
        s_part[(2) * E + env] = lgsk(d, 50.0f) * s_coef[C_DIST];
        s_part[(3) * E + env] = s_coef[C_OBJMOVE] * (d - dprev);
        s_part[(4) * E + env] = d;
      } else {
        const Quat gq{goal[3], goal[4], goal[5], goal[6]};
        if (rw == 2) {
          // object_rot (rewards.py:134-139): w * (gate*dt) / (scale*|theta| + scale)
          const Quat oq{obj[3], obj[4], obj[5], obj[6]};
          const float theta = quat_diff_rad(oq, gq);
          const float den = s_coef[C_ROT_SCALE] * fabsf(theta) + s_coef[C_ROT_SCALE];
          s_part[(5) * E + env] = (__frcp_rn(den) * s_coef[C_ROT_SCHED]) * s_coef[C_ROT_W];
          s_part[(6) * E + env] = theta;
        } else {
          // previous-orientation angle for object_rot_delta (rewards.py:179)
          const Quat pq{hist[12], hist[13], hist[14], hist[15]};
          s_part[(7) * E + env] = fabsf(quat_diff_rad(pq, gq));
        }
      }
      // extension (no reference code, SURVEY.md §8c(i)): keypoint pose reward
      //   w dt mean_k lgsk(|kp_k - kp_k^goal|; scale, eps), kp_k = p + R(q) c_k over the 8 cube corners;
      // two corners per reward warp, summed by the combine warp
      if (EXT && ((P.term_active_mask >> LG_TERM_KEYPOINT) & 1)) {
        const Quat oq{obj[3], obj[4], obj[5], obj[6]};
        const Quat gq{goal[3], goal[4], goal[5], goal[6]};
        const float h = (float)P.cube_half_size;
        float acc = 0.0f;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int kk = 2 * rw + q;
          const float cx = (kk & 1) ? h : -h, cy = (kk & 2) ? h : -h, cz = (kk & 4) ? h : -h;
          float ax, ay, az, bx, by, bz;
          quat_rotate(oq, cx, cy, cz, ax, ay, az);
          quat_rotate(gq, cx, cy, cz, bx, by, bz);
          const float dd = norm3((obj[0] + ax) - (gx + bx), (obj[1] + ay) - (gy + by), (obj[2] + az) - (gz + bz));
          acc = acc + lgsk(dd, s_coef[C_KP_SCALE], s_coef[C_KP_EPS]);
        }
        s_part[(8 + rw) * E + env] = acc;
      }
    }
    LG_TP(0, 5, tid == 0); LG_TP(0, 16, tid == 32); LG_TP(0, 17, tid == 64); LG_TP(0, 18, tid == 96);
  }
}

// Second half of the reward chain, called by the combine warp (kCombineWarp) alone, after it has stored its own
// columns: it waits for the other three reward warps' arrival at barrier 1, then combines the sub-task results,
// terminates, counts and accumulates the statistics.
template <int E, bool EXT>
__device__ __forceinline__ void reward_combine(const LgParams& P, const LgBuffers& B, int64_t e0, int nvalid,
                                               const float* s_coef, const float* s_part,
                                               uint8_t in_goal_reset, uint8_t in_succ, uint8_t in_reset, int64_t in_steps,
                                               float in_return, float4* s_term_row, const StatScale& stat_scale) {
  const int tid = threadIdx.x;
  const int renv = tid & 31;
  asm volatile("bar.sync 1, 128;" ::: "memory");  // the other three reward warps have arrived: their results are in s_part
  LG_TP(0, 6, renv == 0);
  {
    // ---- combine, terminate, count (one lane per env) -------------------------------------------------
    const int env = renv;
    const bool live = renv < nvalid;
    float terms[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // per-env values of the statistics (0 beyond the tile)
    float reward = 0.0f;  // trifinger_env.py:511, :551-553 — accumulation in dict order (the extension term last)
    bool pos_ok = false, rot_ok = false, succ = false, reset = false, dn = false;
    // extension (episode statistics): the record of an episode that ended since the previous pass (length 0: none)
    int64_t ep_len = 0;
    float ep_return = 0.0f;
    bool ep_succ = false;
    if (live) {
      const int64_t e = e0 + env;
      const float dist = s_part[(4) * E + env], theta = s_part[(6) * E + env];
      // object_rot_delta (rewards.py:180-184): w * (ramp * (|theta| - |theta'|))
      const float t_delta = s_coef[C_DELTA_W] * (s_coef[C_DELTA_RAMP] * (fabsf(theta) - s_part[(7) * E + env]));
      const bool kp_on = EXT && ((P.term_active_mask >> LG_TERM_KEYPOINT) & 1);
      terms[0] = s_part[(0) * E + env]; terms[1] = s_part[(1) * E + env]; terms[2] = s_part[(2) * E + env];
      terms[3] = s_part[(5) * E + env]; terms[4] = t_delta; terms[5] = s_part[(3) * E + env];
      terms[6] = kp_on ? s_coef[C_KP_W] * ((((s_part[(8) * E + env] + s_part[(9) * E + env]) + s_part[(10) * E + env]) + s_part[(11) * E + env]) * 0.125f)
                       : 0.0f;
#pragma unroll
      for (int k = 0; k < 7; ++k) {
        if ((P.term_active_mask >> k) & 1) reward = reward + terms[k];
        if (B.term_rewards) B.term_rewards[(int64_t)k * P.num_envs + e] = terms[k];
      }
      // __check_termination (trifinger_env.py:1053-1099)
      pos_ok = dist <= s_coef[C_POS_TOL];
      rot_ok = theta <= s_coef[C_ROT_TOL];
      bool done;
      if (P.task_difficulty < 4) done = pos_ok;
      else if (P.task_difficulty == 4) done = pos_ok && rot_ok;
      else done = rot_ok;
      bool goal_reset = in_goal_reset != 0;
      succ = in_succ != 0;
      if (P.success_activate) {
        if (done) reward = reward + s_coef[C_BONUS];
        goal_reset = done;
        succ = succ || goal_reset;
        B.goal_reset[e] = goal_reset;
      } else {
        succ = goal_reset && succ;
      }
      B.successes[e] = succ;
      B.reward[e] = reward;
      // step counter, timeout, dones (envs/env_base.py:391-399)
      reset = in_reset != 0;
      if (P.fuse_bookkeeping) {
        const int64_t steps = in_steps + 1;
        B.steps_count[e] = steps;
        if (P.episode_length >= 0) reset = reset || (steps >= P.episode_length);
        B.reset[e] = reset;
      }
      dn = reset && goal_reset;
      if (B.dones) B.dones[e] = dn;
      // extension (no reference code): running return, and the record a reset wrote since the previous pass.  That
      // reset zeroed the step counter, so the record is fresh exactly when in_steps == 0 and it holds an episode.
      if (EXT && B.episode_return) {
        B.episode_return[e] = in_return + reward;
        if (in_steps == 0) {
          const int64_t len = B.last_episode_length[e];
          if (len > 0) { ep_len = len; ep_return = B.last_episode_return[e]; ep_succ = B.last_episode_success[e] != 0; }
        }
      }
      // extension (per-term episode returns): the env's running row, staged in shared memory by the copy issued with
      // the flag loads, takes each active term's value as the reward above took it, and the bonus when it was paid
      if (EXT && B.episode_term_return) {
        async_copy_wait_all();
        float4 a = s_term_row[0], b = s_term_row[1];
        const unsigned m = (unsigned)P.term_active_mask;
        if (m & 1u) a.x = a.x + terms[0];
        if (m & 2u) a.y = a.y + terms[1];
        if (m & 4u) a.z = a.z + terms[2];
        if (m & 8u) a.w = a.w + terms[3];
        if (m & 16u) b.x = b.x + terms[4];
        if (m & 32u) b.y = b.y + terms[5];
        if (m & 64u) b.z = b.z + terms[6];
        if (P.success_activate && goal_reset) b.w = b.w + s_coef[C_BONUS];   // goal_reset == done: the bonus was paid
        float4* run = reinterpret_cast<float4*>(B.episode_term_return + e * LG_NUM_EPISODE_TERMS);
        run[0] = a; run[1] = b;
      }
    }
    LG_TP(0, 7, renv == 0);
    // ---- episode statistics (trifinger_env.py:554, :1067-1068, :1076, :1098-1099): per-CTA sums over the warp's
    // lanes (lane = env), lane s keeps slot s, then ONE reduction instruction carries all slots of the CTA to the 104
    // contiguous bytes of the statistics vector — no fence, no second kernel, one L2 atomic transaction per CTA (one
    // per slot was measured at 12.3 instead of 7.1 us for the whole kernel at 16 384 envs).
    // Counts come from ballots.  The float sums (terms and reward) are taken in 2^-30 fixed point through the
    // warp-reduce unit: a dependent fp64 operation costs this warp ~0.1-0.2 us on this part (measured: 20
    // dependent DADDs = 1.9 us; I2F + DMUL = 0.42 us), and integer sums do not depend on the order of the additions.  Exact for |x| >= 2^-6, resolution 9.3e-10 below; values that do not fit (|x| >= 2^28, inf, NaN)
    // take the fp64 butterflies (stat_sums_fp64, cold) so that a diverged env still shows up as inf / NaN.
    unsigned active = (unsigned)P.term_active_mask & 0x7fu;
    bool fits = fabsf(reward) < kStatFixMax;
#pragma unroll
    for (int k = 0; k < 7; ++k) fits = fits && (!((active >> k) & 1) || fabsf(terms[k]) < kStatFixMax);
    const unsigned m_pos = __ballot_sync(0xffffffffu, pos_ok), m_rot = __ballot_sync(0xffffffffu, rot_ok);
    const unsigned m_succ = __ballot_sync(0xffffffffu, succ), m_reset = __ballot_sync(0xffffffffu, reset);
    const unsigned m_dn = __ballot_sync(0xffffffffu, dn);
    double mine;
    LG_TP(0, 23, renv == 0);
    if (__all_sync(0xffffffffu, fits)) {
      // all eight sums unconditionally (an inactive term contributes zeros): no branches between them, so the
      // conversions and reductions of the slots overlap
      long long tot[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float x = k < 7 ? (((active >> k) & 1) ? terms[k] : 0.0f) : reward;
        tot[k] = warp_sum_i64(__float2ll_rn(x * kStatFixScale));   // scaling by 2^30 is exact
      }
      LG_TP(0, 24, renv == 0);
      long long fixed = 0;
#pragma unroll
      for (int k = 0; k < 7; ++k)
        if (env == LG_STAT_TERM0 + k) fixed = tot[k];
      if (env == LG_STAT_REWARD) fixed = tot[7];
      if (env == LG_STAT_POSITION_GOAL) fixed = __popc(m_pos);
      if (env == LG_STAT_ORIENTATION_GOAL) fixed = __popc(m_rot);
      if (env == LG_STAT_SUCCESSES) fixed = __popc(m_succ);
      if (env == LG_STAT_RESETS) fixed = __popc(m_reset);
      if (env == LG_STAT_DONES) fixed = __popc(m_dn);
      // this lane's slot: x 2^-30 / N (float means), 1 / N (success rate) or 1 (counts)
      if (stat_scale.pow2) mine = i64_times_pow2(fixed, stat_scale.shift);
      else mine = i64_times_factor(fixed, stat_scale.factor);   // out of line: keeps the fp64 pipe off the common path
    } else {
      mine = stat_sums_fp64(terms[0], terms[1], terms[2], terms[3], terms[4], terms[5], terms[6], reward, active, env);
      if (env == LG_STAT_POSITION_GOAL) mine = (double)__popc(m_pos);
      if (env == LG_STAT_ORIENTATION_GOAL) mine = (double)__popc(m_rot);
      if (env == LG_STAT_SUCCESSES) mine = (double)__popc(m_succ);
      if (env == LG_STAT_RESETS) mine = (double)__popc(m_reset);
      if (env == LG_STAT_DONES) mine = (double)__popc(m_dn);
      const bool is_mean = env < LG_STAT_POSITION_GOAL || env == LG_STAT_SUCCESSES || env == LG_STAT_REWARD;
      if (is_mean) mine = mine / (double)(P.stats_num_envs > 0 ? P.stats_num_envs : P.num_envs);
    }
#ifdef LG_TRACE
    if (mine == 1.2345e300) return;   // make the stamp below wait for the scaled value
#endif
    LG_TP(0, 25, renv == 0);
    // extension: finished episodes on the lanes after LG_STAT_DONES, by the same means — ballots and integer sums
    // (exact), the returns in 2^-30 fixed point with the fp64 butterflies for |x| >= 2^28, inf and NaN.  A warp
    // without fresh records adds nothing.
    if (EXT && B.episode_stats) {
      const unsigned m_ep = __ballot_sync(0xffffffffu, ep_len > 0);
      if (m_ep) {
        const unsigned m_ep_succ = __ballot_sync(0xffffffffu, ep_succ);
        const long long len_sum = warp_sum_i64(ep_len);
        double ret_sum;
        if (__all_sync(0xffffffffu, fabsf(ep_return) < kStatFixMax))
          ret_sum = i64_times_pow2(warp_sum_i64(__float2ll_rn(ep_return * kStatFixScale)), -30);
        else
          ret_sum = warp_sum_fp64(ep_return);   // cold
        const int slot = env - (LG_STAT_DONES + 1);
        double ep = (double)__popc(m_ep);
        if (slot == LG_EPISODE_RETURN_SUM) ep = ret_sum;
        if (slot == LG_EPISODE_LENGTH_SUM) ep = (double)len_sum;
        if (slot == LG_EPISODE_SUCCESSES) ep = (double)__popc(m_ep_succ);
        if (slot >= 0 && slot < LG_NUM_EPISODE_STATS) atomicAdd(B.episode_stats + slot, ep);
        // per-term returns on the next eight lanes: one decision for the warp, as for the step statistics
        if (B.episode_term_stats) episode_term_fold(B, ep_len > 0 ? e0 + env : -1, slot - LG_NUM_EPISODE_STATS);
      }
    }
    if (env <= LG_STAT_DONES) atomicAdd(B.step_stats + env, mine);
    LG_TP(0, 8, renv == 0);
  }
}

template <int A, bool ASYM, bool REWARD, bool CLIP, int E, bool EXT>
__global__ void __launch_bounds__(kPostThreads, 4)
post_physics_kernel(const __grid_constant__ LgParams P, const __grid_constant__ LgSimState S,
                    const __grid_constant__ LgBuffers B, const __grid_constant__ LgCoef CF) {
  using L = Layout<A, ASYM>;
  using R = Roles<A, ASYM, E>;          // E envs per CTA
  constexpr int EP = R::EP;
  constexpr int HS = LG_HISTORY_COLS + 1;  // padded row: lane-per-env reads stay conflict free
  // only what the reward terms read is staged in shared memory (raw, unscaled)
  __shared__ float s_obj[E * 7];        // object pose
  __shared__ float s_goal[E * 7];       // goal pose
  __shared__ float s_tips[E * 9];       // fingertip positions
  __shared__ float s_hist[E * HS];      // previous fingertip positions (9) + previous object pose (7)
  __shared__ float s_coef[C_COUNT];
  __shared__ float s_part[12][E];       // sub-task results of the reward warps
  __shared__ float s_noise[EXT ? L::OBS : 1][EXT ? E + 1 : 1];   // extension: standard normals of the obs columns
  __shared__ float4 s_term_run[EXT ? 2 * E : 1];   // extension: the tile's running per-term episode returns
  __shared__ float s_bias[EXT ? L::OBS : 1][EXT ? E + 1 : 1];   // extension: per-episode offsets of the obs columns

  const int tid = threadIdx.x;
  const int64_t e0 = (int64_t)blockIdx.x * E;
  const int nvalid = (int)min((int64_t)E, P.num_envs - e0);
  LG_TP(0, 0, tid == 0); LG_TP(0, 12, tid == 128);

  // ---- role of this lane ---------------------------------------------------------------------------
  int role = tid % R::LANES;
  if (role >= R::R_END) role -= (R::LANES - R::R_END);  // spare lanes duplicate a column (same value, same address)
  const bool front = (tid % R::LANES) / 32 * 32 < R::FRONT;  // warp-uniform: this warp holds obs/stage/history roles
  StatScale stat_scale = {0.0, 0, false};
  if (REWARD && (tid >> 5) == kCombineWarp) stat_scale = stat_lane_scale(P, tid & 31);   // statistics lanes (prologue work)
  const int env_first = (tid / R::LANES) * EP;     // first env (within the tile) of this lane's part
  const float* src;             // source of (env_first, column)
  int stride;                   // source row stride in floats
  int dcol;                     // output column (scaled): states[:, dcol], obs[:, dcol] if dcol < OBS; -1: none
  float* stage = nullptr;       // shared destination of env_first's raw value, or null
  int stage_stride = 0;
  int hist_col = -1;            // column of the NEXT history entry this lane provides, or -1
  // this lane's scale_transform constants (torch_utils.py:33-36) in half-span form:
  // 2 (x - c) / span == (x - c) / (span / 2), both scalings exact.  normalize_obs = False: x / 1.
  float centre = 0.0f, half_span = 2.0f, rcp_half = 0.5f;   // span and 1 / span; halved / doubled below (x / 1 when raw)
  {
    const RoleInfo r = role_info<A, ASYM>(P, role);
    const int src_id = r.src_id, src_off = r.src_off, stage_id = r.stage_id, stage_off = r.stage_off;
    stride = r.stride; dcol = r.dcol; stage_stride = r.stage_stride; hist_col = r.hist_col;
    const float* base = src_id == 0 ? S.dof_state : src_id == 1 ? S.root_state : src_id == 2 ? B.goal_pose
                      : src_id == 3 ? B.action : src_id == 4 ? S.rigid_body : src_id == 5 ? S.ft_sensors : S.dof_force;
    src = base + src_off;
    if (stage_id) stage = (stage_id == 1 ? s_obj : stage_id == 2 ? s_goal : s_tips) + stage_off;
  }
  src += (e0 + env_first) * stride;
  const int cnt = max(0, min(EP, nvalid - env_first));   // envs of this lane: env_first .. env_first + cnt - 1
  const bool full = nvalid == E;                                  // every CTA but possibly the last
  // reward warps: thread (w, env) = (tid / 32, tid % 32), w < 4.  Each fetches one 16-byte piece of the
  // env's previous history entry (64-byte rows), the combine warp also the env's flags and step counter.
  const int rw = tid >> 5, renv = tid & 31;
  const bool rlive = REWARD && rw < 4 && renv < nvalid;
  // Everything the first instructions after the dependency wait need is resolved BEFORE it: kernel parameters sit in
  // the constant bank, in a buffer of their own per launch, and the first read of each of their lines (and of the
  // driver's global-memory descriptor the first global load needs) is a constant-cache miss.  The pointers are
  // pinned in registers here, the per-column constants are fetched here (launch constants, never written by a
  // kernel), and the coefficients passed by value are copied here — off the path between the wait and the loads.
  const float4* hist_src = reinterpret_cast<const float4*>(B.history + (e0 + renv) * LG_HISTORY_COLS) + rw;
  const uint8_t* p_goal_reset = B.goal_reset + e0 + renv;
  const uint8_t* p_succ = B.successes + e0 + renv;
  const uint8_t* p_reset = B.reset + e0 + renv;
  const int64_t* p_steps = B.steps_count + e0 + renv;
  asm volatile("" : "+l"(hist_src), "+l"(p_goal_reset), "+l"(p_succ), "+l"(p_reset), "+l"(p_steps), "+l"(src));
  if (P.normalize_obs && dcol >= 0) {   // fetched here, used (and halved / doubled) only after the tile's loads are issued
    centre = __ldg(B.scale_table + dcol);
    half_span = __ldg(B.scale_table + LG_MAX_STATE_DIM + dcol);
    rcp_half = __ldg(B.scale_table + 2 * LG_MAX_STATE_DIM + dcol);
  }
  if (!(REWARD && P.use_device_clock) && tid < C_COUNT) s_coef[tid] = CF.v[tid];
  pdl_wait();  // everything above is independent of the previous kernel's results
  LG_TP(0, 1, tid == 0); LG_TP(0, 13, tid == 128);

  // ---- phase 1: every global load of the tile in flight, what the reward chain needs first -----------
  float4 hprev = make_float4(0.f, 0.f, 0.f, 0.f);
  uint8_t in_goal_reset = 0, in_succ = 0, in_reset = 0;
  int64_t in_steps = 0;
  if (rlive) hprev = ld_hist4(hist_src);
  float v[EP];
  if (full) {
#pragma unroll
    for (int k = 0; k < EP; ++k) v[k] = ld_stream1(src + (int64_t)k * stride);
  } else {
#pragma unroll
    for (int k = 0; k < EP; ++k) v[k] = k < cnt ? ld_stream1(src + (int64_t)k * stride) : 0.0f;
  }
  // extension (per-episode DR offsets): an observation lane whose column carries an offset copies it for its envs into
  // shared memory with the tile's other loads (lanes hold consecutive columns: coalesced along the row), by cp.async so
  // that no register waits for it; the same lane reads it back when it emits the column.  Every other lane issues
  // nothing, and dr_bias_mask == 0 skips it all (dr_activate, in the hot parameter lines, is tested first).
  const bool biased = EXT && P.dr_activate && P.dr_bias_mask != 0 && front && dcol >= 0 && dcol < L::OBS && ((P.dr_bias_mask >> dcol) & 1);
  if (biased) {
    const float* bsrc = B.obs_bias + (e0 + env_first) * L::OBS + dcol;
#pragma unroll
    for (int k = 0; k < EP; ++k)
      if (full || k < cnt) async_copy4(&s_bias[dcol][env_first + k], bsrc + (int64_t)k * L::OBS);
    async_copy_commit();
  }
  // The flags and the step counter are needed last (by the combine): fetched after the tile's loads.  In front of them
  // the compiler turned the flag bytes into predicates at once — a full round trip in which the combine warp had not
  // yet issued its column loads.
  asm volatile("" : "+l"(p_goal_reset), "+l"(p_succ), "+l"(p_reset), "+l"(p_steps));
  if (rlive && rw == kCombineWarp) { in_goal_reset = *p_goal_reset; in_succ = *p_succ; in_reset = *p_reset; in_steps = *p_steps; }
  float in_return = 0.0f;   // extension: the env's running return (episode statistics)
  if (EXT && REWARD && rlive && rw == kCombineWarp && B.episode_return) in_return = B.episode_return[e0 + renv];
  // extension: the env's running per-term row (32 contiguous bytes) lands in shared memory by itself — no register
  // waits for it, and the combine warp picks it up after its reward math
  if (EXT && REWARD && rlive && rw == kCombineWarp && B.episode_term_return) {
    const float4* row = reinterpret_cast<const float4*>(B.episode_term_return + (e0 + renv) * LG_NUM_EPISODE_TERMS);
    async_copy16(&s_term_run[2 * renv], row);
    async_copy16(&s_term_run[2 * renv + 1], row + 1);
    async_copy_commit();
  }
  pdl_launch_dependents();  // the next kernel may start launching; it still waits for this grid to finish
  // same for the scale constants: a CTA that starts late must not wait for them before it has issued its loads
  asm volatile("" : "+f"(half_span), "+f"(rcp_half));
  half_span = 0.5f * half_span;
  rcp_half = 2.0f * rcp_half;
  LG_TP(0, 2, tid == 0);

  // ---- reward coefficients: from the launch arguments, or (device clock) from what lg_pre_physics wrote ----
  if (REWARD && P.use_device_clock && tid < C_COUNT) s_coef[tid] = __ldg(B.reward_coef + tid);

  // ---- phase 2: stage what the reward terms read, then ONE barrier -------------------------------
  // Only the warps that hold staged columns wait for (a small part of) their data here; the others
  // reach the barrier right after issuing their loads.  The reward math then runs on warps 0-3 while
  // the bulk of the tile is still arriving and being scaled and stored by warps 4-7.
  if (rlive) {
    float* h = s_hist + renv * HS + rw * 4;
    h[0] = hprev.x; h[1] = hprev.y; h[2] = hprev.z; h[3] = hprev.w;
  }
  // extension (DR observation noise): the tile's standard normals, generated by ALL threads while the loads are in
  // flight — one Philox block + two Box-Muller pairs per (column, group of 4 envs by GLOBAL index), so the stream
  // does not depend on tiling or sharding.  Columns with sigma = 0 are skipped.
  if (EXT && P.dr_activate) {
    const uint64_t base = (uint64_t)(P.env_offset + e0);
    const uint64_t g0 = base >> 2;
    const int ngroups = (int)(((base + E - 1) >> 2) - g0) + 1;
    const uint32_t noise_epoch = __float_as_uint((REWARD && P.use_device_clock) ? __ldg(B.reward_coef + C_NOISE_EPOCH)
                                                                                  : CF.v[C_NOISE_EPOCH]);
    for (int i = tid; i < L::OBS * ngroups; i += kPostThreads) {
      const int col = i / ngroups, g = i - col * ngroups;
      if (__ldg(B.scale_table + 3 * LG_MAX_STATE_DIM + col) != 0.0f) {
        const uint64_t grp = g0 + g;
        const U4 r = philox4x32_10(U4{(uint32_t)grp, (uint32_t)(grp >> 32) ^ kPurposeNoise, (uint32_t)col, noise_epoch},
                                   (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
        float n[4];
        box_muller(r.x, r.y, n[0], n[1]);
        box_muller(r.z, r.w, n[2], n[3]);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int64_t local = (int64_t)(4 * grp + q) - (int64_t)base;
          if (local >= 0 && local < E) s_noise[col][local] = n[q];
        }
      }
    }
  }
  if (front && stage) {
    float* dst = stage + env_first * stage_stride;
    if (full) {
#pragma unroll
      for (int k = 0; k < EP; ++k) dst[k * stage_stride] = v[k];
    } else {
#pragma unroll
      for (int k = 0; k < EP; ++k)
        if (k < cnt) dst[k * stage_stride] = v[k];
    }
  }
  LG_TP(0, 3, tid == 0);
  // Staging barrier: the reward warps wait for the front warps' staged columns (and the front warps, which write
  // the next history entry below, for the reward warps' reads of the previous one).  The other warps hold nothing
  // anyone waits for: they go straight on to scale and store their columns as their data arrives.
  if (EXT || !REWARD) __syncthreads();   // extension: the noise tile is read by every observation lane
  else if (R::STAGE_WARPS * 32 == kPostThreads) __syncthreads();
  else if (rw < 4 || front) asm volatile("bar.sync 3, %0;" :: "n"(R::STAGE_WARPS * 32) : "memory");
  LG_TP(0, 4, tid == 0); LG_TP(0, 14, tid == 128);

  // ---- phase 3 (all warps; the reward warps come back to it after their math): scale and store the columns -----
  auto emit_outputs = [&](auto full_c) {
    constexpr bool FULLC = decltype(full_c)::value;  // full tile: no per-element bound checks at all
    // history shift (deque.appendleft, trifinger_env.py:974-975): current -> entry read next step.
    // After the staging barrier: every read of the previous entry has completed.
    if (front && hist_col >= 0) {
      float* dst = B.history + (e0 + env_first) * LG_HISTORY_COLS + hist_col;
#pragma unroll
      for (int k = 0; k < EP; ++k)
        if (FULLC || k < cnt) dst[k * LG_HISTORY_COLS] = v[k];
    }
    float amax = 0.0f;  // largest numerator seen: beyond 2^100 (never, for physical data) the column is redone exactly
    const float clip = P.clip_obs;
    const int st_off = env_first * L::STATE + dcol, ob_off = env_first * L::OBS + dcol;
    float* st = ASYM ? B.states + e0 * L::STATE + st_off : nullptr;                          // trifinger_env.py:990-994
    float* stc = (CLIP && ASYM) ? B.states_clipped + e0 * L::STATE + st_off : nullptr;       // vec_task.py:147
    const bool to_obs = front && dcol >= 0 && dcol < L::OBS;
    float* ob = B.obs + e0 * L::OBS + ob_off;                                                // trifinger_env.py:983-987
    float* obc = CLIP ? B.obs_clipped + e0 * L::OBS + ob_off : nullptr;                      // vec_task.py:167
    // extension (no reference code; the TODO at trifinger_env.py:979): additive Gaussian noise on the RAW
    // actor observation, before scale_transform; the critic's states stay clean.  sigma = 0 -> skipped.  The env's
    // per-episode offset (loaded above) comes first: (raw + offset) + sigma n.
    const float sigma = (EXT && P.dr_activate && to_obs) ? __ldg(B.scale_table + 3 * LG_MAX_STATE_DIM + dcol) : 0.0f;
    const bool noisy = EXT && __any_sync(0xffffffffu, sigma != 0.0f);
    const bool perturbed = noisy || biased;
    if (EXT && biased) async_copy_wait_all();   // this lane's own offsets have landed
    // optional bf16 copies for the policy / value networks (SURVEY.md 8 f2): of the clipped values when the
    // wrapper's clamp is fused in, else of the scaled values
    uint16_t* stb = (EXT && ASYM && B.states_bf16) ? B.states_bf16 + e0 * L::STATE + st_off : nullptr;
    uint16_t* obb = (EXT && B.obs_bf16) ? B.obs_bf16 + e0 * L::OBS + ob_off : nullptr;
    // outputs go out with streaming stores (st.global.cs): nothing on the device reads them again before the
    // learner does, and evict-first keeps them from displacing the simulator rows in L2 (measured: 84.0 -> 80.3 us
    // at 262 144 envs, 7.25 -> 7.15 us at 16 384).  Assembling the tile in shared memory and sending it as bulk
    // stores was measured too: 7.95-8.18 us (profiles/experiments/r02_post_bulk_store_variant.cuh.txt).
    if (dcol >= 0) {
      auto emit_one = [&](int k, float sv, float ov) {
        if (ASYM) {
          __stcs(st + k * L::STATE, sv);
          const float svc = CLIP ? clamp_nan(sv, -clip, clip) : sv;
          if (CLIP) __stcs(stc + k * L::STATE, svc);
          if (EXT && stb) __stcs(stb + k * L::STATE, to_bf16(svc));
        }
        if (to_obs) {
          __stcs(ob + k * L::OBS, ov);
          const float ovc = CLIP ? clamp_nan(ov, -clip, clip) : ov;
          if (CLIP) __stcs(obc + k * L::OBS, ovc);
          if (EXT && obb) __stcs(obb + k * L::OBS, to_bf16(ovc));
        }
      };
#pragma unroll
      for (int k = 0; k < EP; ++k) {
        const float sv = div_by_const(v[k] - centre, half_span, rcp_half, amax);
        float ov = sv;
        // sigma = 0 columns (and non-observation lanes) skip it: their noise row is never generated, and 0 * a stale
        // inf / NaN left in shared memory by an earlier CTA would be NaN.  Columns without an offset skip the add:
        // raw + 0.0f would turn -0 into +0.
        if (perturbed && (biased || sigma != 0.0f)) {
          float x = v[k];
          if (biased) x = x + s_bias[dcol][env_first + k];
          if (noisy && sigma != 0.0f) x = x + sigma * s_noise[dcol][env_first + k];   // generated before the barrier
          ov = div_by_const(x - centre, half_span, rcp_half, amax);
        }
        if (FULLC || k < cnt) emit_one(k, sv, ov);
      }
      if (!(amax < kDivSafeMax)) {  // cold: a numerator left the fast division's window: IEEE division
        const float c0 = P.scale_centre[dcol], span = P.scale_span[dcol];
#pragma unroll
        for (int k = 0; k < EP; ++k) {   // unrolled: v[] must stay in registers
          if (FULLC || k < cnt) {
            const float x = P.normalize_obs ? __fdiv_rn(2.0f * (v[k] - c0), span) : v[k];
            float xo = x;
            if (perturbed && (biased || sigma != 0.0f)) {   // the lane's finite envs keep their noise: bit-identical to the fast path
              float vn = v[k];
              if (biased) vn = vn + s_bias[dcol][env_first + k];
              if (noisy && sigma != 0.0f) vn = vn + sigma * s_noise[dcol][env_first + k];
              xo = P.normalize_obs ? __fdiv_rn(2.0f * (vn - c0), span) : vn;
            }
            emit_one(k, x, xo);
          }
        }
      }
    }
    // moving goal (__update_goal_movement_post, trifinger_env.py:1279-1284): after the rewards, the goal pose
    // buffer takes the pose the simulator integrated for the goal body.  The goal-role lanes own their elements
    // of goal_pose (read above, overwritten here), so no other lane observes the change within this step.
    if (EXT && REWARD && P.goal_rotation && front && role >= 25 && role < 32) {
      const int c = role - 25, actor_stride = P.actors_per_env * 13;
      const float* g_src = S.root_state + ((e0 + env_first) * P.actors_per_env + P.goal_slot) * 13 + c;
      float* g_dst = B.goal_pose + (e0 + env_first) * 7 + c;
#pragma unroll
      for (int k = 0; k < EP; ++k)
        if (FULLC || k < cnt) g_dst[k * 7] = g_src[(int64_t)k * actor_stride];
    }
  };
  // Order of the tail, per warp: the three reward warps with the longer sub-tasks only ARRIVE at the reward barrier
  // and go on to their columns; the warp with the shortest sub-task (kCombineWarp) stores its columns first — by
  // then the others have arrived — and then combines, terminates and accumulates the statistics.  No warp waits,
  // and the CTA's longest chain is sub-task -> combine -> statistics instead of that plus a column pass.
  if (REWARD && rw < 4) {
    reward_subtasks<E, EXT>(P, nvalid, s_obj, s_goal, s_tips, s_hist, s_coef, &s_part[0][0]);
    if (rw != kCombineWarp) asm volatile("bar.arrive 1, 128;" ::: "memory");
  }
  if (full) emit_outputs(std::true_type{});
  else emit_outputs(std::false_type{});
  LG_TP(0, 9, tid == 0);
  if (REWARD && rw == kCombineWarp)
    reward_combine<E, EXT>(P, B, e0, nvalid, s_coef, &s_part[0][0], in_goal_reset, in_succ, in_reset, in_steps, in_return,
                           &s_term_run[EXT ? 2 * renv : 0], stat_scale);
  LG_TP(0, 15, tid == 128); LG_TP(0, 19, tid == 32); LG_TP(0, 20, tid == 64); LG_TP(0, 21, tid == 96);
}

// history seeding (trifinger_env.py:619-628): both entries = initial simulator state
__global__ void init_history_kernel(const __grid_constant__ LgParams P, const LgSimState S, const LgBuffers B) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.num_envs * LG_HISTORY_COLS) return;
  const int64_t e = i >> 4;
  const int c = (int)(i & 15);
  float v;
  if (c < 9) v = S.rigid_body[(e * P.bodies_per_env + P.fingertip_body[c / 3]) * 13 + (c % 3)];
  else v = S.root_state[((int64_t)P.actors_per_env * e + P.object_slot) * 13 + (c - 9)];
  B.history[i] = v;
}

}  // namespace lg
