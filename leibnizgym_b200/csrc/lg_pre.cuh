// pre-physics pass of the TriFinger MDP hot path (sm_100a): ordered mask compaction (decoupled look-back, or a direct
// count of the flag bytes for one-wave grids) fused with reset / goal-reset sampling and scatter, action store and
// action -> torque; tile slabs by TMA bulk copy.
// Also the stand-alone compaction and the hook kernels on explicit id lists.
// Included by lg_kernels.cu (single translation unit).  Reference paths are relative to /root/reference/leibnizgym/.
#pragma once

#include "lg_device.cuh"
#include "lg_post.cuh"   // pdl_wait / pdl_launch_dependents, compute_coefs

namespace lg {

// =========================================================================================
// pre-physics: ordered compaction by decoupled look-back, fused with the resets
// =========================================================================================
constexpr int kScanThreads = 128;  // threads of one scan group = envs per tile = predecessors inspected per round trip
constexpr int kPreTile = kScanThreads;   // envs per CTA of the pre-physics kernel
constexpr int kPreThreads = 256;   // warps 0-3: one env row per thread (action, torque); warps 4-7: the compaction scan

// status word: [63:48] epoch | [47:46] state | [45:23] count A | [22:0] count B
constexpr uint64_t kStateAggregate = 1, kStateInclusive = 2;
__device__ __forceinline__ uint64_t pack_status(uint32_t epoch, uint64_t state, uint32_t a, uint32_t b) {
  return ((uint64_t)(epoch & 0xffffu) << 48) | (state << 46) | ((uint64_t)(a & 0x7fffffu) << 23) | (uint64_t)(b & 0x7fffffu);
}
__device__ __forceinline__ bool status_valid(uint64_t w, uint32_t epoch) {
  return (uint32_t)(w >> 48) == (epoch & 0xffffu) && ((w >> 46) & 3u) != 0;
}

// barrier over one 128-thread group of a CTA (named barrier BAR; BAR = 0 in a 128-thread CTA is __syncthreads)
template <int BAR>
__device__ __forceinline__ void group_sync() { asm volatile("bar.sync %0, %1;" :: "n"(BAR), "n"(kScanThreads) : "memory"); }

// Exclusive prefix of (a, b) over all tiles before `tile`.  Group-wide: thread i of the 128-thread group inspects
// predecessor tile-1-i (128 predecessors per round trip to L2), each warp reduces up to its nearest tile that
// already holds an inclusive prefix, thread 0 chains the warps.  Called by every thread of the group (`gt` = its
// index in the group); returns the prefix to all of them.
template <int BAR>
__device__ __forceinline__ void lookback(uint64_t* status, int tile, uint32_t epoch, uint32_t my_a, uint32_t my_b, int gt,
                                         uint32_t& ex_a, uint32_t& ex_b) {
  __shared__ uint32_t s_sum[kScanThreads / 32][2];
  __shared__ int s_found[kScanThreads / 32];
  __shared__ uint32_t s_res[3];
  const int lane = gt & 31, warp = gt >> 5;
  uint32_t acc_a = 0, acc_b = 0;
  int pos = tile - 1;
  bool done = tile == 0;
  while (!done) {
    const int idx = pos - gt;
    uint64_t w = 0;
    if (idx >= 0) {
      do { w = ld_volatile_u64(status + idx); } while (!status_valid(w, epoch));
    }
    const bool incl = idx >= 0 && ((w >> 46) & 3u) == kStateInclusive;
    const unsigned incl_mask = __ballot_sync(0xffffffffu, incl);
    const int stop = incl_mask ? __ffs(incl_mask) - 1 : 31;  // nearest predecessor holding an inclusive prefix
    uint32_t a = (idx >= 0 && lane <= stop) ? (uint32_t)((w >> 23) & 0x7fffffu) : 0u;
    uint32_t b = (idx >= 0 && lane <= stop) ? (uint32_t)(w & 0x7fffffu) : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
    if (lane == 0) { s_sum[warp][0] = a; s_sum[warp][1] = b; s_found[warp] = incl_mask != 0; }
    group_sync<BAR>();
    if (gt == 0) {
      bool found = false;
      for (int k = 0; k < kScanThreads / 32 && !found; ++k) { acc_a += s_sum[k][0]; acc_b += s_sum[k][1]; found = s_found[k] != 0; }
      s_res[0] = acc_a; s_res[1] = acc_b; s_res[2] = found || pos - kScanThreads < 0;
    }
    group_sync<BAR>();
    done = s_res[2] != 0;
    acc_a = s_res[0]; acc_b = s_res[1];
    pos -= kScanThreads;
    group_sync<BAR>();   // s_res is rewritten in the next round
  }
  if (gt == 0 && tile > 0)
    atomicExch(reinterpret_cast<unsigned long long*>(status + tile),
               (unsigned long long)pack_status(epoch, kStateInclusive, acc_a + my_a, acc_b + my_b));
  ex_a = acc_a; ex_b = acc_b;
}

struct TileScan {
  int tile;
  uint32_t epoch;
  uint32_t rank_a, rank_b;   // this thread's rank inside the tile (valid where its flag is set)
  uint32_t total_a, total_b; // tile totals
};

// Resolves the global exclusive prefix (returned to every thread of the group); the last tile re-arms ticket and
// epoch for the next launch.
template <bool TICKET, int BAR>
__device__ __forceinline__ void tile_scan_finish(LgControl* ctl, uint64_t* status, const TileScan& t, int num_tiles, int gt,
                                                 uint32_t& ex_a, uint32_t& ex_b, int32_t* counts_out) {
  lookback<BAR>(status, t.tile, t.epoch, t.total_a, t.total_b, gt, ex_a, ex_b);
  if (gt == 0 && t.tile == num_tiles - 1) {
    // every tile has read the epoch and taken its ticket by now (their aggregates are visible)
    if (counts_out) { counts_out[0] = (int32_t)(ex_a + t.total_a); counts_out[1] = (int32_t)(ex_b + t.total_b); }
    if (TICKET) { ctl->scan_ticket = 0; __threadfence(); }
    ctl->scan_epoch = t.epoch + 1;
  }
}

// Block scan of two flag masks over one 128-thread group: ranks inside the tile and tile totals.
template <int BAR>
__device__ __forceinline__ void tile_scan_local(bool fa, bool fb, int gt, uint32_t* s_wa, uint32_t* s_wb, TileScan& t) {
  const int lane = gt & 31, warp = gt >> 5;
  const unsigned ba = __ballot_sync(0xffffffffu, fa), bb = __ballot_sync(0xffffffffu, fb);
  if (lane == 0) { s_wa[warp] = __popc(ba); s_wb[warp] = __popc(bb); }
  group_sync<BAR>();
  uint32_t pa = 0, pb = 0, ta = 0, tb = 0;
#pragma unroll
  for (int w = 0; w < kScanThreads / 32; ++w) {
    if (w < warp) { pa += s_wa[w]; pb += s_wb[w]; }
    ta += s_wa[w]; tb += s_wb[w];
  }
  const unsigned below = (1u << lane) - 1u;
  t.rank_a = pa + __popc(ba & below);
  t.rank_b = pb + __popc(bb & below);
  t.total_a = ta; t.total_b = tb;
}

// ---- direct prefix (grids of at most kDirectMaxTiles tiles) ------------------------------------------------------
// Instead of waiting for its predecessors' aggregates, a CTA counts the flagged envs in front of its tile ITSELF: the
// flag bytes of all predecessors (at most 127 x 128 bytes per mask, hot in L2) are fetched as 128-bit words by all 256
// threads right at entry — addresses known at launch, one round trip — and counted next to the tile's own block scan.
// No CTA ever waits for another one's progress, so a late tile cannot hold up the rest of the grid (look-back done:
// median 2.0, max 3.0 us after entry).
constexpr int kDirectMaxTiles = 128;
constexpr int kDirectVecs = (kDirectMaxTiles - 1) * kPreTile / 16 / kPreThreads + 1;   // 128-bit words per thread and mask: 4

__device__ __forceinline__ uint32_t nonzero_bytes(uint32_t x) {   // how many of the four bytes are != 0
  return (uint32_t)__popc((((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u);
}
// count | count << 16 of the flagged envs among the first `nvec` x 16 envs, the share of thread `tid` of the CTA.
// The forced masks (`_reset_buf |= mask`) are optional.  Flag bytes are 0 or 1 wherever they come from a bool tensor:
// one dot-product instruction per word sums them; any other non-zero value (seen in the OR of all words) sends the
// thread through the exact count.
__device__ __forceinline__ uint32_t count_flagged_before(const uint8_t* __restrict__ reset, const uint8_t* __restrict__ goal,
                                                         const uint8_t* __restrict__ force_reset,
                                                         const uint8_t* __restrict__ force_goal, int nvec, int tid) {
  const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
  uint4 vr[kDirectVecs], vg[kDirectVecs];
#pragma unroll
  for (int k = 0; k < kDirectVecs; ++k) {
    const int i = tid + k * kPreThreads;
    vr[k] = i < nvec ? __ldcg(reinterpret_cast<const uint4*>(reset) + i) : zero;
    vg[k] = i < nvec ? __ldcg(reinterpret_cast<const uint4*>(goal) + i) : zero;
  }
  if (force_reset) {
#pragma unroll
    for (int k = 0; k < kDirectVecs; ++k) {
      const int i = tid + k * kPreThreads;
      if (i < nvec) {
        const uint4 f = __ldcg(reinterpret_cast<const uint4*>(force_reset) + i);
        vr[k].x |= f.x; vr[k].y |= f.y; vr[k].z |= f.z; vr[k].w |= f.w;
      }
    }
  }
  if (force_goal) {
#pragma unroll
    for (int k = 0; k < kDirectVecs; ++k) {
      const int i = tid + k * kPreThreads;
      if (i < nvec) {
        const uint4 f = __ldcg(reinterpret_cast<const uint4*>(force_goal) + i);
        vg[k].x |= f.x; vg[k].y |= f.y; vg[k].z |= f.z; vg[k].w |= f.w;
      }
    }
  }
  uint32_t a = 0, b = 0, any = 0;
#pragma unroll
  for (int k = 0; k < kDirectVecs; ++k) {
    const uint4 x = vr[k], y = vg[k];
    a = __dp4a(x.x, 0x01010101u, a); a = __dp4a(x.y, 0x01010101u, a); a = __dp4a(x.z, 0x01010101u, a); a = __dp4a(x.w, 0x01010101u, a);
    b = __dp4a(y.x, 0x01010101u, b); b = __dp4a(y.y, 0x01010101u, b); b = __dp4a(y.z, 0x01010101u, b); b = __dp4a(y.w, 0x01010101u, b);
    any |= (x.x | x.y) | (x.z | x.w) | (y.x | y.y) | (y.z | y.w);
  }
  if (any & 0xfefefefeu) {   // cold: a flag byte other than 0 / 1
    a = 0; b = 0;
#pragma unroll
    for (int k = 0; k < kDirectVecs; ++k) {
      a += nonzero_bytes(vr[k].x) + nonzero_bytes(vr[k].y) + nonzero_bytes(vr[k].z) + nonzero_bytes(vr[k].w);
      b += nonzero_bytes(vg[k].x) + nonzero_bytes(vg[k].y) + nonzero_bytes(vg[k].z) + nonzero_bytes(vg[k].w);
    }
  }
  return a | (b << 16);
}

// extension (no reference code): additive Gaussian noise on one env's action row — one Philox block -> four normals ->
// four action columns.  Out of line: off by default, and the hot path should not carry its code.
template <int A>
__device__ __noinline__ void action_noise(const LgParams& P, uint64_t genv, uint32_t epoch, float* act) {
#pragma unroll
  for (int c4 = 0; c4 < A; c4 += 4) {
    const U4 r = philox4x32_10(U4{(uint32_t)genv, (uint32_t)(genv >> 32) ^ kPurposeNoise, 0x41435400u + c4, epoch},
                               (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
    float n[4];
    box_muller(r.x, r.y, n[0], n[1]);
    box_muller(r.z, r.w, n[2], n[3]);
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (c4 + q < A) act[c4 + q] = act[c4 + q] + P.dr_action_sigma * n[q];
  }
}

// extension (no reference code): domain randomisation of one env's action row — its per-episode offset (`bias`, the
// row its last reset drew; null when off), then the Gaussian noise (`noise`).  One call site in the kernel, out of line.
template <int A>
__device__ __noinline__ void perturb_action(const LgParams& P, const float* __restrict__ bias, bool noise, uint64_t genv,
                                            uint32_t epoch, float* act) {
  if (bias) {
#pragma unroll
    for (int c = 0; c < A; ++c) act[c] = act[c] + bias[c];
  }
  if (noise) action_noise<A>(P, genv, epoch, act);
}

// What the first instructions of the kernel need, as the FIRST kernel parameter: kernel parameters sit in the constant
// bank in a buffer of their own per launch, so every 64-byte line of them costs a constant-cache miss on first use;
// the slab copies can be issued after one miss instead of four (pointers otherwise spread over LgSimState, LgBuffers,
// LgParams and the trailing arguments).
struct PreHot {
  const float* action_in;
  const float* dof_state;
  float* applied_torque;
  int64_t num_envs;
  int32_t num_tiles;
  int32_t _pad;
};

// One CTA = one tile of 128 envs, two 128-thread groups working on two independent chains:
//   row group  (warps 0-3, thread = env): the tile's action and joint-state rows arrive as TMA bulk copies; the action
//              row is clamped (+ offset and noise, extension), zeroed for resetting envs and kept for the torque;
//   scan group (warps 4-7, thread = env): flag bytes -> ballot/popcount block scan of both masks -> aggregate
//              published -> block-wide decoupled look-back -> ascending id lists (torch.nonzero order) and the
//              simulator's actor-index lists.
// They meet for the resets (block-uniform branch: ten reset sub-tasks as work items over the eight warps, lane =
// listed env); the row group then computes the torque from the shared-memory slabs while the scan group resolves its
// look-back; action and torque rows leave as bulk stores.
// MINB = CTAs per SM the register allocation must allow: 3 (<= 85 registers) for grids of one wave, where
// the kernel is a latency chain (30 % resets at 16 384 envs: 17.3 against 18.0 us/step), 4 (64 registers) for larger
// grids, where more rows in flight per SM is what counts (65 536 envs with goal resampling: 37.7 against 42.3 us/step).
//
// DIRECT (grids of 32 .. kDirectMaxTiles tiles, one CTA per SM): no look-back — every tile counts the flagged envs in
// front of it itself (count_flagged_before above), so no tile waits for another one's progress; the only grid-wide
// hand-shake left protects the clearing of flag bytes by tiles with resets (scan_readers / scan_exits, below).
//
// TORCH (P.rng_stream == LG_RNG_TORCH): the resets draw torch's CUDA Philox stream (TorchDraws), which needs each
// resetting env's global rank (the lists are resolved first, as for injected draws) and the list lengths and base offset
// of this launch, which the counting launch in front (torch_count_kernel) left in B.torch_rng.
//
// SPLIT = false is the same pass with ONE 128-thread group doing both chains one after the other (look-back last, when
// every predecessor has long published): grids of many waves are bound by the rows in flight per SM, not by the length
// of a CTA's chain, and half-idle CTAs of 256 threads cost them a third of their throughput (1 048 576 envs: 84 against
// 54 us).  Used together with the ticket path.
template <int A, bool TICKET, int MINB, bool SPLIT, bool DIRECT = false, bool TORCH = false>
__global__ void __launch_bounds__(SPLIT ? kPreThreads : kScanThreads, MINB)
pre_physics_kernel(const __grid_constant__ PreHot H, const __grid_constant__ LgParams P,
                   const __grid_constant__ LgSimState S, const __grid_constant__ LgBuffers B) {
  const float* __restrict__ action_in = H.action_in;
  const int num_tiles = H.num_tiles;
  constexpr int E = kPreTile;
  __shared__ __align__(128) float s_act[E * A];
  __shared__ __align__(128) float s_dof[E * 18];
  __shared__ __align__(128) float s_tq[E * 9];
  __shared__ __align__(8) uint64_t s_mbar;
  __shared__ int s_tile;
  __shared__ uint32_t s_wa[kScanThreads / 32], s_wb[kScanThreads / 32];
  __shared__ uint8_t s_flag[E];            // bit 0 reset, bit 1 goal reset
  __shared__ uint32_t s_scan[4];           // tile totals (a, b) and the global exclusive prefix (a, b)
  __shared__ uint16_t s_reset_list[E], s_goal_list[E];
  __shared__ uint32_t s_before[kPreThreads / 32];   // DIRECT: flagged envs in front of the tile, per warp

  static_assert(!DIRECT || (SPLIT && !TICKET), "the direct prefix is a variant of the two-group, co-resident kernel");
  const int tid = threadIdx.x;
  constexpr int NT = SPLIT ? kPreThreads : kScanThreads;   // threads of the CTA
  const int gt = tid & (kScanThreads - 1);
  const bool row_group = !SPLIT || tid < kScanThreads;
  const bool scan_group = !SPLIT || tid >= kScanThreads;
  LG_TP(1, 0, tid == 0);
  // May be launched programmatically after lg_post_physics (see pdl_mode): nothing the preceding kernel writes is read
  // before pdl_wait() below — only the action and joint-state slabs, which the caller / simulator completed before that
  // kernel was allowed past its own dependency wait.  The control block (epoch, ticket) is read after the wait: it is
  // written by this kernel's own previous launch, which is not yet complete when two of these passes follow each other
  // directly.
  int tile = blockIdx.x;
  uint32_t epoch = 0;
  if (TICKET) {  // grids larger than what is co-resident: tiles by ticket, so predecessors always run
    pdl_wait();
    epoch = ld_volatile_u32(&B.control->scan_epoch);   // every thread, before the tile publishes anything (the last tile advances it)
    if (tid == 0) s_tile = (int)atomicAdd(&B.control->scan_ticket, 1u);
    __syncthreads();
    tile = s_tile;
  }
  const int64_t e0 = (int64_t)tile * E;
  const int64_t e = e0 + gt;               // this thread's env (both groups)
  const int nvalid = (int)min((int64_t)E, H.num_envs - e0);
  const bool live = gt < nvalid;
  const bool want_torque = H.applied_torque != nullptr;
  const bool full_tile = nvalid == E;   // bulk copies need 16-byte multiples: ragged last tile goes lane by lane

  // ---- row group: every global load of the tile's rows up front ------------------------------------------
  if (row_group) {
    if (full_tile) {
      if (tid == 0) {
        mbar_init(&s_mbar, 1);
        mbar_expect_tx(&s_mbar, (uint32_t)(sizeof(float) * E * (A + (want_torque ? 18 : 0))));
        bulk_load(s_act, action_in + e0 * A, sizeof(float) * E * A, &s_mbar);
        if (want_torque) bulk_load(s_dof, H.dof_state + e0 * 18, sizeof(float) * E * 18, &s_mbar);
      }
    } else if (live) {
#pragma unroll
      for (int c = 0; c < A; ++c) s_act[gt * A + c] = action_in[e * A + c];
      if (want_torque) {
#pragma unroll
        for (int c = 0; c < 18; ++c) s_dof[gt * 18 + c] = S.dof_state[e * 18 + c];
      }
    }
  }
  LG_TP(1, 1, tid == 0);
  if (!TICKET) {
    pdl_wait();   // the flags, counters and statistics below are results of the preceding post-physics pass
    epoch = ld_volatile_u32(&B.control->scan_epoch);   // every thread, before the tile publishes anything (the last tile advances it)
  }
  LG_TP(1, 2, tid == 0);
  // scan group: this env's own flag bytes, fetched FIRST — in the same round trip as (DIRECT) the predecessors' bytes,
  // not after they have been counted
  uint8_t flag_r = 0, flag_g = 0, flag_fr = 0, flag_fg = 0;
  if (scan_group && live) {
    flag_r = B.reset[e]; flag_g = B.goal_reset[e];
    if (B.force_reset) flag_fr = B.force_reset[e];             // `_reset_buf |= mask` folded into the pass
    if (B.force_goal_reset) flag_fg = B.force_goal_reset[e];
  }
  uint32_t before = 0;   // DIRECT: this thread's share of the flagged envs in front of the tile (a | b << 16)
  if (DIRECT) before = count_flagged_before(B.reset, B.goal_reset, B.force_reset, B.force_goal_reset, tile * (E / 16), tid);

  // ---- scan group: block scan of both masks + aggregate publication (env_base.py:374-379) ------------------
  // Needs only the two flag bytes, so the tile's aggregate is visible to its successors while the action /
  // joint-state slabs are still in flight.
  TileScan t;
  t.tile = tile; t.epoch = epoch;
  bool f_reset = false, f_goal = false;
  if (scan_group) {
    f_reset = (flag_r | flag_fr) != 0; f_goal = (flag_g | flag_fg) != 0;
    tile_scan_local<1>(f_reset, f_goal, gt, s_wa, s_wb, t);
    s_flag[gt] = (uint8_t)((f_reset ? 1 : 0) | (f_goal ? 2 : 0));
    if (f_reset) s_reset_list[t.rank_a] = (uint16_t)(gt | (f_goal ? 0x8000 : 0));   // flagged envs by rank in the tile
    if (f_goal) s_goal_list[t.rank_b] = (uint16_t)gt;
    if (gt == 0) {
      if (!DIRECT) {
        const uint64_t st = tile == 0 ? kStateInclusive : kStateAggregate;
        atomicExch(reinterpret_cast<unsigned long long*>(B.scan_status + tile),
                   (unsigned long long)pack_status(epoch, st, t.total_a, t.total_b));
      }
      s_scan[0] = t.total_a; s_scan[1] = t.total_b;
    }
    LG_TP(1, 3, tid == NT - kScanThreads);
    // Tile 0's housekeeping comes AFTER its aggregate is published: every other tile's look-back ends at tile 0's
    // inclusive prefix, and the coefficient arithmetic below is a chain of fp64 operations.
    if (tile == 0 && gt < LG_NUM_STATS && B.step_stats) B.step_stats[gt] = 0.0;  // accumulated by lg_post_physics
    if (tile == 0 && gt < LG_NUM_EPISODE_STATS && B.episode_stats) B.episode_stats[gt] = 0.0;  // likewise (extension)
    if (tile == 0 && gt < LG_NUM_EPISODE_TERMS && B.episode_term_stats) B.episode_term_stats[gt] = 0.0;
    if (tile == 0 && gt == kScanThreads - 1 && P.use_device_clock) {
      // device clock: advance the frame counter and publish the reward coefficients of the coming
      // post-physics pass (env_steps_count = frames x global env count, envs/env_base.py:286-289)
      const int64_t frame = B.control->frame_count + P.control_decimation;
      B.control->frame_count = frame;
      if (B.reward_coef) compute_coefs(P, (double)(frame * P.global_num_envs), B.reward_coef);
    }
  }
  if (DIRECT) {
    before = __reduce_add_sync(0xffffffffu, before);
    if ((tid & 31) == 0) s_before[tid >> 5] = before;
  }
  __syncthreads();   // flags, tile totals and reset lists are visible to everyone; the mbarrier is initialised
  const int na = (int)s_scan[0], nb = (int)s_scan[1];
  const bool resets = (na | nb) != 0;                         // block-uniform
  // A tile without resets lets the post-physics pass start launching right here: its CTAs (two or three fit next to
  // this one) run their ~0.8 us of set-up while this tile finishes, instead of after it (16 384 envs: 10.26 -> 10.08
  // us/step).  A tile with resets triggers after its torque phase (below): parked CTAs next to a long reset phase
  // were measured slower (15.4 against 15.1 us/step at 30 % resets), triggering at entry likewise for larger grids.
  if (!resets) pdl_launch_dependents();
  const bool rank_first = resets && (TORCH || P.inject_draws != 0);   // injected / torch draws are indexed by rank
  // DIRECT: grid-wide hand-shake about the flag bytes, kept off the row group's chain (one thread of the scan group,
  // which has slack).  `scan_readers` counts the tiles whose reads of their predecessors' flag bytes have completed (the
  // values went into the counts); a tile that is going to CLEAR flag bytes (resets) first waits for all of them.
  // `scan_exits` counts the tiles that no longer look at `scan_readers`; the last one re-arms both and advances the
  // epoch (the RNG epoch of the fused resets), which every thread of the grid has read at entry by then.
  auto tile_passed = [&]() {
    if (atomicAdd(&B.control->scan_exits, 1u) == (uint32_t)num_tiles - 1u) {
      B.control->scan_readers = 0; B.control->scan_exits = 0;
      B.control->scan_epoch = epoch + 1;
    }
  };
  const bool handshake = DIRECT && tid == NT - 2;   // a thread of the scan group without other duties
  uint32_t direct_a = 0, direct_b = 0;   // DIRECT: the global exclusive prefix, known to every thread from here on
  if (DIRECT) {
    uint32_t sum = 0;
#pragma unroll
    for (int w = 0; w < kPreThreads / 32; ++w) sum += s_before[w];
    direct_a = sum & 0xffffu; direct_b = sum >> 16;
    if (handshake) {
      __threadfence();
      atomicAdd(&B.control->scan_readers, 1u);
      if (!resets) tile_passed();
    }
  }

  // ---- scan group: global exclusive prefix, then the ordered id lists (env_base.py:374-379;
  // trifinger_env.py:413-416, :435-436).  Runs next to the row group's work; a tile with resets does it after them
  // (every warp helps with the resets) unless the injected test draws need the rank first.
  auto finish_scan = [&]() {
    uint32_t ex_a = direct_a, ex_b = direct_b;
    if (DIRECT) {
      if (gt == 0 && tile == num_tiles - 1 && B.counts) {
        B.counts[0] = (int32_t)(ex_a + t.total_a); B.counts[1] = (int32_t)(ex_b + t.total_b);
      }
    } else {
      tile_scan_finish<TICKET, 1>(B.control, B.scan_status, t, num_tiles, gt, ex_a, ex_b, B.counts);
    }
    if (gt == 0) { s_scan[2] = ex_a; s_scan[3] = ex_b; }
    if (f_reset) {
      const int64_t j = (int64_t)ex_a + t.rank_a;
      const int32_t base = (int32_t)(P.actors_per_env * e);
      B.reset_ids[j] = e;
      if (B.robot_indices) B.robot_indices[j] = base + P.robot_slot;
      if (B.reset_root_indices) {  // unique(cat(robot, object, goal)) == sorted, and sorted == per-env triples
        B.reset_root_indices[3 * j] = base + P.robot_slot;
        B.reset_root_indices[3 * j + 1] = base + P.object_slot;
        B.reset_root_indices[3 * j + 2] = base + P.goal_slot;
      }
    }
    if (f_goal) {
      const int64_t j = (int64_t)ex_b + t.rank_b;
      B.goal_reset_ids[j] = e;
      if (B.goal_root_indices) B.goal_root_indices[j] = (int32_t)(P.actors_per_env * e) + P.goal_slot;
    }
    LG_TP(1, 4, tid == NT - kScanThreads);
  };
  if (rank_first) {
    if (scan_group) finish_scan();
    __syncthreads();
  } else if (SPLIT && !resets && scan_group) {
    finish_scan();
  }

  // ---- row group: this env's action row: noise (extension), clamp, reset ----------------------------------
  float act[A];
  if (row_group) {
    if (full_tile) mbar_wait(&s_mbar, 0);   // the slabs have landed
    LG_TP(1, 5, tid == 0);
    if (live) {
      const bool zero_row = (s_flag[gt] & 1) != 0;
#pragma unroll
      for (int c = 0; c < A; ++c) act[c] = s_act[gt * A + c];
      // extension (no reference code): per-episode action offset, then Gaussian action noise.  An env that resets in
      // this step stores 0 below, so its offset row being redrawn by this pass meanwhile does not matter.
      // dr_activate (hot parameter line) is tested first: the two sigmas sit in cold lines of the parameter block.
      const bool noise = P.dr_activate && P.dr_action_sigma != 0.0f;
      if (P.dr_activate && (noise || P.dr_action_bias_sigma != 0.0f)) {
        float noisy[A];                                    // a copy: `act` itself must stay in registers
#pragma unroll
        for (int c = 0; c < A; ++c) noisy[c] = act[c];
        perturb_action<A>(P, P.dr_action_bias_sigma != 0.0f ? B.action_bias + e * A : nullptr, noise,
                          (uint64_t)(P.env_offset + e), epoch, noisy);
#pragma unroll
        for (int c = 0; c < A; ++c) act[c] = noisy[c];
      }
      if (P.clip_input_actions) {   // the wrapper's clamp (wrappers/vec_task.py:162)
        const float clip = P.clip_actions;
#pragma unroll
        for (int c = 0; c < A; ++c) act[c] = clamp_nan(act[c], -clip, clip);
      }
      if (zero_row) {               // the row is zeroed after the store (envs/env_base.py:369, trifinger_env.py:387)
#pragma unroll
        for (int c = 0; c < A; ++c) act[c] = 0.0f;
      }
#pragma unroll
      for (int c = 0; c < A; ++c) s_act[gt * A + c] = act[c];
    }
    LG_TP(1, 6, tid == 0);
  }
  // ---- resets (trifinger_env.py:373-440) -----------------------------------------------------------------
  // Block-uniform branch: a tile without flagged envs neither fetches nor executes sampler code.  The flagged envs
  // are listed in shared memory by their rank in the tile, and the eight reset sub-tasks are spread over the eight
  // warps (lane = listed env): uniform control flow, and a serial chain of ~2 Philox blocks per warp instead of ten
  // per resetting thread.
  if (resets) {
    if (full_tile && !row_group) mbar_wait(&s_mbar, 0);   // new joint rows are mirrored into the landed slab (the row group has waited)
    const uint32_t ex_a = s_scan[2], ex_b = s_scan[3];     // meaningful with injected / torch draws only (rank_first)
    const int warp = tid >> 5, lane = tid & 31;
    uint64_t t_seed = 0, t_base = 0;
    uint32_t t_kr = 0, t_kg = 0;
    if constexpr (TORCH) {   // written by the counting launch, which completed before this grid started
      t_seed = B.torch_rng->seed; t_base = B.torch_rng->launch_base;
      t_kr = (uint32_t)B.torch_rng->launch_counts[0]; t_kg = (uint32_t)B.torch_rng->launch_counts[1];
    }
    auto run_sub = [&](int sub, int first, int step) {
#pragma unroll 1
      for (int r = first; r < na; r += step) {
        const int ent = s_reset_list[r], local = ent & 0x7fff;
        const int64_t env = e0 + local;
        if constexpr (TORCH) {
          const TorchDraws dr = make_torch_draws(P, t_seed, t_base, t_kr, false, (int64_t)ex_a + r);
          reset_subtask(P, S, B, env, sub, dr, (ent & 0x8000) != 0, s_dof + local * 18, !DIRECT);
        } else {
          const DrawSource dr = make_draws(P, (uint64_t)epoch, env, kPurposeReset, B.inject_reset_u, B.inject_reset_n,
                                           (int64_t)ex_a + r);
          reset_subtask(P, S, B, env, sub, dr, (ent & 0x8000) != 0, s_dof + local * 18, !DIRECT);
        }
      }
    };
    // Work items = (sub-task, chunk of 32 listed envs).  The four long sub-tasks (object position 5 / yaw 8, goal
    // position 6 / orientation 9) come first, one item per warp; the six short ones (joint blocks 0..4, bookkeeping 7)
    // follow, dealt round-robin.
    constexpr int kWarps = NT / 32;
    {
      const int long_subs[4] = {5, 8, 6, 9};
      if (SPLIT) run_sub(long_subs[warp >> 1], (warp & 1) * 32 + lane, 64);   // two warps per long sub-task
      else run_sub(long_subs[warp], lane, 32);
      const int short_subs[6] = {0, 1, 2, 3, 4, 7};
      constexpr int kChunks = SPLIT ? 2 : 1;
#pragma unroll 1
      for (int item = warp; item < 6 * kChunks; item += kWarps)
        run_sub(short_subs[item / kChunks], (item % kChunks) * 32 + lane, 32 * kChunks);
    }
    // goal resets second, as in env_base.py:374-379: position and orientation halves on different halves of the CTA
    if (nb) {
      const int half = tid >= NT / 2 ? 1 : 0, t2 = tid - half * (NT / 2);
#pragma unroll 1
      for (int r = t2; r < nb; r += NT / 2) {
        const int64_t env = e0 + s_goal_list[r];
        if (!DIRECT && half == 0) B.goal_reset[env] = 0;  // trifinger_env.py:427
        if constexpr (TORCH) {   // the goal-reset list draws after the whole reset list's calls
          const TorchDraws dr = make_torch_draws(P, t_seed, t_base + torch_plan(P, t_kr, false).total(), t_kg, true,
                                                 (int64_t)ex_b + r);
          apply_goal_sample(P, S, B, env, dr, half);
        } else {
          const DrawSource dr = make_draws(P, (uint64_t)epoch, env, kPurposeGoal, B.inject_goal_u, B.inject_goal_n,
                                           (int64_t)ex_b + r);
          apply_goal_sample(P, S, B, env, dr, half);
        }
      }
    }
    LG_TP(1, 7, tid == 0);
    if (handshake) {
      // the flag bytes of this tile may only be cleared once no tile reads them any more (all tiles run: the grid is
      // co-resident; by now — a whole reset phase after the reads were issued — the wait is over before it starts)
      while (ld_volatile_u32(&B.control->scan_readers) < (uint32_t)num_tiles) {}
      __threadfence();
    }
    __syncthreads();   // the mirrored joint rows are final before the torque reads them
    if (handshake) tile_passed();
    if (DIRECT) {      // trifinger_env.py:382 (`_reset_buf[env_ids] = 0`), :427
      for (int r = tid; r < na; r += NT) B.reset[e0 + (s_reset_list[r] & 0x7fff)] = 0;
      for (int r = tid; r < nb; r += NT) B.goal_reset[e0 + s_goal_list[r]] = 0;
    }
    if (SPLIT && !rank_first && scan_group) finish_scan();
  }
  // ---- moving goal (__update_goal_movement_pre, trifinger_env.py:1267-1277): every step the goal body's
  // angular velocity is re-imposed from the movement buffer (freshly sampled above for envs that reset)
  if (P.goal_rotation && row_group && live) {
    float* row = S.root_state + (P.actors_per_env * e + P.goal_slot) * 13;
    const float* gm = B.goal_movement + e * 6;
    row[10] = gm[3]; row[11] = gm[4]; row[12] = gm[5];
  }
  // ---- action -> torque (trifinger_env.py:442-498), on the post-reset joint state (row group, thread = env) ----
  if (want_torque && row_group && live) {
    torque_one_env(P, act, s_dof + gt * 18, s_tq + gt * 9);   // resets mirrored their joint rows into s_dof
  }
  // The post-physics pass may start launching now at the latest (tiles without resets said so after their block scan).
  LG_TP(1, 8, tid == 0);
  pdl_launch_dependents();
  if (full_tile) {
    fence_async_proxy();           // generic-proxy writes to the slabs -> visible to the bulk-copy engine
    // the slabs that leave are written by the row group alone: the scan group (still busy with its id lists, or waiting
    // for an atomic's answer) is not waited for
    if (!SPLIT) __syncthreads();
    else if (row_group) group_sync<2>();
    if (tid == 0) {
      bulk_store(B.action + e0 * A, s_act, sizeof(float) * E * A);
      if (want_torque) bulk_store(B.applied_torque + e0 * 9, s_tq, sizeof(float) * E * 9);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      LG_TP(1, 9, tid == 0);
      // shared memory must outlive the bulk stores that read it
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
  } else {
    __syncthreads();
    for (int i = tid; i < nvalid * A; i += NT) B.action[e0 * A + i] = s_act[i];
    if (want_torque)
      for (int i = tid; i < nvalid * 9; i += NT) B.applied_torque[e0 * 9 + i] = s_tq[i];
  }
  if (!SPLIT && !rank_first) finish_scan();   // one group: the look-back and the id lists come last
  LG_TP(1, 11, tid == 0);
}

// standalone compaction (torch.nonzero(mask).view(-1))
__global__ void __launch_bounds__(kScanThreads)
compact_kernel(const uint8_t* __restrict__ mask, int64_t n, int64_t* __restrict__ ids, int32_t* counts2,
               uint64_t* status, LgControl* ctl, int num_tiles) {
  __shared__ int s_tile;
  __shared__ uint32_t s_epoch;
  __shared__ uint32_t s_wa[kScanThreads / 32], s_wb[kScanThreads / 32];
  if (threadIdx.x == 0) {
    s_epoch = ld_volatile_u32(&ctl->scan_epoch);
    s_tile = (int)atomicAdd(&ctl->scan_ticket, 1u);
  }
  __syncthreads();
  const int gt = threadIdx.x;
  const int64_t e = (int64_t)s_tile * kScanThreads + gt;
  const bool f = e < n && mask[e] != 0;
  TileScan t;
  t.tile = s_tile; t.epoch = s_epoch;
  tile_scan_local<0>(f, false, gt, s_wa, s_wb, t);
  if (gt == 0)
    atomicExch(reinterpret_cast<unsigned long long*>(status + t.tile),
               (unsigned long long)pack_status(t.epoch, t.tile == 0 ? kStateInclusive : kStateAggregate, t.total_a, 0));
  uint32_t ex_a, ex_b;
  tile_scan_finish<true, 0>(ctl, status, t, num_tiles, gt, ex_a, ex_b, counts2);
  if (f) ids[(int64_t)ex_a + t.rank_a] = e;
}

// LG_RNG_TORCH, in front of the pre-physics pass: the lengths of both lists (flags OR forced masks), and the base
// offset of the launch; advances the generator by all of the launch's calls.  No CTA waits for another: the last one to
// finish (ticket) publishes.  The pre-physics pass is launched in stream order behind it.
constexpr int kCountThreads = 256;
__global__ void __launch_bounds__(kCountThreads)
torch_count_kernel(const uint8_t* __restrict__ reset, const uint8_t* __restrict__ goal, const uint8_t* __restrict__ force_reset,
                   const uint8_t* __restrict__ force_goal, int64_t n, const __grid_constant__ LgParams P, LgTorchRng* rng) {
  __shared__ uint32_t s_cnt[kCountThreads / 32][2];
  __shared__ bool s_last;
  uint32_t a = 0, b = 0;
  for (int64_t i = (int64_t)blockIdx.x * kCountThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kCountThreads) {
    a += (reset[i] | (force_reset ? force_reset[i] : 0)) != 0;
    b += (goal[i] | (force_goal ? force_goal[i] : 0)) != 0;
  }
  a = __reduce_add_sync(0xffffffffu, a);
  b = __reduce_add_sync(0xffffffffu, b);
  if ((threadIdx.x & 31) == 0) { s_cnt[threadIdx.x >> 5][0] = a; s_cnt[threadIdx.x >> 5][1] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    a = b = 0;
    for (int w = 0; w < kCountThreads / 32; ++w) { a += s_cnt[w][0]; b += s_cnt[w][1]; }
    if (a) atomicAdd(&rng->acc[0], a);
    if (b) atomicAdd(&rng->acc[1], b);
    __threadfence();
    s_last = atomicAdd(&rng->ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (s_last && threadIdx.x == 0) {
    __threadfence();
    const uint32_t kr = ld_volatile_u32(&rng->acc[0]), kg = ld_volatile_u32(&rng->acc[1]);
    const uint64_t base = rng->offset;
    rng->launch_base = base;
    rng->launch_counts[0] = (int32_t)kr; rng->launch_counts[1] = (int32_t)kg;
    rng->offset = base + torch_plan(P, kr, false).total() + torch_plan(P, kg, true).total();
    rng->acc[0] = 0; rng->acc[1] = 0; rng->ticket = 0;
  }
}

// torch.rand(n) / torch.randn(n) as the batched primitive lg_torch_philox: one element per thread
__global__ void torch_philox_kernel(uint64_t seed, uint64_t offset, uint32_t n, uint32_t gmax, int normal, float* out) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  int lane;
  const U4 w = torch_block(seed, offset, n, gmax, j, lane);
  out[j] = normal ? torch_normal(w, lane) : torch_uniform(u4_lane(w, lane));
}

// the hooks' torch stream: the list's calls were drawn from the offset the launch read; advance it past them
__global__ void torch_advance_kernel(LgTorchRng* rng, uint64_t adv) { rng->offset += adv; }

// hooks on explicit id lists: what one listed env gets, for either draw source
template <class D>
__device__ __forceinline__ void hook_goal_env(const LgParams& P, const LgSimState& S, const LgBuffers& B, int64_t e,
                                              int64_t j, const D dr) {
  B.goal_reset[e] = 0;
  apply_goal_sample(P, S, B, e, dr);
  if (B.goal_root_indices) B.goal_root_indices[j] = (int32_t)(P.actors_per_env * e) + P.goal_slot;
}
template <class D>
__device__ __forceinline__ void hook_reset_env(const LgParams& P, const LgSimState& S, const LgBuffers& B, int64_t e,
                                               int64_t j, const D dr) {
  reset_one_env(P, S, B, e, dr);
  const int32_t base = (int32_t)(P.actors_per_env * e);
  if (B.robot_indices) B.robot_indices[j] = base + P.robot_slot;
  if (B.reset_root_indices) {
    B.reset_root_indices[3 * j] = base + P.robot_slot;
    B.reset_root_indices[3 * j + 1] = base + P.object_slot;
    B.reset_root_indices[3 * j + 2] = base + P.goal_slot;
  }
}
template <bool TORCH = false>
__global__ void reset_ids_kernel(const __grid_constant__ LgParams P, const LgSimState S, const LgBuffers B,
                                 const int64_t* __restrict__ ids, int64_t k, int goal_only) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= k) return;
  const int64_t e = ids[j];
  // never collides with the fused path's epochs; keys the own stream's draws and, on either stream, the DR offsets
  const uint64_t epoch = B.control->rng_epoch | (1ull << 63);
  if constexpr (TORCH) {   // the list's rank j is the env's index in the reference's calls
    const TorchDraws dr = make_torch_draws(P, B.torch_rng->seed, B.torch_rng->offset, (uint32_t)k, goal_only != 0, j);
    if (goal_only) hook_goal_env(P, S, B, e, j, dr);
    else hook_reset_env(P, S, B, e, j, dr);
    if (!goal_only && (B.obs_bias || B.action_bias)) draw_bias(P, B, e, epoch);   // extension: new offsets
  } else {
    if (goal_only) {
      const DrawSource dr = make_draws(P, epoch, e, kPurposeGoal, B.inject_goal_u, B.inject_goal_n, j);
      hook_goal_env(P, S, B, e, j, dr);
    } else {
      const DrawSource dr = make_draws(P, epoch, e, kPurposeReset, B.inject_reset_u, B.inject_reset_n, j);
      hook_reset_env(P, S, B, e, j, dr);
      if (B.obs_bias || B.action_bias) draw_bias(P, B, e, epoch);
    }
  }
}
__global__ void bump_epoch_kernel(LgControl* ctl) { ctl->rng_epoch += 1; }

// extension (per-episode DR offsets): the envs the pre-physics launch in front of it reset (its reset list) draw their
// new offsets, keyed like that launch's own draws by the compaction epoch it ran under (it advanced scan_epoch by one on
// its way out).  One warp per listed env, lane = Philox block (draw_bias_block), grid-stride over the list.  A launch of
// its own, made only when the offsets are on: inside the pre-physics pass the draw cost every one of its instantiations
// spills, whether the offsets were on or not.  Launched programmatically: it becomes resident while that pass finishes.
constexpr int kDrawBiasThreads = 256;
__global__ void __launch_bounds__(kDrawBiasThreads) draw_bias_kernel(const __grid_constant__ LgParams P, const LgBuffers B) {
  pdl_launch_dependents();   // the post-physics pass may become resident; it waits for this grid to complete
  pdl_wait();                // the reset list and the epoch are results of the pre-physics pass
  const int64_t n = (int64_t)B.counts[0] * 32;
  const uint64_t epoch = (uint32_t)(ld_volatile_u32(&B.control->scan_epoch) - 1u);
  for (int64_t t = (int64_t)blockIdx.x * kDrawBiasThreads + threadIdx.x; t < n; t += (int64_t)gridDim.x * kDrawBiasThreads)
    draw_bias_block(P, B, B.reset_ids[t >> 5], epoch, (int)(t & 31));
}

__global__ void pre_step_kernel(const __grid_constant__ LgParams P, const LgSimState S, const LgBuffers B) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P.num_envs) return;
  float act[LG_MAX_ACTION_DIM];
  for (int c = 0; c < P.action_dim; ++c) act[c] = B.action[e * P.action_dim + c];
  torque_one_env(P, act, S.dof_state + e * 18, B.applied_torque + e * 9);
  if (P.goal_rotation) {  // __update_goal_movement_pre (trifinger_env.py:1267-1277)
    float* row = S.root_state + (P.actors_per_env * e + P.goal_slot) * 13;
    const float* gm = B.goal_movement + e * 6;
    row[10] = gm[3]; row[11] = gm[4]; row[12] = gm[5];
  }
}

}  // namespace lg
