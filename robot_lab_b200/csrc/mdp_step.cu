// mdp_step.cu - fused per-step MDP pipeline for sm_100a (B200).
//
// One launch evaluates, for every env of a CTA's tile: termination terms, all reward terms (+ episode sums
// and per-term step rewards), the velocity-command update, both observation groups and the ordered
// compaction of reset ids. Reference behaviour restated (paths relative to /root/reference, V/ =
// source/robot_lab/robot_lab/tasks/manager_based/locomotion/velocity/): V/mdp/rewards.py:22-687,
// V/mdp/observations.py:17-35, V/mdp/commands.py:22-85, V/velocity_env_cfg.py:106-254,379-664 and the
// IsaacLab manager loops / upstream terms listed in SURVEY.md Appendix A.
//
// Execution model (HBM-bound by arithmetic intensity, ~0.5 FLOP/B, no tensor cores; at a few thousand envs bound
// by first-touch latency - see DESIGN.md 2 and profiles/r1_summary.md):
//   * a CTA owns a tile of 32 consecutive envs; in the compute phase lane e of every warp IS env e (no lane
//     repeats another lane's per-env scalar work) and the warps differ in which terms they evaluate (a constexpr
//     longest-processing-time schedule, reached through one binary-search branch per warp);
//   * load phase: the AoS sensor rows (contact-force history, height-scan ray hits) are staged into shared
//     memory with 1-D TMA bulk copies (cp.async.bulk + mbarrier complete_tx), the small per-env SoA fields with
//     16-byte cp.async into an SoA [word][32] record - all global reads of the tile are in flight before any
//     arithmetic starts, one join;
//   * stage 1 works on shared memory only, every warp finishes its terms (weight, dt, episode sum, step reward)
//     and assembles its observation columns in the shared-memory rows; stage 2 (warp 0) adds the reward up in
//     manager order;
//   * store phase: observation rows leave with bulk stores (cp.async.bulk.global.shared::cta), the SoA outputs
//     with 16-byte stores; the last CTA to finish compacts the reset ids from per-CTA bit masks / combines the
//     reset-logging partials.
//
// Built with -fmad=false on purpose: the reference is eager PyTorch, every op rounds on its own, and not
// contracting a*b+c keeps threshold decisions (contact > 1 N, |cmd| > 0.1, ...) bit-identical.

#include "mdp_terms.cuh"
#include "mdp_ctx.h"



namespace {


// ---------------------------------------------------------------------------------------------------
// Tile movers (one code copy each)
// ---------------------------------------------------------------------------------------------------
// The small per-env fields: field f is moved by warp f mod NW, its lanes stride over the field's rows (a "row" is
// one component of one field; record word w of local env e lives at sm[w*kE + e]). Deliberately a LOOP over
// per-field metadata and not per-field code: every SM sees this code exactly once per launch, so its size - not
// its instruction count - is what the load phase costs (profiles/r1_front_end.md).
__device__ __noinline__ void field_load_elems(float* sm, FieldD fd, int nc, int w0, int env0, int nvalid,
                                              const int32_t* ids, int lane) {
  if (lane >= nvalid) return;   // any strides, ragged tiles, env-id lists: lane = env, one element per copy
  const long long env = ids ? (long long)ids[env0 + lane] : (long long)(env0 + lane);
  const float* src = static_cast<const float*>(fd.ptr) + env * fd.es;
  float* dst = sm + w0 * kE + lane;
#pragma unroll 4
  for (int c = 0; c < nc; ++c) cp_async4(dst + c * kE, src + (long long)c * fd.cs);
}
__device__ __noinline__ void field_store_elems(const float* sm, FieldD fd, int nc, int w0, int env0, int nvalid,
                                               const int32_t* ids, int lane) {
  if (lane >= nvalid) return;
  const long long env = ids ? (long long)ids[env0 + lane] : (long long)(env0 + lane);
  float* dst = static_cast<float*>(const_cast<void*>(fd.ptr)) + env * fd.es;
  const float* src = sm + w0 * kE + lane;
#pragma unroll 4
  for (int c = 0; c < nc; ++c) dst[(long long)c * fd.cs] = src[c * kE];
}
__device__ __forceinline__ void load_fields(float* sm, const KArgs& a, int env0, int nvalid, const int32_t* ids,
                                            bool full, int warp, int lane, int nwarps) {
#pragma unroll 1
  for (int f = warp; f < IF_COUNT; f += nwarps) {
    if (!((a.in_mask >> f) & 1u)) continue;
    const FieldD fd = a.in[f];
    const int nc = fd.meta & 0xffff, w0 = fd.meta >> 16;
    if (full && ((a.in_vec4 >> f) & 1u)) {   // SoA rows: 16 bytes (4 envs) per copy
      const float* src = static_cast<const float*>(fd.ptr) + env0;
#pragma unroll 1
      for (int j = lane; j < nc * (kE / 4); j += 32)
        cp_async16(sm + (w0 + (j >> 3)) * kE + 4 * (j & 7), src + (size_t)(j >> 3) * fd.cs + 4 * (j & 7));
    } else {
      field_load_elems(sm, fd, nc, w0, env0, nvalid, ids, lane);
    }
  }
}
__device__ __forceinline__ void store_fields(const float* sm, const KArgs& a, uint32_t omask, int env0, int nvalid,
                                             const int32_t* ids, bool full, int warp, int lane, int nwarps) {
#pragma unroll 1
  for (int f = warp; f < OF_COUNT; f += nwarps) {
    if (!((omask >> f) & 1u)) continue;
    const FieldD fd = a.outf[f];
    const int nc = fd.meta & 0xffff, w0 = fd.meta >> 16;
    if (full && ((a.out_vec4 >> f) & 1u)) {
      float* dst = static_cast<float*>(const_cast<void*>(fd.ptr)) + env0;
#pragma unroll 1
      for (int j = lane; j < nc * (kE / 4); j += 32)
        *reinterpret_cast<float4*>(dst + (size_t)(j >> 3) * fd.cs + 4 * (j & 7)) =
            *reinterpret_cast<const float4*>(sm + (w0 + (j >> 3)) * kE + 4 * (j & 7));
    } else {
      field_store_elems(sm, fd, nc, w0, env0, nvalid, ids, lane);
    }
  }
}

// AoS span [kE][pitch] <-> global rows, element-wise (used when a span is not one aligned contiguous block or the
// shared-memory pitch is padded)
__device__ __noinline__ void span_load_elems(float* dst, int pitch, FieldD fd, int ncomp, int env0, int nvalid,
                                             const int32_t* ids, int tid, int nthreads) {
  const int warp = tid >> 5, lane = tid & 31, nw = nthreads >> 5;
  for (int el = warp; el < nvalid; el += nw) {   // a warp walks one env's row: coalesced when rows are contiguous
    const long long env = ids ? (long long)ids[env0 + el] : (long long)(env0 + el);
    const float* src = static_cast<const float*>(fd.ptr) + env * fd.es;
    for (int c = lane; c < ncomp; c += 32) cp_async4(dst + el * pitch + c, src + (long long)c * fd.cs);
  }
}
__device__ __noinline__ void span_store_elems(const float* src, int pitch, float* ptr, long long es, int ncomp,
                                              int env0, int nvalid, const int32_t* ids, int tid, int nthreads) {
  const int warp = tid >> 5, lane = tid & 31, nw = nthreads >> 5;
  for (int el = warp; el < nvalid; el += nw) {
    const long long env = ids ? (long long)ids[env0 + el] : (long long)(env0 + el);
    for (int c = lane; c < ncomp; c += 32) ptr[env * es + c] = src[el * pitch + c];
  }
}
// one aligned contiguous [kE][ncomp] block in global memory AND an unpadded shared-memory pitch
__device__ __forceinline__ bool span_bulk_ok(const FieldD& fd, int ncomp, int pitch, int env0) {
  if (fd.ptr == nullptr || ncomp <= 0 || pitch != ncomp || fd.cs != 1 || fd.es != ncomp) return false;
  const uintptr_t p = reinterpret_cast<uintptr_t>(fd.ptr) + (uintptr_t)env0 * (uintptr_t)ncomp * 4u;
  return ((p & 15u) == 0) && ((((long long)kE * ncomp * 4) & 15) == 0);
}
__device__ __forceinline__ void store_u8(const float* sm, int off, const FieldD& fd, int env0, int nvalid,
                                         const int32_t* ids, int tid) {
  if (fd.ptr != nullptr && tid < nvalid) {
    const long long env = ids ? (long long)ids[env0 + tid] : (long long)(env0 + tid);
    static_cast<uint8_t*>(const_cast<void*>(fd.ptr))[env * fd.es] = (uint8_t)__float_as_int(sm[off + tid]);
  }
}

// ---------------------------------------------------------------------------------------------------
// The fused step kernel: kE = 32 envs per CTA, NW warps. MODE 0 = step, MODE 1 = single-term evaluation.
//   load   : everything asynchronous (TMA bulk copies + cp.async), one join
//   stage 1: every warp runs its share of the schedule, thread-per-env (lane e = env e)
//   stage 2: warp 0 adds the reward up in manager order (and finishes is_terminated)
//   store  : bulk stores for the observation rows, per-field loops for the SoA outputs; last CTA compacts reset ids
// ---------------------------------------------------------------------------------------------------
template <class P, int NW, int MODE, bool DBG>
__global__ void __launch_bounds__(NW * 32) mdp_step_kernel(const KArgs a) {
  extern __shared__ __align__(128) float sm[];
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ int s_last;
  const Scalars S = P::scalars(a);
  const Layout L = P::layout(a);
  constexpr bool CN = false;    // HIST_MAX_NORM computes the contact-force norms where they are used (the cluster kernels cache them)
  constexpr int NT = NW * 32;   // threads per CTA = per tile
  const int tid = (int)threadIdx.x;
  const int vb = (int)blockIdx.x;        // tile index
  const int vgrid = (int)gridDim.x;
  auto tile_sync = [&]() __attribute__((always_inline)) { __syncthreads(); };
  auto tile_sync_or = [&](bool pred) __attribute__((always_inline)) -> int { return __syncthreads_or(pred); };
#define RL_STAMP(i) do { if constexpr (DBG) { if (tid == 0) a.dbg[(size_t)vb * RL_DEBUG_STRIDE + (i)] = clock64(); } } while (0)
#define RL_SUB(i) RL_STAMP(8 + RL_MAX_TASKS + 32 + (i))   /* finer stamps inside the load phase (debug build only) */
  RL_STAMP(0);
  const int warp = tid >> 5;
  const int e = tid & 31;       // compute phase: this lane's env inside the tile
  const uint32_t ph = a.phases;
  if (a.use_pdl) {
    // launch-latency overlap only: every read below may depend on the predecessor, so wait first
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
  }
  const int n_total = a.has_ids ? *a.n_env_ids : a.N;
  const int env0 = vb * kE;
  const int K = S.num_reward_terms;
  // RESET comes in two forms: on an env-id list (gathered tiles, every env of the launch is reset) or - without
  // a list - over all envs, resetting those whose terminated | truncated byte is set (full-tile fast path)
  const bool do_reset = (MODE == 0) && (ph & RL_PHASE_RESET) != 0;
  const bool reset_masked = do_reset && !a.has_ids;
  // (the masked form reads its reset count only in the tail: a dependent global load up here would stall the
  // whole prologue; the id-list form needs its count for the bounds anyway)
  if (do_reset && !reset_masked && n_total == 0 && vb == 0 && tid < RL_LOG_STRIDE) {
    // nothing to reset and no CTA reaches the tail: the logged scalars are defined as 0
    if (tid < K) { if (a.out.reset_log.episode_sum_mean) a.out.reset_log.episode_sum_mean[tid] = 0.f; }
    else if (tid < K + RL_MAX_DONE_TERMS) { if (a.out.reset_log.done_term_count) a.out.reset_log.done_term_count[tid - K] = 0.f; }
    else if (tid < K + RL_MAX_DONE_TERMS + 2) { if (a.out.reset_log.metric_mean) a.out.reset_log.metric_mean[tid - K - RL_MAX_DONE_TERMS] = 0.f; }
  }
  if (env0 >= n_total && !(ph & RL_PHASE_COMPACT)) return;
  const int nvalid = max(0, min(kE, n_total - env0));
  const int32_t* ids = a.has_ids ? a.env_ids : nullptr;
  const int J = S.num_joints, A = S.n_actions;
  const int R = S.num_rays;
  const int HW = S.hist_len * S.num_hist_bodies * 3;
  const bool need_hist = (MODE == 1) || (ph & (RL_PHASE_DONES | RL_PHASE_REWARDS));
  const bool need_rays = (MODE == 0) && (ph & RL_PHASE_OBS) && R > 0 && a.rays.ptr != nullptr;
  const bool full = (nvalid == kE) && (ids == nullptr);
  RandState rs;
  rs.seed = a.rnd.seed;
  rs.step = a.rnd.step + (a.rnd.step_counter ? *a.rnd.step_counter : 0ull);
  rs.env_id_offset = a.rnd.env_id_offset;

  // ---- load phase: everything is asynchronous, nothing below waits until the single join point ---------
  if (nvalid > 0) {
    // the big transfers first: their DRAM latency overlaps everything else the prologue does
    const bool hist_bulk = need_hist && full && span_bulk_ok(a.hist, HW, L.hist_pitch, env0);
    const bool rays_bulk = need_rays && full && span_bulk_ok(a.rays, R, L.rays_pitch, env0);
    if (tid == 0) {
      mbar_init(&s_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      uint32_t bytes = 0;
      if (hist_bulk) bytes += (uint32_t)(kE * HW * 4);
      if (rays_bulk) bytes += (uint32_t)(kE * R * 4);
      mbar_expect_tx(&s_bar, bytes);
      if (hist_bulk) bulk_g2s(sm + L.hist, static_cast<const float*>(a.hist.ptr) + (size_t)env0 * HW, (uint32_t)(kE * HW * 4), &s_bar);
      if (rays_bulk) bulk_g2s(sm + L.rays, static_cast<const float*>(a.rays.ptr) + (size_t)env0 * R, (uint32_t)(kE * R * 4), &s_bar);
    }
    // byte-sized per-env flags: plain loads into registers, issued early so that their latency overlaps the
    // issue of everything else
    const bool want_cmd_flags = (MODE == 0) && (ph & (RL_PHASE_COMMAND | RL_PHASE_RESET)) != 0;
    const bool want_done_bits = do_reset && a.out.done_bits != nullptr;
    int u8_head = 0, u8_stand = 0, u8_bits = 0, u8_reset = do_reset ? 1 : 0;
    if (tid < nvalid) {
      const long long ev = ids ? (long long)ids[env0 + tid] : (long long)(env0 + tid);
      if (reset_masked) u8_reset = (a.out.terminated[ev] | a.out.truncated[ev]) != 0;
      if (want_cmd_flags) {
        if (a.is_heading.ptr) u8_head = static_cast<const uint8_t*>(a.is_heading.ptr)[ev * a.is_heading.es];
        if (a.is_standing.ptr) u8_stand = static_cast<const uint8_t*>(a.is_standing.ptr)[ev * a.is_standing.es];
      }
      if (want_done_bits) u8_bits = a.out.done_bits[ev];
    }
    RL_SUB(0);                  // prologue + bulk copies issued
    load_fields(sm, a, env0, nvalid, ids, full, warp, e, NW);
    RL_SUB(1);                  // per-field copies issued
    if (need_hist && !hist_bulk && a.hist.ptr) span_load_elems(sm + L.hist, L.hist_pitch, a.hist, HW, env0, nvalid, ids, tid, NT);
    if (need_rays && !rays_bulk) span_load_elems(sm + L.rays, L.rays_pitch, a.rays, R, env0, nvalid, ids, tid, NT);
    if (ph & RL_PHASE_REWARDS)
      for (int i = tid; i < K * kE; i += NT) {
        if ((a.rw_zero >> (i / kE)) & 1ull) {   // weight-0 terms: no task evaluates them
          sm[L.stepr + i] = 0.f;
          sm[L.termv + i] = 0.f;
        }
      }
    RL_SUB(2);                  // span loads issued
    // per-joint constants: ONE coalesced read of the [5][J] table in device memory (lane-indexed reads of the constant
    // bank serialise per address and miss one by one: 3.2 k cycles of a cold launch, measured in round 2)
    for (int i = tid; i < 5 * J; i += NT) sm[L.cj + i] = __ldg(a.cj + i);
    if (tid < nvalid) {         // the byte flags were requested at the top of the load phase
      if (want_cmd_flags) { sm[L.ishead + tid] = __int_as_float(u8_head); sm[L.isstand + tid] = __int_as_float(u8_stand); }
      if (want_done_bits) sm[L.flags + tid] = __int_as_float(u8_bits);
    }
    if (do_reset && tid < kE) sm[L.rmask + tid] = __int_as_float(tid < nvalid ? u8_reset : 0);
    RL_STAMP(1);                // all loads issued
    cp_async_wait_all();
    tile_sync();            // record + mbarrier init visible to everyone
    mbar_wait(&s_bar, 0);       // bulk copies landed
    RL_STAMP(2);                // tile resident
  }

  // Tickets of the two "last CTA" tails are taken EARLY - as soon as what the last CTA will read has been written -
  // and only looked at in the tail: the fence + atomic round trip (~1 us) overlaps the rest of the tile's work.
  unsigned early_prev = 0;
  const bool compact = (ph & RL_PHASE_COMPACT) && (ph & RL_PHASE_DONES) && !a.has_ids;
  constexpr int kCompactWarp = 1;   // idle during stage 2 (warp 0 sums the reward up)
  auto compact_arrive = [&]() __attribute__((always_inline)) {   // one warp: the tile's done mask, then its ticket
    const int f2 = (e < nvalid) ? __float_as_int(sm[L.flags + e]) : 0;
    const unsigned m = __ballot_sync(0xffffffffu, (f2 >> 8) & 3);
    if (e == 0) {
      a.cta_mask[vb] = m;
      early_prev = ticket_arrive_release(a.ticket);
    }
  };
  const bool valid = e < nvalid;
  const long long env = valid ? (ids ? (long long)ids[env0 + e] : (long long)(env0 + e)) : 0;
  if (nvalid > 0) {
    // ---- manager reset of the tile's envs that are being reset ------------------------------------------
    const int tile_resets = do_reset ? tile_sync_or(tid < kE && __float_as_int(sm[L.rmask + (tid & 31)]) != 0) : 0;
    if (do_reset && !tile_resets) {   // CTA-uniform: nothing to reset here, the logging partials are zero
      if (warp == 0) {
        for (int q = e; q < K + RL_MAX_DONE_TERMS + 2; q += 32) a.log_partials[(size_t)vb * RL_LOG_STRIDE + q] = 0.f;
        __syncwarp();
        // the tile's arrival at the logging reduction, long before the tail needs the answer (see the tail)
        if (e == 0) early_prev = ticket_arrive_release(a.ticket);
      }
    }
    if (tile_resets) {
      const bool rme = __float_as_int(sm[L.rmask + e]) != 0;
      // logging partials of this CTA (combined by the last CTA in a fixed order -> deterministic):
      // quantity q is reduced by warp q mod NW over its lanes (= envs) with a fixed shuffle tree
#pragma unroll 1
      for (int q = warp; q < K + RL_MAX_DONE_TERMS + 2; q += NW) {
        float x = 0.f;
        if (rme) {
          if (q < K) x = sm[L.sums + q * kE + e];
          else if (q < K + RL_MAX_DONE_TERMS)
            x = (a.out.done_bits != nullptr) ? (float)((__float_as_int(sm[L.flags + e]) >> (q - K)) & 1) : 0.f;
          else x = sm[(q == K + RL_MAX_DONE_TERMS ? L.mxy : L.myaw) + e];
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(0xffffffffu, x, d);
        if (e == 0) a.log_partials[(size_t)vb * RL_LOG_STRIDE + q] = x;
      }
      tile_sync();
      if (tid == 0) early_prev = ticket_arrive_release(a.ticket);   // partials of every warp ordered by the barrier
      // RewardManager / ActionManager / CommandTerm .reset [IL], episode_length_buf = 0
      for (int i = tid; i < kE * K; i += NT) if (__float_as_int(sm[L.rmask + (i & 31)]) != 0) sm[L.sums + i] = 0.f;
      for (int i = tid; i < kE * A; i += NT)
        if (__float_as_int(sm[L.rmask + (i & 31)]) != 0) { sm[L.act + i] = 0.f; sm[L.pact + i] = 0.f; }
      if (tid < kE && __float_as_int(sm[L.rmask + tid]) != 0) {
        const int el = tid;
        sm[L.mxy + el] = 0.f; sm[L.myaw + el] = 0.f;
        sm[L.eplen + el] = __int_as_float(0); sm[L.epnew + el] = __int_as_float(0);
        const auto& cc = P::command(a);
        const long long ev = ids ? (long long)ids[env0 + min(el, nvalid - 1)] : (long long)(env0 + el);
        float u[RL_NUM_CMD_UNIFORMS];
        if (a.rnd.cmd_uniforms != nullptr) {
#pragma unroll
          for (int q = 0; q < RL_NUM_CMD_UNIFORMS; ++q) u[q] = sm[L.cmdu + q * kE + el];
        } else {
          const uint4 r0 = rl_philox(rs, ev, RL_STREAM_RESET_COMMAND, 0), r1 = rl_philox(rs, ev, RL_STREAM_RESET_COMMAND, 1);
          u[0] = u01(r0.x); u[1] = u01(r0.y); u[2] = u01(r0.z); u[3] = u01(r0.w);
          u[4] = u01(r1.x); u[5] = u01(r1.y); u[6] = u01(r1.z);
        }
        float c0 = u[1] * (cc.lin_vel_x_hi - cc.lin_vel_x_lo) + cc.lin_vel_x_lo;
        float c1 = u[2] * (cc.lin_vel_y_hi - cc.lin_vel_y_lo) + cc.lin_vel_y_lo;
        const float c2 = u[3] * (cc.ang_vel_z_hi - cc.ang_vel_z_lo) + cc.ang_vel_z_lo;
        const float keep = (sqrtf(c0 * c0 + c1 * c1) > cc.small_cmd_threshold) ? 1.f : 0.f;
        c0 *= keep; c1 *= keep;
        sm[L.cmd + 0 * kE + el] = c0; sm[L.cmd + 1 * kE + el] = c1; sm[L.cmd + 2 * kE + el] = c2;
        sm[L.cmdn + 0 * kE + el] = c0; sm[L.cmdn + 1 * kE + el] = c1; sm[L.cmdn + 2 * kE + el] = c2;
        sm[L.tleft + el] = u[0] * (cc.resampling_time_hi - cc.resampling_time_lo) + cc.resampling_time_lo;
        if (cc.heading_command) {
          sm[L.head + el] = u[4] * (cc.heading_hi - cc.heading_lo) + cc.heading_lo;
          sm[L.ishead + el] = __int_as_float((u[5] <= cc.rel_heading_envs) ? 1 : 0);
        }
        sm[L.isstand + el] = __int_as_float((u[6] <= cc.rel_standing_envs) ? 1 : 0);
      }
      // envs that are NOT reset keep their episode length: the OF_EPLEN row is stored from the `epnew` word, which the
      // DONES task (absent from a RESET launch) would otherwise have written (round-1 advisor finding: stale shared
      // memory was stored for the live lanes of a tile with at least one reset)
      if (tid < kE && __float_as_int(sm[L.rmask + tid]) == 0) sm[L.epnew + tid] = sm[L.eplen + tid];
      tile_sync();
    }

    // ---- stage 1: thread-per-env, warps run different tasks ------------------------------------------------
    EnvCtx c = make_ctx(sm, L, e);
    if (MODE == 1) {
      if (warp == 0) {
        if (a.ext_terminated != nullptr && valid) c.terminated = a.ext_terminated[env] != 0;
        const float v = reward_term<CN>(*a.adhoc, *a.adhoc, S, L, sm, e, c, 0, 64);
        if (valid) a.term_out[env] = v;
      }
      return;
    }
    const int eplen_now = __float_as_int(SMF(L.eplen, 0)) + ((ph & RL_PHASE_DONES) ? 1 : 0);
    // TerminationManager.compute [IL] for this lane's env: bits | terminated << 8 | time_out << 9
    auto eval_dones = [&]() -> int {
      uint32_t bits = 0, term = 0, trunc = 0;
      const float* h = sm + L.hist + e * L.hist_pitch;
      P::for_dones(a, [&](const RlDoneTerm& t, int d) __attribute__((always_inline)) {
        int fired = 0;
        if (t.type == RL_DONE_TIME_OUT) {
          fired = eplen_now >= S.max_episode_length;
        } else if (t.type == RL_DONE_TERRAIN_OUT_OF_BOUNDS) {
          fired = (t.p[2] != 0.f) && ((fabsf(c.pos.x) > t.p[0]) || (fabsf(c.pos.y) > t.p[1]));
        } else if (t.type == RL_DONE_ILLEGAL_CONTACT) {
          _Pragma("unroll 1")
          for (int b = 0; b < S.num_hist_bodies; ++b)
            if (((t.body_mask >> b) & 1ull) && (HIST_MAX_NORM(h, b) > t.p[0])) fired = 1;
        }
        if (fired) { bits |= 1u << d; if (t.time_out) trunc = 1; else term = 1; }
      });
      return (int)(bits | (term << 8) | (trunc << 9));
    };
    if constexpr (DBG) { if (e == 0) a.dbg[(size_t)vb * RL_DEBUG_STRIDE + 8 + RL_MAX_TASKS + warp] = clock64(); }
    P::template for_tasks<NW>(a, warp, [&](auto, const Task& tk, const RlRewardTerm& rt, const RlObsTerm& ot, const bool corrupt,
                                          const int task_idx) __attribute__((always_inline)) {
      long long t_begin = 0;
      if constexpr (DBG) t_begin = clock64();
      [&]() __attribute__((always_inline)) {
      if (tk.kind == TK_REWARD) {
        if (!(ph & RL_PHASE_REWARDS)) return;
        const float raw = reward_term<CN>(rt, c_spec[a.slot].rewards[tk.a], S, L, sm, e, c, tk.lo, tk.hi);
        const int k = tk.a;
        // RewardManager.compute [IL]: value = func * weight * dt; sums += value; step_reward = value / dt
        const float val = (raw * rt.weight) * S.step_dt;
        SMF(L.termv, k) = val;
        SMF(L.sums, k) = SMF(L.sums, k) + val;
        SMF(L.stepr, k) = rl_div(val, S.step_dt);
      } else if (tk.kind == TK_OBS) {
        if (!(ph & RL_PHASE_OBS) || a.out.obs[tk.a] == nullptr) return;
        obs_task(sm, L, S, ot, c_spec[a.slot].obs[tk.a].terms[tk.b], corrupt, a, rs, tk.a, tk.b, tk.col0, tk.lo, tk.hi, e, env, c, eplen_now);
      } else if (tk.kind == TK_DONES) {
        if (!(ph & RL_PHASE_DONES)) return;
        SMF(L.epnew, 0) = __int_as_float(eplen_now);
        SMF(L.flags, 0) = __int_as_float(eval_dones());
      } else {  // TK_COMMAND: CommandManager.compute + the observation columns that show the new command
        if (!(ph & (RL_PHASE_COMMAND | RL_PHASE_OBS))) return;
        if (ph & RL_PHASE_COMMAND) {
          bool skip = false;
          if ((ph & RL_PHASE_SKIP_DONE_ENVS) && (ph & RL_PHASE_DONES)) skip = ((eval_dones() >> 8) & 3) != 0;
          command_update(sm, L, S, P::command(a), a, rs, e, env, c, !skip);
        } else if (!(ph & RL_PHASE_RESET)) {
          SMF(L.cmdn, 0) = c.c0; SMF(L.cmdn, 1) = c.c1; SMF(L.cmdn, 2) = c.c2;
        }
        if (ph & RL_PHASE_OBS) {
          P::for_cmd_obs(a, [&](const RlObsTerm& t, int g, int ti, int col0, bool corr) __attribute__((always_inline)) {
            if (a.out.obs[g] == nullptr) return;
            obs_task(sm, L, S, t, c_spec[a.slot].obs[g].terms[ti], corr, a, rs, g, ti, col0, 0, t.dim, e, env, c, eplen_now);
          });
        }
      }
      }();
      if constexpr (DBG) { if (e == 0) a.dbg[(size_t)vb * RL_DEBUG_STRIDE + 8 + task_idx] = clock64() - t_begin; }
    });
    tile_sync();
    RL_STAMP(3);                // stage 1 done
    if (compact && warp == kCompactWarp) compact_arrive();   // the termination flags are final

    // ---- stage 2: warp 0 finishes the late terms and adds the reward up in manager order ------------------
    if ((ph & RL_PHASE_REWARDS) && warp == 0) {
      // Kept as small as possible: warp 0 runs this alone, right after a barrier, on code no warp has touched -
      // what it costs is its length in instruction-cache lines. Weight-0 terms were zeroed in the load phase.
      float total = 0.f;
      if (a.rw_late != 0) {   // only is_terminated, which needs the termination result, is finished here
        const int fl = (ph & RL_PHASE_DONES) ? __float_as_int(SMF(L.flags, 0)) : 0;
        const bool terminated = ((fl >> 8) & 1) != 0;
#pragma unroll 1
        for (uint64_t m = a.rw_late & ~a.rw_zero; m != 0; m &= m - 1) {
          const int k = __ffsll((long long)m) - 1;
          const float raw = ((a.rw_isterm >> k) & 1ull) ? (terminated ? 1.f : 0.f) : SMF(L.termv, k);
          const float val = (raw * a.rw_weight[k]) * S.step_dt;
          SMF(L.termv, k) = val;
          SMF(L.sums, k) = SMF(L.sums, k) + val;
          SMF(L.stepr, k) = rl_div(val, S.step_dt);
        }
      }
      RL_SUB(3);                // late terms finished
#pragma unroll 1
      for (int k = 0; k < K; ++k) total += SMF(L.termv, k);   // manager order
      SMF(L.rew, 0) = total;
      RL_SUB(4);                // reward summed
    }
    tile_sync();
    RL_STAMP(4);                // stage 2 done

    // ---- store phase ----------------------------------------------------------------------------
    if (ph & RL_PHASE_OBS) {
      fence_proxy_async();
      tile_sync();
#pragma unroll
      for (int g = 0; g < RL_NUM_OBS_GROUPS; ++g) {
        const int D = P::obs_dim(a, g);
        if (a.out.obs[g] == nullptr || D <= 0) continue;
        const FieldD od{a.out.obs[g], (int)a.out.obs_pitch[g], 1};
        if (full && span_bulk_ok(od, D, LOBSP(g), env0)) {
          if (tid == 0) bulk_s2g(a.out.obs[g] + (size_t)env0 * D, sm + LOBS(g), (uint32_t)(kE * D * 4));
        } else {
          span_store_elems(sm + LOBS(g), LOBSP(g), a.out.obs[g], a.out.obs_pitch[g], D, env0, nvalid, ids, tid, NT);
        }
      }
      if (tid == 0) bulk_commit();
    }
    {
      uint32_t omask = a.out_mask;
      if (do_reset && !tile_resets) {   // nothing was reset here: those fields are unchanged
        omask &= ~((1u << OF_SUMS) | (1u << OF_ACT) | (1u << OF_PACT));
        if (!(ph & RL_PHASE_DONES)) omask &= ~(1u << OF_EPLEN);
      }
      store_fields(sm, a, omask, env0, nvalid, ids, full, warp, e, NW);
    }
    if (ph & RL_PHASE_DONES) {
      if (tid < nvalid) {
        const int f2 = __float_as_int(sm[L.flags + tid]);
        const long long ev = ids ? (long long)ids[env0 + tid] : (long long)(env0 + tid);
        if (a.out.done_bits) a.out.done_bits[ev] = (uint8_t)(f2 & 0xff);
        if (a.out.terminated) a.out.terminated[ev] = (uint8_t)((f2 >> 8) & 1);
        if (a.out.truncated) a.out.truncated[ev] = (uint8_t)((f2 >> 9) & 1);
      }
    }
    if ((ph & RL_PHASE_COMMAND) || do_reset) {
      store_u8(sm, L.ishead, a.is_heading, env0, nvalid, ids, tid);
      store_u8(sm, L.isstand, a.is_standing, env0, nvalid, ids, tid);
    }
  }

  RL_STAMP(5);                  // stores issued
  // ---- ordered compaction of reset ids (ManagerBasedRLEnv.step: reset_buf.nonzero() [IL]) -----------
  if (compact) {
    if (nvalid == 0 && warp == kCompactWarp) compact_arrive();   // tiles past the end: an empty mask
    if (tid == kCompactWarp * 32) s_last = (early_prev == (unsigned)(vgrid - 1));
    tile_sync();
    if (s_last) {
      __threadfence();
      int* s_cnt = reinterpret_cast<int*>(sm);  // this CTA's tile is dead once its own stores have been issued
      if ((ph & RL_PHASE_OBS) && nvalid > 0) { if (tid == 0) bulk_wait_read0(); }
      tile_sync();
      // one mask per CTA; thread i takes mask base+i, a block-wide exclusive scan of the popcounts gives its
      // first output slot -> ids come out ascending
      const int G = vgrid;
      int run = 0;
#pragma unroll 1
      for (int base = 0; base < G; base += NT) {
        const int g = base + tid;
        unsigned m = (g < G) ? __ldcg(a.cta_mask + g) : 0u;
        const int cnt = __popc(m);
        int incl = cnt;   // inclusive scan inside the warp
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, incl, d); if (e >= d) incl += y; }
        if (e == 31) s_cnt[warp] = incl;
        tile_sync();
        if (warp == 0) {
          int wt = (e < NW) ? s_cnt[e] : 0, wi = wt;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, wi, d); if (e >= d) wi += y; }
          if (e < NW) s_cnt[e] = wi - wt;           // exclusive prefix of the warp totals
          if (e == 31) s_cnt[32] = wi;              // chunk total
        }
        tile_sync();
        int pos = run + s_cnt[warp] + incl - cnt;
        if (a.out.reset_ids)
          while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1;
            a.out.reset_ids[pos++] = g * kE + b;
          }
        run += s_cnt[32];
        tile_sync();
      }
      if (tid == 0) {
        if (a.out.n_reset) *a.out.n_reset = run;
        *a.ticket = 0u;
      }
      return;
    }
  }
  if (do_reset && nvalid > 0) {
    const int n_cta = (n_total + kE - 1) / kE;
    if (tid == 0) s_last = (early_prev == (unsigned)(n_cta - 1));   // arrived right after the partials were written
    tile_sync();
    if (s_last) {
      __threadfence();
      // quantity q = lane, the CTAs' partials strided over the warps, then the warps' sums in warp order
      float* s_red = sm;   // this CTA's tile is dead once its own stores have been issued
      if ((ph & RL_PHASE_OBS) && tid == 0) bulk_wait_read0();
      tile_sync();
      for (int q = e; q < K + RL_MAX_DONE_TERMS + 2; q += 32) {
        float part = 0.f;
        for (int g = warp; g < n_cta; g += NW) part += __ldcg(a.log_partials + (size_t)g * RL_LOG_STRIDE + q);
        s_red[warp * RL_LOG_STRIDE + q] = part;
      }
      tile_sync();
      if (tid < K + RL_MAX_DONE_TERMS + 2) {
        float tot = 0.f;
        for (int w = 0; w < NW; ++w) tot += s_red[w * RL_LOG_STRIDE + tid];
        const RlResetLog& lg = a.out.reset_log;
        const int n_reset_total = reset_masked ? *a.out.n_reset : n_total;
        const float cnt = (float)max(n_reset_total, 1);
        if (n_reset_total == 0) tot = 0.f;
        if (tid < K) { if (lg.episode_sum_mean) lg.episode_sum_mean[tid] = tot / cnt; }
        else if (tid < K + RL_MAX_DONE_TERMS) { if (lg.done_term_count) lg.done_term_count[tid - K] = tot; }
        else if (lg.metric_mean) lg.metric_mean[tid - K - RL_MAX_DONE_TERMS] = tot / cnt;
      }
      if (tid == 0) *a.ticket = 0u;
    }
  }
  RL_STAMP(6);
  if ((ph & RL_PHASE_OBS) && nvalid > 0 && tid == 0) bulk_wait_read0();  // smem must outlive the bulk reads
  RL_STAMP(7);
}

// ---------------------------------------------------------------------------------------------------
// process_action: ActionManager.process_action + JointAction.process_actions [IL]
// ---------------------------------------------------------------------------------------------------
// One CTA = 32 consecutive envs. Phase 1 reads the policy's action rows in the order they lie in memory into shared
// memory; phase 2 walks (column, env) with env fastest, so that every SoA destination (stored action, previous
// action, joint targets) is written as coalesced rows - and any other layout through the same strides.
// The per-column action table (scale, offset, clip, joint id, target kind) comes from a packed device copy with one
// coalesced read: six lane-uniform reads of six different __constant__ arrays are six serialised cold misses, 1 us of a
// 3 us launch (launch probe of round 2: an empty kernel node costs 0.6 us).
constexpr int kPaEnvs = 32;
// table layout, [A] each: scale | offset | clip_lo | clip_hi | (joint id | target kind << 8) as int bits
__global__ void __launch_bounds__(256) process_action_kernel(int N, int A, int has_clip, const float* __restrict__ tab, RlField new_action,
                                                            RlField action, RlField prev_action, RlField target, RlField vel_target,
                                                            unsigned long long* step_counter, int use_pdl) {
  __shared__ float s_act[kPaEnvs * (RL_MAX_JOINTS + 1)];
  __shared__ float s_tab[5 * RL_MAX_JOINTS];
  if (use_pdl) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
  }
  if (step_counter != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *step_counter += 1ull;
  const int env0 = (int)blockIdx.x * kPaEnvs;
  const int ne = min(kPaEnvs, N - env0);
  const int P = A + 1;   // odd-ish pitch: phase 2 reads a column of the tile without bank conflicts for the usual A
  const bool env_major = (new_action.env_stride == 1);
  for (int i = threadIdx.x; i < 5 * A; i += blockDim.x) s_tab[i] = __ldg(tab + i);
  // the stored actions this thread will overwrite in phase 2 are requested NOW, together with the policy's rows: one
  // memory round trip for the launch instead of two dependent ones (kPaEnvs * RL_MAX_JOINTS / 256 = 8 values at most)
  constexpr int kMine = kPaEnvs * RL_MAX_JOINTS / 256;
  float old_a[kMine];
#pragma unroll
  for (int q = 0; q < kMine; ++q) {
    const int i = threadIdx.x + q * 256;
    old_a[q] = 0.f;
    if (i < ne * A && blockDim.x == 256)
      old_a[q] = static_cast<const float*>(action.ptr)[(long long)(env0 + i % ne) * action.env_stride + (long long)(i / ne) * action.comp_stride];
  }
  for (int i = threadIdx.x; i < ne * A; i += blockDim.x) {
    int el, col;
    if (env_major) { el = i % ne; col = i / ne; } else { col = i % A; el = i / A; }
    s_act[el * P + col] = static_cast<const float*>(new_action.ptr)[(long long)(env0 + el) * new_action.env_stride + (long long)col * new_action.comp_stride];
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < kMine; ++q) {
    const int i = threadIdx.x + q * 256;
    if (i >= ne * A) break;
    const int el = i % ne, col = i / ne;
    const long long env = env0 + el;
    const float nv = s_act[el * P + col];
    if (prev_action.ptr)
      static_cast<float*>(prev_action.ptr)[env * prev_action.env_stride + (long long)col * prev_action.comp_stride] = old_a[q];
    static_cast<float*>(action.ptr)[env * action.env_stride + (long long)col * action.comp_stride] = nv;
    const int idk = __float_as_int(s_tab[4 * A + col]);
    const RlField& dst = ((idk >> 8) == RL_ACTION_JOINT_VELOCITY) ? vel_target : target;
    if (dst.ptr) {
      float v = nv * s_tab[col] + s_tab[A + col];
      if (has_clip) v = clampf(v, s_tab[2 * A + col], s_tab[3 * A + col]);
      static_cast<float*>(dst.ptr)[env * dst.env_stride + (long long)(idk & 0xff) * dst.comp_stride] = v;
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Reset events: reset_root_state_uniform (V/mdp/events.py:205-271) + reset_joints_by_scale [IL]. One thread per
// env being reset (they are few); isaaclab.utils.math [IL]: quat_from_euler_xyz, quat_mul, sample_uniform.
// ---------------------------------------------------------------------------------------------------
struct ResetStateArgs {
  int N, slot, has_ids;
  RlResetStateCfg cfg;
  RlField origins, pos, quat, lin, ang, jpos, jvel;
  const uint8_t* terminated;
  const uint8_t* truncated;
  const int32_t* env_ids;
  const int32_t* n_env_ids;
  RlRandom rnd;
  const float* uniforms;   // [12 + 2J][N] or NULL
  const uint8_t* pits;     // [N] is_env_assigned_to_terrain(env, "pits") or NULL
};
__global__ void reset_scene_state_kernel(const ResetStateArgs a) {
  const RlStepSpec& S = c_spec[a.slot];
  const int n = a.has_ids ? *a.n_env_ids : a.N;
  RandState rs;
  rs.seed = a.rnd.seed;
  rs.step = a.rnd.step + (a.rnd.step_counter ? *a.rnd.step_counter : 0ull);
  rs.env_id_offset = a.rnd.env_id_offset;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    long long env = i;
    if (a.has_ids) env = a.env_ids[i];
    else if (!((a.terminated && a.terminated[i]) || (a.truncated && a.truncated[i]))) continue;
    float u[12];
    if (a.uniforms) {
#pragma unroll
      for (int q = 0; q < 12; ++q) u[q] = a.uniforms[(long long)q * a.N + env];
    } else {
#pragma unroll
      for (int blk = 0; blk < 3; ++blk) {
        const uint4 r = rl_philox(rs, env, RL_STREAM_RESET_STATE, (uint32_t)blk);
        u[4 * blk] = u01(r.x); u[4 * blk + 1] = u01(r.y); u[4 * blk + 2] = u01(r.z); u[4 * blk + 3] = u01(r.w);
      }
    }
    const RlResetStateCfg& c = a.cfg;
    const float* org = static_cast<const float*>(a.origins.ptr);
    if (a.pits != nullptr && a.pits[env]) {
      // V/mdp/events.py:237-244: envs assigned to the "pits" sub-terrain get the default root state at their
      // origin, zero velocity, no random perturbation (the joints are still reset by reset_joints_by_scale below)
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const float o = org ? org[env * a.origins.env_stride + (long long)q * a.origins.comp_stride] : 0.f;
        st_f(a.pos, env, q, c.default_root_state[q] + o);
        st_f(a.lin, env, q, 0.f);
        st_f(a.ang, env, q, 0.f);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) st_f(a.quat, env, q, c.default_root_state[3 + q]);
    } else {
    float pose[6], vel[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) {   // sample_uniform [IL]: (hi - lo) * u + lo
      pose[q] = (c.pose_hi[q] - c.pose_lo[q]) * u[q] + c.pose_lo[q];
      vel[q] = (c.vel_hi[q] - c.vel_lo[q]) * u[6 + q] + c.vel_lo[q];
    }
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      const float o = org ? org[env * a.origins.env_stride + (long long)q * a.origins.comp_stride] : 0.f;
      st_f(a.pos, env, q, (c.default_root_state[q] + o) + pose[q]);
    }
    // quat_from_euler_xyz [IL] (roll, pitch, yaw)
    const float cr = rl_cosf(pose[3] * 0.5f), sr = rl_sinf(pose[3] * 0.5f);
    const float cp = rl_cosf(pose[4] * 0.5f), sp = rl_sinf(pose[4] * 0.5f);
    const float cy = rl_cosf(pose[5] * 0.5f), sy = rl_sinf(pose[5] * 0.5f);
    const float dw = (cy * cr) * cp + (sy * sr) * sp;
    const float dx = (cy * sr) * cp - (sy * cr) * sp;
    const float dy = (cy * cr) * sp + (sy * sr) * cp;
    const float dz = (sy * cr) * cp - (cy * sr) * sp;
    // quat_mul(default_quat, delta) [IL]
    const float w1 = c.default_root_state[3], x1 = c.default_root_state[4], y1 = c.default_root_state[5], z1 = c.default_root_state[6];
    const float ww = (z1 + x1) * (dx + dy), yy = (w1 - y1) * (dw + dz), zz = (w1 + y1) * (dw - dz);
    const float xx = ww + yy + zz;
    const float qq = 0.5f * (xx + (z1 - x1) * (dx - dy));
    st_f(a.quat, env, 0, qq - ww + (z1 - y1) * (dy - dz));
    st_f(a.quat, env, 1, qq - xx + (x1 + w1) * (dx + dw));
    st_f(a.quat, env, 2, qq - yy + (w1 - x1) * (dy + dz));
    st_f(a.quat, env, 3, qq - zz + (z1 + y1) * (dw - dx));
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      st_f(a.lin, env, q, c.default_root_state[7 + q] + vel[q]);
      st_f(a.ang, env, q, c.default_root_state[10 + q] + vel[3 + q]);
    }
    }
    // reset_joints_by_scale [IL]
    const int J = S.num_joints;
    for (int j = 0; j < J; ++j) {
      float up, uv;
      if (a.uniforms) {
        up = a.uniforms[(long long)(12 + j) * a.N + env];
        uv = a.uniforms[(long long)(12 + J + j) * a.N + env];
      } else {
        const uint4 r = rl_philox(rs, env, RL_STREAM_RESET_JOINTS, (uint32_t)(j >> 1));
        up = u01((j & 1) ? r.z : r.x); uv = u01((j & 1) ? r.w : r.y);
      }
      float qp = S.default_joint_pos[j] * ((c.joint_pos_scale_hi - c.joint_pos_scale_lo) * up + c.joint_pos_scale_lo);
      float qv = S.default_joint_vel[j] * ((c.joint_vel_scale_hi - c.joint_vel_scale_lo) * uv + c.joint_vel_scale_lo);
      qp = clampf(qp, S.soft_pos_limit_lo[j], S.soft_pos_limit_hi[j]);
      qv = clampf(qv, -S.soft_vel_limit[j], S.soft_vel_limit[j]);
      if (a.jpos.ptr) st_f(a.jpos, env, j, qp);
      if (a.jvel.ptr) st_f(a.jvel, env, j, qv);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// ContactSensor update [IL]: history roll (or ring-slot write) + air / contact timers. One thread per
// (env, history element) for the history, one per (env, timer body) for the timers.
// ---------------------------------------------------------------------------------------------------
struct SensorArgs {
  int N, B, T, Bt, ring_slot;
  float dt, thr;
  RlField net, hist, cair, lair, ccon, lcon;
  int t2h[RL_MAX_TIME_BODIES];
};
__global__ void contact_sensor_kernel(const SensorArgs a) {
  // Work items: N * B*3 history elements, then N * Bt timer bodies. Consecutive threads walk the contiguous axis of
  // the tensor they write (components for AoS rows, envs for SoA) so that either layout coalesces.
  const int n_hist = a.N * a.B * 3, total = n_hist + a.N * a.Bt;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    if (i < n_hist) {
      int env, item;
      if (a.hist.comp_stride == 1) { item = i % (a.B * 3); env = i / (a.B * 3); } else { env = i % a.N; item = i / a.N; }
      const float v = static_cast<const float*>(a.net.ptr)[(long long)env * a.net.env_stride + (long long)item * a.net.comp_stride];
      float* h = static_cast<float*>(a.hist.ptr) + (long long)env * a.hist.env_stride;
      const long long cs = a.hist.comp_stride;
      if (a.ring_slot >= 0) {
        h[(long long)(a.ring_slot * a.B * 3 + item) * cs] = v;
      } else {
        // newest first: slot 0 <- net, slot t <- old slot t-1. All loads first, then all stores (hist_len <= 8):
        // one memory round trip instead of a load -> store chain per slot
        float old[8];
#pragma unroll
        for (int t = 0; t < 7; ++t)
          if (t < a.T - 1) old[t] = h[(long long)(t * a.B * 3 + item) * cs];
        h[(long long)item * cs] = v;
#pragma unroll
        for (int t = 1; t < 8; ++t)
          if (t < a.T) h[(long long)(t * a.B * 3 + item) * cs] = old[t - 1];
      }
    } else {
      const int j = i - n_hist;
      int env, f;
      if (a.cair.comp_stride == 1 && a.Bt > 1) { f = j % a.Bt; env = j / a.Bt; } else { env = j % a.N; f = j / a.N; }
      const int b = a.t2h[f];
      const float* net = static_cast<const float*>(a.net.ptr) + (long long)env * a.net.env_stride;
      const float fx = net[(long long)(3 * b) * a.net.comp_stride], fy = net[(long long)(3 * b + 1) * a.net.comp_stride],
                  fz = net[(long long)(3 * b + 2) * a.net.comp_stride];
      const bool contact = sqrtf((fx * fx + fy * fy) + fz * fz) > a.thr;
      float* ca = static_cast<float*>(a.cair.ptr) + (long long)env * a.cair.env_stride + (long long)f * a.cair.comp_stride;
      float* la = static_cast<float*>(a.lair.ptr) + (long long)env * a.lair.env_stride + (long long)f * a.lair.comp_stride;
      float* cc = static_cast<float*>(a.ccon.ptr) + (long long)env * a.ccon.env_stride + (long long)f * a.ccon.comp_stride;
      float* lc = static_cast<float*>(a.lcon.ptr) + (long long)env * a.lcon.env_stride + (long long)f * a.lcon.comp_stride;
      const float cur_air = *ca, cur_con = *cc;
      const bool first_contact = (cur_air > 0.f) && contact, first_detach = (cur_con > 0.f) && !contact;
      if (first_contact) *la = cur_air + a.dt;
      *ca = contact ? 0.f : cur_air + a.dt;
      if (first_detach) *lc = cur_con + a.dt;
      *cc = contact ? cur_con + a.dt : 0.f;
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------------
}  // namespace

// struct RlCtx: csrc/mdp_ctx.h (shared with mdp_step_v2.cu)

int rl_ctx_device_of(const RlCtx* ctx) { return ctx->device; }
const RlStepSpec* rl_ctx_spec_of(const RlCtx* ctx) { return &ctx->spec; }

namespace {


bool to_fd(const RlField& f, FieldD* out) {
  if (f.env_stride > 0x7fffffffLL || f.comp_stride > 0x7fffffffLL || f.env_stride < 0 || f.comp_stride < 0) return false;
  out->ptr = f.ptr; out->es = (int)f.env_stride; out->cs = (int)f.comp_stride;
  return true;
}
bool vec4_ok(const FieldD& d, int ncomp) {
  return d.ptr != nullptr && d.es == 1 && (ncomp == 1 || (d.cs % 4) == 0) && (reinterpret_cast<uintptr_t>(d.ptr) & 15u) == 0;
}

// Field descriptors + masks of one launch. `state` may be NULL (reset-only launches).
int fill_args(RlCtx* ctx, KArgs& a, int64_t num_envs, const RlStateView* st, const RlMdpState* mdp, const RlStepOut* out,
              const RlRandom* rnd, uint32_t ph, int mode) {
  const RlStepSpec& s = ctx->spec;
  memset(&a, 0, sizeof(a));
  a.N = (int)num_envs; a.slot = ctx->slot; a.phases = ph;
  a.L = ctx->L; a.sched = ctx->sched_dev;
  {
    const Schedule& sc = ctx->sched;
    for (int k = 0; k < s.num_reward_terms; ++k) {
      a.rw_weight[k] = s.rewards[k].weight;
      if (sc.late[k]) a.rw_late |= 1ull << k;
      if (s.rewards[k].type == RL_REW_IS_TERMINATED) a.rw_isterm |= 1ull << k;
      if (s.rewards[k].weight == 0.f) a.rw_zero |= 1ull << k;
    }
  }
  a.cj = ctx->cj_dev;
  a.ticket = ctx->ticket; a.cta_mask = ctx->cta_mask; a.log_partials = ctx->log_partials; a.use_pdl = ctx->use_pdl;
  a.dbg = ctx->dbg;
  if (out) a.out = *out;
  if (rnd) a.rnd = *rnd;
  bool ok = true;
  RlField none{nullptr, 0, 0};
  auto S = [&](const RlField RlStateView::*m) -> const RlField& { return st ? st->*m : none; };
  ok &= to_fd(S(&RlStateView::root_pos_w), &a.in[IF_ROOT_POS]); ok &= to_fd(S(&RlStateView::root_quat_w), &a.in[IF_QUAT]);
  ok &= to_fd(S(&RlStateView::root_lin_vel_w), &a.in[IF_LIN_VEL]); ok &= to_fd(S(&RlStateView::root_ang_vel_w), &a.in[IF_ANG_VEL]);
  ok &= to_fd(S(&RlStateView::joint_pos), &a.in[IF_JPOS]); ok &= to_fd(S(&RlStateView::joint_vel), &a.in[IF_JVEL]);
  ok &= to_fd(S(&RlStateView::joint_acc), &a.in[IF_JACC]); ok &= to_fd(S(&RlStateView::applied_torque), &a.in[IF_JTAU]);
  ok &= to_fd(S(&RlStateView::current_air_time), &a.in[IF_CAIR]); ok &= to_fd(S(&RlStateView::last_air_time), &a.in[IF_LAIR]);
  ok &= to_fd(S(&RlStateView::current_contact_time), &a.in[IF_CCON]); ok &= to_fd(S(&RlStateView::last_contact_time), &a.in[IF_LCON]);
  ok &= to_fd(S(&RlStateView::body_pos_w), &a.in[IF_BPOS]); ok &= to_fd(S(&RlStateView::body_lin_vel_w), &a.in[IF_BVEL]);
  ok &= to_fd(S(&RlStateView::ray_sensor_pos_z), &a.in[IF_RAYPOS]);
  ok &= to_fd(S(&RlStateView::net_forces_w_history), &a.hist); ok &= to_fd(S(&RlStateView::ray_hits_z), &a.rays);
  ok &= to_fd(mdp->command, &a.in[IF_CMD]); ok &= to_fd(mdp->heading_target, &a.in[IF_HEAD]);
  ok &= to_fd(mdp->time_left, &a.in[IF_TLEFT]); ok &= to_fd(mdp->metric_error_vel_xy, &a.in[IF_MXY]);
  ok &= to_fd(mdp->metric_error_vel_yaw, &a.in[IF_MYAW]); ok &= to_fd(mdp->episode_length, &a.in[IF_EPLEN]);
  ok &= to_fd(mdp->episode_sums, &a.in[IF_SUMS]);
  ok &= to_fd(mdp->action, &a.in[IF_ACT]); ok &= to_fd(mdp->prev_action, &a.in[IF_PACT]);
  ok &= to_fd(mdp->is_heading_env, &a.is_heading); ok &= to_fd(mdp->is_standing_env, &a.is_standing);
  if (!ok) return fail(RL_EINVAL, "field strides must be non-negative and below 2^31 elements%s", "");
  a.in[IF_CMDU] = FieldD{a.rnd.cmd_uniforms, 1, (int)num_envs};
  const bool need_hist = (mode == 1) || (ph & (RL_PHASE_DONES | RL_PHASE_REWARDS));
  uint32_t m = (1u << IF_ROOT_POS) | (1u << IF_QUAT) | (1u << IF_LIN_VEL) | (1u << IF_ANG_VEL) | (1u << IF_JPOS) |
               (1u << IF_JVEL) | (1u << IF_CMD) | (1u << IF_EPLEN) | (1u << IF_ACT);
  if (need_hist)
    m |= (1u << IF_PACT) | (1u << IF_JACC) | (1u << IF_JTAU) | (1u << IF_CAIR) | (1u << IF_LAIR) | (1u << IF_CCON) | (1u << IF_LCON) |
         (1u << IF_BPOS) | (1u << IF_BVEL);
  if (mode == 0 && (ph & RL_PHASE_REWARDS)) m |= 1u << IF_SUMS;
  if (mode == 0 && (ph & RL_PHASE_COMMAND)) m |= (1u << IF_HEAD) | (1u << IF_TLEFT) | (1u << IF_MXY) | (1u << IF_MYAW) | (1u << IF_CMDU);
  // (IF_PACT: the RESET launch stores the previous-action rows of every tile that resets anything - the live lanes must
  //  carry their own values, not whatever the record held. Found in round 2: at more than one wave of tiles the general
  //  kernel wrote stale shared memory into prev_action of envs that were NOT reset.)
  if (mode == 0 && (ph & RL_PHASE_RESET)) m |= (1u << IF_SUMS) | (1u << IF_MXY) | (1u << IF_MYAW) | (1u << IF_HEAD) | (1u << IF_CMDU) | (1u << IF_PACT);
  if (mode == 0 && (ph & RL_PHASE_OBS) && s.num_rays > 0) m |= 1u << IF_RAYPOS;
  uint32_t v4 = 0;
  for (int f = 0; f < IF_COUNT; ++f) {
    if (a.in[f].ptr == nullptr) m &= ~(1u << f);
    else if (vec4_ok(a.in[f], in_field_ncomp(s, f))) v4 |= 1u << f;
  }
  a.in_mask = m; a.in_vec4 = v4;
  for (int f = 0; f < IF_COUNT; ++f) a.in[f].meta = in_field_ncomp(s, f) | (in_field_word(s, f) << 16);
  // outputs
  if (mode == 0) {
    a.outf[OF_REWARD] = FieldD{a.out.reward, 1, 0};
    a.outf[OF_EPLEN] = a.in[IF_EPLEN]; a.outf[OF_SUMS] = a.in[IF_SUMS];
    FieldD sr; if (!to_fd(a.out.step_reward, &sr)) return fail(RL_EINVAL, "bad step_reward strides%s", "");
    a.outf[OF_STEPR] = sr;
    a.outf[OF_CMD] = a.in[IF_CMD]; a.outf[OF_HEAD] = a.in[IF_HEAD]; a.outf[OF_TLEFT] = a.in[IF_TLEFT];
    a.outf[OF_MXY] = a.in[IF_MXY]; a.outf[OF_MYAW] = a.in[IF_MYAW];
    a.outf[OF_ACT] = a.in[IF_ACT]; a.outf[OF_PACT] = a.in[IF_PACT];
    uint32_t om = 0;
    if (ph & RL_PHASE_DONES) om |= 1u << OF_EPLEN;
    if (ph & RL_PHASE_REWARDS) om |= (1u << OF_REWARD) | (1u << OF_SUMS) | (1u << OF_STEPR);
    if (ph & (RL_PHASE_COMMAND | RL_PHASE_RESET)) om |= (1u << OF_CMD) | (1u << OF_HEAD) | (1u << OF_TLEFT) | (1u << OF_MXY) | (1u << OF_MYAW);
    if (ph & RL_PHASE_RESET) om |= (1u << OF_SUMS) | (1u << OF_EPLEN) | (1u << OF_ACT) | (1u << OF_PACT);
    const int oc[OF_COUNT] = {1, 1, s.num_reward_terms, s.num_reward_terms, 3, 1, 1, 1, 1, s.action.n_actions, s.action.n_actions};
    uint32_t ov4 = 0;
    for (int f = 0; f < OF_COUNT; ++f) {
      if (a.outf[f].ptr == nullptr) om &= ~(1u << f);
      else if (vec4_ok(a.outf[f], oc[f])) ov4 |= 1u << f;
    }
    a.out_mask = om; a.out_vec4 = ov4;
    for (int f = 0; f < OF_COUNT; ++f) a.outf[f].meta = out_field_ncomp(s, f) | (out_field_word(ctx->L, f) << 16);
  }
  return RL_OK;
}

int validate_spec(const RlStepSpec* s) {
  if (s->abi_version != RL_ABI_VERSION) return fail(RL_EINVAL, "spec.abi_version %s%lld != library %lld", "", s->abi_version, RL_ABI_VERSION);
  if (s->num_joints < 1 || s->num_joints > RL_MAX_JOINTS) return fail(RL_EINVAL, "num_joints out of range%s (%lld)", "", s->num_joints);
  if (s->num_hist_bodies < 0 || s->num_hist_bodies > RL_MAX_BODIES) return fail(RL_EINVAL, "num_hist_bodies out of range%s (%lld)", "", s->num_hist_bodies);
  if (s->hist_len < 0 || s->hist_len > 8) return fail(RL_EINVAL, "hist_len out of range%s (%lld)", "", s->hist_len);
  if (s->num_time_bodies < 0 || s->num_time_bodies > RL_MAX_TIME_BODIES) return fail(RL_EINVAL, "num_time_bodies out of range%s (%lld)", "", s->num_time_bodies);
  if (s->num_asset_bodies < 0 || s->num_asset_bodies > RL_MAX_ASSET_BODIES) return fail(RL_EINVAL, "num_asset_bodies out of range%s (%lld)", "", s->num_asset_bodies);
  if (s->num_rays < 0 || s->num_rays > 4096) return fail(RL_EINVAL, "num_rays out of range%s (%lld)", "", s->num_rays);
  if (s->num_reward_terms < 0 || s->num_reward_terms > RL_MAX_REWARD_TERMS) return fail(RL_EINVAL, "num_reward_terms out of range%s (%lld)", "", s->num_reward_terms);
  if (s->num_done_terms < 0 || s->num_done_terms > RL_MAX_DONE_TERMS) return fail(RL_EINVAL, "num_done_terms out of range%s (%lld)", "", s->num_done_terms);
  if (s->action.n_actions < 0 || s->action.n_actions > RL_MAX_JOINTS) return fail(RL_EINVAL, "n_actions out of range%s (%lld)", "", s->action.n_actions);
  if (!(s->step_dt > 0.f)) return fail(RL_EINVAL, "step_dt must be positive%s", "");
  for (int a = 0; a < s->action.n_actions; ++a)
    if (s->action.joint_ids[a] >= s->num_joints) return fail(RL_EINVAL, "action.joint_ids[%s%lld] out of range", "", a);
  for (int k = 0; k < s->num_reward_terms; ++k) {
    const RlRewardTerm& t = s->rewards[k];
    if (t.type <= RL_REW_NONE || t.type >= RL_REW_TYPE_COUNT) return fail(RL_EINVAL, "reward term %s%lld: unknown type %lld", "", k, t.type);
    if (t.n_idx < 0 || t.n_idx > RL_MAX_IDX) return fail(RL_EINVAL, "reward term %s%lld: n_idx out of range", "", k);
    if (t.type == RL_REW_FEET_AIR_TIME_VARIANCE && t.n_idx < 2) return fail(RL_EINVAL, "reward term %s%lld: variance needs >= 2 feet", "", k);
    if (t.type == RL_REW_FEET_GAIT && t.n_idx != 4) return fail(RL_EINVAL, "reward term %s%lld: feet_gait needs two synced pairs", "", k);
  }
  for (int g = 0; g < RL_NUM_OBS_GROUPS; ++g) {
    const RlObsGroup& G = s->obs[g];
    if (G.n_terms < 0 || G.n_terms > RL_MAX_OBS_TERMS) return fail(RL_EINVAL, "obs group %s%lld: n_terms out of range", "", g);
    int dim = 0;
    for (int t = 0; t < G.n_terms; ++t) {
      const RlObsTerm& o = G.terms[t];
      if (o.type <= RL_OBS_NONE || o.type >= RL_OBS_TYPE_COUNT) return fail(RL_EINVAL, "obs group %s%lld term %lld: unknown type", "", g, t);
      if (o.type == RL_OBS_HEIGHT_SCAN && o.dim != s->num_rays) return fail(RL_EINVAL, "obs group %s%lld: height_scan dim != num_rays", "", g);
      if ((o.type == RL_OBS_JOINT_POS_REL || o.type == RL_OBS_JOINT_VEL_REL || o.type == RL_OBS_JOINT_POS_REL_WITHOUT_WHEEL) && o.dim > RL_MAX_JOINTS)
        return fail(RL_EINVAL, "obs group %s%lld: joint term wider than RL_MAX_JOINTS", "", g);
      dim += o.dim;
    }
    if (dim != G.dim) return fail(RL_EINVAL, "obs group %s%lld: dim %lld != sum of term dims", "", g, G.dim);
  }
  return RL_OK;
}

template <class P, int NW, int MODE, bool DBG>
int launch_step_variant(RlCtx* ctx, const KArgs& a_in, int n_items, cudaStream_t st) {
  const size_t smem = (size_t)ctx->L.total_words * 4;
  static thread_local int configured_device = -1;
  static thread_local size_t configured_smem = 0;
  if (configured_device != ctx->device || configured_smem < smem) {
    CUDA_TRY(cudaFuncSetAttribute(mdp_step_kernel<P, NW, MODE, DBG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured_device = ctx->device; configured_smem = smem;
  }
  const int vgrid = (n_items + kE - 1) / kE;
  if (vgrid <= 0) return RL_OK;
  KArgs a = a_in;
  a.vgrid = vgrid;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(vgrid); cfg.blockDim = dim3(NW * 32); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = a.use_pdl ? 1 : 0;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, mdp_step_kernel<P, NW, MODE, DBG>, a));
  return RL_OK;
}
// the clock-stamp variant (rl_ctx_set_debug_buffer) is a separate instantiation: the production kernel carries
// no trace of it
template <class P, int NW, int MODE>
int launch_step(RlCtx* ctx, const KArgs& a, int n_items, cudaStream_t st) {
  if constexpr (MODE == 0) {
    if (a.dbg != nullptr) return launch_step_variant<P, NW, MODE, true>(ctx, a, n_items, st);
  }
  return launch_step_variant<P, NW, MODE, false>(ctx, a, n_items, st);
}

// warps per CTA compiled for the generic kernel / for every baked spec
#define RL_DYN_CONFIGS(X) X(4) X(8) X(16)
#define RL_STATIC_CONFIGS(X) X(16)   /* baked specs at 4 / 8 warps per tile run the generic kernel */

template <class P, int MODE>
int dispatch_config(RlCtx* ctx, const KArgs& a, int n_items, cudaStream_t st, bool* found) {
  *found = true;
  if constexpr (P::kStatic) {
#define RL_CASE(W_) if (ctx->NW == (W_)) return launch_step<P, W_, MODE>(ctx, a, n_items, st);
    RL_STATIC_CONFIGS(RL_CASE)
#undef RL_CASE
  } else {
#define RL_CASE(W_) if (ctx->NW == (W_)) return launch_step<P, W_, MODE>(ctx, a, n_items, st);
    RL_DYN_CONFIGS(RL_CASE)
#undef RL_CASE
  }
  *found = false;
  return RL_OK;
}

template <int MODE>
int dispatch_step(RlCtx* ctx, const KArgs& a, int n_items, cudaStream_t st) {
  bool found = false;
  if (MODE == 0 && ctx->baked >= 0) {
    int idx = 0, rc = RL_OK;
#define RL_TRY_BAKED(B) if (idx++ == ctx->baked) rc = dispatch_config<StaticPolicy<baked::B>, 0>(ctx, a, n_items, st, &found);
    RL_BAKED_LIST(RL_TRY_BAKED)
#undef RL_TRY_BAKED
    if (found) return rc;
  }
  // generic kernel (compiled for 4, 8 and 16 warps). The single-term mode ignores the schedule, so any
  // configured warp count maps to a compiled one; the step mode needs the schedule's warp count exactly.
  RlCtx tmp = *ctx;
  if (MODE == 1) tmp.NW = tmp.NW >= 16 ? 16 : (tmp.NW >= 8 ? 8 : 4);
  int rc = dispatch_config<DynPolicy, MODE>(&tmp, a, n_items, st, &found);
  if (!found) return fail(RL_EINVAL, "the generic kernel is compiled for 4, 8 or 16 warps per CTA, not %s%lld", "", ctx->NW);
  return rc;
}

int ensure_scratch(RlCtx* ctx, int grid) {
  if (grid <= ctx->cta_mask_cap) return RL_OK;
  if (ctx->cta_mask) CUDA_TRY(cudaFree(ctx->cta_mask));
  if (ctx->log_partials) CUDA_TRY(cudaFree(ctx->log_partials));
  ctx->cta_mask = nullptr;
  ctx->log_partials = nullptr;
  const int cap = grid * 2 + 64;
  CUDA_TRY(cudaMalloc(&ctx->cta_mask, sizeof(uint32_t) * cap));
  CUDA_TRY(cudaMemset(ctx->cta_mask, 0, sizeof(uint32_t) * cap));
  CUDA_TRY(cudaMalloc(&ctx->log_partials, sizeof(float) * (size_t)cap * RL_LOG_STRIDE));
  CUDA_TRY(cudaMemset(ctx->log_partials, 0, sizeof(float) * (size_t)cap * RL_LOG_STRIDE));
  ctx->cta_mask_cap = cap;
  return RL_OK;
}

bool g_slots[16][RL_SPEC_SLOTS];

}  // namespace

extern "C" {

int rl_abi_version(void) { return RL_ABI_VERSION; }
const char* rl_last_error(void) { return g_err; }

int64_t rl_struct_sizeof(const char* name) {
  if (!name) return -1;
#define RL_SZ(T) if (strcmp(name, #T) == 0) return (int64_t)sizeof(T)
  RL_SZ(RlRewardTerm); RL_SZ(RlObsTerm); RL_SZ(RlObsGroup); RL_SZ(RlDoneTerm); RL_SZ(RlCommandCfg);
  RL_SZ(RlActionCfg); RL_SZ(RlStepSpec); RL_SZ(RlField); RL_SZ(RlStateView); RL_SZ(RlMdpState);
  RL_SZ(RlStepOut); RL_SZ(RlRandom); RL_SZ(RlResetLog); RL_SZ(RlResetStateCfg);
  RL_SZ(RlActuatorCfg); RL_SZ(RlTerrainGrid); RL_SZ(RlHeightField); RL_SZ(RlIntervalEventCfg);
#undef RL_SZ
  return -1;
}

int64_t rl_tile_record_bytes(const RlStepSpec* spec) {
  if (!spec || validate_spec(spec) != RL_OK) return -1;
  return (int64_t)make_layout(*spec).total_words * 4;
}

int rl_ctx_create(const RlStepSpec* spec, int device, RlCtx** out) {
  if (!spec || !out) return fail(RL_EINVAL, "rl_ctx_create: null argument%s", "");
  *out = nullptr;
  int rc = validate_spec(spec);
  if (rc != RL_OK) return rc;
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev || device >= 16) return fail(RL_EINVAL, "rl_ctx_create: bad device%s %lld", "", device);
  DeviceGuard guard(device);
  if (!guard.ok) return fail(RL_ECUDA, "rl_ctx_create: cudaSetDevice failed%s", "");
  int slot = -1;
  for (int i = 0; i < RL_SPEC_SLOTS; ++i) if (!g_slots[device][i]) { slot = i; break; }
  if (slot < 0) return fail(RL_ENOMEM, "rl_ctx_create: all %s%lld constant-memory spec slots of this device are in use", "", RL_SPEC_SLOTS);
  RlCtx* ctx = new (std::nothrow) RlCtx();
  if (!ctx) return fail(RL_ENOMEM, "rl_ctx_create: out of host memory%s", "");
  memset(ctx, 0, sizeof(*ctx));
  ctx->device = device;
  ctx->slot = slot;
  ctx->spec = *spec;
  ctx->NW = 16;
  ctx->L = make_layout(ctx->spec);
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  ctx->sm_count = prop.multiProcessorCount;
  ctx->smem_optin = (size_t)prop.sharedMemPerBlockOptin;
  if ((size_t)ctx->L.total_words * 4 > (size_t)prop.sharedMemPerBlockOptin) {
    delete ctx;
    return fail(RL_EUNSUPPORTED, "the tile of %s%lld envs needs %lld bytes of shared memory", "", kE, (long long)make_layout(*spec).total_words * 4);
  }
  CUDA_TRY(cudaMalloc(&ctx->sched_dev, sizeof(Schedule)));
  ctx->sched = make_schedule(ctx->spec, ctx->NW);
  CUDA_TRY(cudaMemcpy(ctx->sched_dev, &ctx->sched, sizeof(Schedule), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpyToSymbol(c_spec, spec, sizeof(RlStepSpec), sizeof(RlStepSpec) * slot));
  CUDA_TRY(cudaMalloc(&ctx->ticket, sizeof(unsigned int)));
  CUDA_TRY(cudaMemset(ctx->ticket, 0, sizeof(unsigned int)));
  CUDA_TRY(cudaMalloc(&ctx->adhoc_dev, sizeof(RlRewardTerm) * 64));
  {
    const int J = spec->num_joints;
    float cj[5 * RL_MAX_JOINTS];
    for (int j = 0; j < J; ++j) {
      cj[0 * J + j] = spec->default_joint_pos[j]; cj[1 * J + j] = spec->default_joint_vel[j];
      cj[2 * J + j] = spec->soft_pos_limit_lo[j]; cj[3 * J + j] = spec->soft_pos_limit_hi[j];
      cj[4 * J + j] = spec->soft_vel_limit[j];
    }
    CUDA_TRY(cudaMalloc(&ctx->cj_dev, sizeof(float) * 5 * RL_MAX_JOINTS));
    CUDA_TRY(cudaMemcpy(ctx->cj_dev, cj, sizeof(float) * 5 * J, cudaMemcpyHostToDevice));
  }
  {
    const RlActionCfg& ac = spec->action;
    const int A = ac.n_actions;
    float tab[5 * RL_MAX_JOINTS];
    for (int c = 0; c < A; ++c) {
      tab[c] = ac.scale[c]; tab[A + c] = ac.offset[c]; tab[2 * A + c] = ac.clip_lo[c]; tab[3 * A + c] = ac.clip_hi[c];
      const int idk = (int)ac.joint_ids[c] | ((int)ac.target_kind[c] << 8);
      memcpy(&tab[4 * A + c], &idk, sizeof(int));
    }
    CUDA_TRY(cudaMalloc(&ctx->action_tab_dev, sizeof(float) * 5 * RL_MAX_JOINTS));
    CUDA_TRY(cudaMemcpy(ctx->action_tab_dev, tab, sizeof(float) * 5 * (A > 0 ? A : 1), cudaMemcpyHostToDevice));
  }
  rc = ensure_scratch(ctx, 4096);
  if (rc != RL_OK) return rc;
  ctx->baked = -1;
  {
    int idx = 0;
#define RL_MATCH_BAKED(B) if (ctx->baked < 0 && memcmp(spec, &baked::B::spec, sizeof(RlStepSpec)) == 0) ctx->baked = idx; ++idx;
    RL_BAKED_LIST(RL_MATCH_BAKED)
#undef RL_MATCH_BAKED
    // RL_MDPSTEP_GENERIC=1 forces the generic (table-driven) kernel: A/B measurements and tests of that path
    const char* force_generic = getenv("RL_MDPSTEP_GENERIC");
    if (force_generic && force_generic[0] == '1') ctx->baked = -1;
  }
  g_slots[device][slot] = true;
  // the cluster kernels of the two env-step launches (csrc/mdp_step_v2.cu) for the build-time specialised specs
  rc = rl_v2_create(ctx);
  if (rc != RL_OK) { rl_ctx_destroy(ctx); return rc; }
  *out = ctx;
  return RL_OK;
}

void rl_ctx_destroy(RlCtx* ctx) {
  if (!ctx) return;
  DeviceGuard guard(ctx->device);
  rl_v2_destroy(ctx);
  if (ctx->ticket) cudaFree(ctx->ticket);
  if (ctx->cta_mask) cudaFree(ctx->cta_mask);
  if (ctx->log_partials) cudaFree(ctx->log_partials);
  if (ctx->adhoc_dev) cudaFree(ctx->adhoc_dev);
  if (ctx->cj_dev) cudaFree(ctx->cj_dev);
  if (ctx->action_tab_dev) cudaFree(ctx->action_tab_dev);
  if (ctx->sched_dev) cudaFree(ctx->sched_dev);
  g_slots[ctx->device][ctx->slot] = false;
  delete ctx;
}

int rl_ctx_set_launch_config(RlCtx* ctx, int envs_per_cta, int warps_per_cta) {
  if (!ctx) return fail(RL_EINVAL, "null ctx%s", "");
  if (envs_per_cta != 0 && envs_per_cta != kE)
    return fail(RL_EINVAL, "envs_per_cta must be %s%lld: a tile is one lane per env (two tiles per CTA measured slower in round 1 and were removed)", "", kE);
  const int nw = warps_per_cta > 0 ? warps_per_cta : 16;
  if (nw != 4 && nw != 8 && nw != 16) return fail(RL_EINVAL, "warps_per_cta must be 4, 8 or 16%s, got %lld", "", nw);
  DeviceGuard guard(ctx->device);
  ctx->sched = make_schedule(ctx->spec, nw);
  CUDA_TRY(cudaMemcpy(ctx->sched_dev, &ctx->sched, sizeof(Schedule), cudaMemcpyHostToDevice));  // synchronous: not for hot loops
  ctx->NW = nw;
  return RL_OK;
}

int rl_ctx_get_launch_config(const RlCtx* ctx, int* envs_per_cta, int* warps_per_tile) {
  if (!ctx || !envs_per_cta || !warps_per_tile) return fail(RL_EINVAL, "null argument%s", "");
  *envs_per_cta = kE;
  *warps_per_tile = ctx->NW;
  return RL_OK;
}

int rl_ctx_get_cluster_config(const RlCtx* ctx, int64_t num_envs, int32_t* cluster_size, int32_t* tiles_per_cta, int32_t* warps_per_cta,
                              int64_t* launches) {
  if (!ctx) return fail(RL_EINVAL, "null ctx%s", "");
  int c = 0, g = 0, w = 0;
  long long n = 0;
  rl_v2_config_for(ctx, num_envs, &c, &g, &w, &n);
  if (cluster_size) *cluster_size = c;
  if (tiles_per_cta) *tiles_per_cta = g;
  if (warps_per_cta) *warps_per_cta = w;
  if (launches) *launches = n;
  return RL_OK;
}

int rl_ctx_get_schedule(RlCtx* ctx, int32_t* out, int32_t* n_tasks) {
  if (!ctx || !out || !n_tasks) return fail(RL_EINVAL, "null argument%s", "");
  const Schedule& sc = ctx->sched;
  *n_tasks = sc.n;
  for (int i = 0; i < sc.n; ++i) {
    const Task& t = sc.t[i];
    const int32_t row[8] = {t.kind, t.a, t.b, t.owner, t.lo, t.hi, t.col0, t.pad};
    for (int q = 0; q < 8; ++q) out[i * 8 + q] = row[q];
  }
  return RL_OK;
}

int rl_ctx_set_debug_buffer(RlCtx* ctx, void* device_i64_buffer) {
  if (!ctx) return fail(RL_EINVAL, "null ctx%s", "");
  ctx->dbg = static_cast<long long*>(device_i64_buffer);
  return RL_OK;
}

int rl_ctx_set_pdl(RlCtx* ctx, int enabled) {
  if (!ctx) return fail(RL_EINVAL, "null ctx%s", "");
  ctx->use_pdl = enabled ? 1 : 0;
  return RL_OK;
}

int rl_reset_scene_state(RlCtx* ctx, int64_t num_envs, const RlResetStateCfg* cfg, const RlField* env_origins,
                         const RlStateView* state, const uint8_t* terminated, const uint8_t* truncated,
                         const int32_t* env_ids, const int32_t* n_env_ids, const RlRandom* rnd,
                         const float* uniforms, const uint8_t* assigned_to_pits, void* stream) {
  if (!ctx || !cfg || !state || !rnd) return fail(RL_EINVAL, "rl_reset_scene_state: null argument%s", "");
  if (num_envs <= 0) return RL_OK;
  if (!state->root_pos_w.ptr || !state->root_quat_w.ptr || !state->root_lin_vel_w.ptr || !state->root_ang_vel_w.ptr)
    return fail(RL_EINVAL, "rl_reset_scene_state: the four root state fields are required%s", "");
  if (env_ids && !n_env_ids) return fail(RL_EINVAL, "rl_reset_scene_state: env_ids needs n_env_ids%s", "");
  if (!env_ids && !terminated && !truncated) return fail(RL_EINVAL, "rl_reset_scene_state: env_ids or the done masks are required%s", "");
  ResetStateArgs a;
  memset(&a, 0, sizeof(a));
  a.N = (int)num_envs; a.slot = ctx->slot; a.has_ids = env_ids != nullptr;
  a.cfg = *cfg;
  if (env_origins) a.origins = *env_origins;
  a.pos = state->root_pos_w; a.quat = state->root_quat_w; a.lin = state->root_lin_vel_w; a.ang = state->root_ang_vel_w;
  a.jpos = state->joint_pos; a.jvel = state->joint_vel;
  a.terminated = terminated; a.truncated = truncated; a.env_ids = env_ids; a.n_env_ids = n_env_ids;
  a.rnd = *rnd; a.uniforms = uniforms; a.pits = assigned_to_pits;
  DeviceGuard guard(ctx->device);
  const int threads = 128;
  const int blocks = (int)((num_envs + threads - 1) / threads);
  reset_scene_state_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  return RL_OK;
}

int rl_contact_sensor_update(RlCtx* ctx, int64_t num_envs, const RlField* net_forces_w, const RlStateView* state,
                             const int32_t* time_body_to_hist, float dt, float force_threshold, int32_t ring_slot,
                             void* stream) {
  if (!ctx || !net_forces_w || !state) return fail(RL_EINVAL, "rl_contact_sensor_update: null argument%s", "");
  if (num_envs <= 0) return RL_OK;
  const RlStepSpec& s = ctx->spec;
  if (!net_forces_w->ptr || !state->net_forces_w_history.ptr) return fail(RL_EINVAL, "rl_contact_sensor_update: net_forces_w and net_forces_w_history required%s", "");
  if (s.num_time_bodies > 0 && (!time_body_to_hist || !state->current_air_time.ptr || !state->last_air_time.ptr ||
                                !state->current_contact_time.ptr || !state->last_contact_time.ptr))
    return fail(RL_EINVAL, "rl_contact_sensor_update: the four timer fields and time_body_to_hist are required%s", "");
  if (ring_slot >= s.hist_len) return fail(RL_EINVAL, "rl_contact_sensor_update: ring_slot %s%lld outside the history length", "", ring_slot);
  if (!(dt > 0.f)) return fail(RL_EINVAL, "rl_contact_sensor_update: dt must be positive%s", "");
  SensorArgs a;
  memset(&a, 0, sizeof(a));
  a.N = (int)num_envs; a.B = s.num_hist_bodies; a.T = s.hist_len; a.Bt = s.num_time_bodies; a.ring_slot = ring_slot;
  a.dt = dt; a.thr = force_threshold;
  a.net = *net_forces_w; a.hist = state->net_forces_w_history;
  a.cair = state->current_air_time; a.lair = state->last_air_time;
  a.ccon = state->current_contact_time; a.lcon = state->last_contact_time;
  for (int f = 0; f < s.num_time_bodies; ++f) {
    if (time_body_to_hist[f] < 0 || time_body_to_hist[f] >= s.num_hist_bodies)
      return fail(RL_EINVAL, "rl_contact_sensor_update: time_body_to_hist[%s%lld] outside the history bodies", "", f);
    a.t2h[f] = time_body_to_hist[f];
  }
  const long long total = num_envs * (long long)(a.B * 3 + a.Bt);
  if (total >= (1ll << 31)) return fail(RL_EINVAL, "rl_contact_sensor_update: problem too large for 32-bit indexing%s", "");
  if (total == 0) return RL_OK;
  DeviceGuard guard(ctx->device);
  const int threads = 256;
  const int blocks = (int)((total + threads - 1) / threads);
  contact_sensor_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  return RL_OK;
}

int rl_process_action(RlCtx* ctx, int64_t num_envs, const RlField* new_action, const RlMdpState* mdp,
                      const RlField* joint_target, const RlField* joint_vel_target, uint64_t* step_counter, void* stream) {
  if (!ctx || !new_action || !mdp) return fail(RL_EINVAL, "rl_process_action: null argument%s", "");
  if (num_envs <= 0) return RL_OK;
  if (!new_action->ptr || !mdp->action.ptr) return fail(RL_EINVAL, "rl_process_action: action pointers required%s", "");
  DeviceGuard guard(ctx->device);
  RlField tgt = joint_target ? *joint_target : RlField{nullptr, 0, 0};
  RlField vtgt = joint_vel_target ? *joint_vel_target : RlField{nullptr, 0, 0};
  const long long total = num_envs * ctx->spec.action.n_actions;
  if (total >= (1ll << 31)) return fail(RL_EINVAL, "rl_process_action: num_envs * n_actions must stay below 2^31%s", "");
  const int threads = 256;
  const int blocks = (int)((num_envs + kPaEnvs - 1) / kPaEnvs);
  if (blocks <= 0 || total <= 0) return RL_OK;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(blocks); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = 0; cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = ctx->use_pdl ? 1 : 0;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, process_action_kernel, (int)num_envs, (int)ctx->spec.action.n_actions, (int)ctx->spec.action.has_clip,
                              (const float*)ctx->action_tab_dev, *new_action, mdp->action, mdp->prev_action, tgt, vtgt,
                              (unsigned long long*)step_counter, ctx->use_pdl));
  return RL_OK;
}

int rl_step(RlCtx* ctx, int64_t num_envs, const RlStateView* state, const RlMdpState* mdp, const RlStepOut* out,
            const RlRandom* rnd, uint32_t phases, const int32_t* env_ids, const int32_t* n_env_ids, void* stream) {
  if (!ctx || !state || !mdp || !out || !rnd) return fail(RL_EINVAL, "rl_step: null argument%s", "");
  if (num_envs <= 0) return RL_OK;
  if (num_envs > 0x7fffffff / 8) return fail(RL_EINVAL, "rl_step: num_envs too large%s", "");
  if ((env_ids == nullptr) != (n_env_ids == nullptr)) return fail(RL_EINVAL, "rl_step: env_ids and n_env_ids go together%s", "");
  const RlStepSpec& s = ctx->spec;
  // required pointers per phase
  if (!state->root_quat_w.ptr || !state->root_lin_vel_w.ptr || !state->root_ang_vel_w.ptr || !state->root_pos_w.ptr ||
      !state->joint_pos.ptr || !state->joint_vel.ptr || !mdp->command.ptr || !mdp->action.ptr || !mdp->episode_length.ptr)
    return fail(RL_EINVAL, "rl_step: root/joint/command/action/episode_length fields are required%s", "");
  if (phases & (RL_PHASE_DONES | RL_PHASE_REWARDS)) {
    if (!state->joint_acc.ptr || !state->applied_torque.ptr || !mdp->prev_action.ptr)
      return fail(RL_EINVAL, "rl_step: joint_acc/applied_torque/prev_action required for rewards%s", "");
    if (s.num_hist_bodies > 0 && !state->net_forces_w_history.ptr) return fail(RL_EINVAL, "rl_step: net_forces_w_history required%s", "");
    if (s.num_time_bodies > 0 && (!state->current_air_time.ptr || !state->last_air_time.ptr || !state->current_contact_time.ptr || !state->last_contact_time.ptr))
      return fail(RL_EINVAL, "rl_step: air/contact time fields required%s", "");
    if (s.num_asset_bodies > 0 && (!state->body_pos_w.ptr || !state->body_lin_vel_w.ptr)) return fail(RL_EINVAL, "rl_step: body_pos_w/body_lin_vel_w required%s", "");
  }
  if ((phases & RL_PHASE_REWARDS) && (!mdp->episode_sums.ptr && s.num_reward_terms > 0))
    return fail(RL_EINVAL, "rl_step: episode_sums required for the reward phase%s", "");
  if (phases & RL_PHASE_COMMAND) {
    if (!mdp->heading_target.ptr || !mdp->time_left.ptr || !mdp->is_heading_env.ptr || !mdp->is_standing_env.ptr ||
        !mdp->metric_error_vel_xy.ptr || !mdp->metric_error_vel_yaw.ptr)
      return fail(RL_EINVAL, "rl_step: command state fields required for the command phase%s", "");
  }
  if ((phases & RL_PHASE_OBS) && s.num_rays > 0 && (!state->ray_hits_z.ptr || !state->ray_sensor_pos_z.ptr)) {
    bool needs = false;
    for (int g = 0; g < RL_NUM_OBS_GROUPS; ++g)
      if (out->obs[g]) for (int t = 0; t < s.obs[g].n_terms; ++t) needs = needs || s.obs[g].terms[t].type == RL_OBS_HEIGHT_SCAN;
    if (needs) return fail(RL_EINVAL, "rl_step: ray_hits_z / ray_sensor_pos_z required for height_scan%s", "");
  }
  for (int g = 0; g < RL_NUM_OBS_GROUPS; ++g)
    if (out->obs[g] && out->obs_pitch[g] < s.obs[g].dim) return fail(RL_EINVAL, "rl_step: obs_pitch[%s%lld] smaller than the group dim", "", g);
  if ((phases & RL_PHASE_RESET) && !env_ids && (!out->terminated || !out->truncated || !out->n_reset))
    return fail(RL_EINVAL, "rl_step: RL_PHASE_RESET without env_ids resets the envs flagged in out->terminated | out->truncated and needs out->n_reset%s", "");
  if ((phases & RL_PHASE_RESET) && (phases & (RL_PHASE_DONES | RL_PHASE_REWARDS))) return fail(RL_EINVAL, "rl_step: RESET combines with COMMAND/OBS only%s", "");
  if ((phases & RL_PHASE_RESET) && !env_ids && !(phases & RL_PHASE_COMMAND))
    return fail(RL_EINVAL, "rl_step: RL_PHASE_RESET over all envs (no env_ids) writes the command state of every env and needs RL_PHASE_COMMAND%s", "");
  if ((phases & RL_PHASE_RESET) && (!mdp->episode_sums.ptr || !mdp->prev_action.ptr || !mdp->heading_target.ptr || !mdp->time_left.ptr ||
      !mdp->is_heading_env.ptr || !mdp->is_standing_env.ptr || !mdp->metric_error_vel_xy.ptr || !mdp->metric_error_vel_yaw.ptr))
    return fail(RL_EINVAL, "rl_step: RL_PHASE_RESET needs every RlMdpState field%s", "");
  if (env_ids && (phases & RL_PHASE_COMPACT)) return fail(RL_EINVAL, "rl_step: compaction is not available on an env_ids subset%s", "");
  if ((phases & RL_PHASE_COMPACT) && !(phases & RL_PHASE_DONES)) return fail(RL_EINVAL, "rl_step: COMPACT needs DONES%s", "");
  DeviceGuard guard(ctx->device);
  const int grid = (int)((num_envs + kE - 1) / kE);
  if (phases & (RL_PHASE_COMPACT | RL_PHASE_RESET)) {
    if (grid > ctx->cta_mask_cap) {
      cudaStreamCaptureStatus cs;
      CUDA_TRY(cudaStreamIsCapturing((cudaStream_t)stream, &cs));
      if (cs != cudaStreamCaptureStatusNone) return fail(RL_EINVAL, "rl_step: first call at this num_envs must happen outside stream capture%s", "");
      int rc = ensure_scratch(ctx, grid);
      if (rc != RL_OK) return rc;
    }
  }
  KArgs a;
  int frc = fill_args(ctx, a, num_envs, state, mdp, out, rnd, phases, 0);
  if (frc != RL_OK) return frc;
  a.has_ids = env_ids != nullptr; a.env_ids = env_ids; a.n_env_ids = n_env_ids;
  if (ctx->v2 && !env_ids) {
    // the two launches of an env step have cluster kernels (csrc/mdp_step_v2.cu); they decline what they do not cover
    constexpr uint32_t kPre = RL_PHASE_DONES | RL_PHASE_REWARDS | RL_PHASE_COMPACT, kPost = RL_PHASE_RESET | RL_PHASE_COMMAND | RL_PHASE_OBS;
    if (phases == kPre || phases == kPost) {
      bool handled = false;
      const int rc = rl_v2_try_launch(ctx, a, phases == kPre ? RL_V2_PRE : RL_V2_POST, (cudaStream_t)stream, &handled);
      if (rc != RL_OK || handled) return rc;
    }
  }
  return dispatch_step<0>(ctx, a, (int)num_envs, (cudaStream_t)stream);
}

int rl_reset_envs(RlCtx* ctx, int64_t num_envs, const RlMdpState* mdp, const uint8_t* done_bits, const RlRandom* rnd,
                  const RlResetLog* log, const int32_t* env_ids, const int32_t* n_env_ids, void* stream) {
  if (!ctx || !mdp || !rnd || !env_ids || !n_env_ids) return fail(RL_EINVAL, "rl_reset_envs: null argument%s", "");
  if (num_envs <= 0) return RL_OK;
  if (!mdp->episode_sums.ptr || !mdp->action.ptr || !mdp->prev_action.ptr || !mdp->command.ptr || !mdp->time_left.ptr ||
      !mdp->heading_target.ptr || !mdp->is_heading_env.ptr || !mdp->is_standing_env.ptr || !mdp->metric_error_vel_xy.ptr ||
      !mdp->metric_error_vel_yaw.ptr || !mdp->episode_length.ptr)
    return fail(RL_EINVAL, "rl_reset_envs: every RlMdpState field is required%s", "");
  DeviceGuard guard(ctx->device);
  const int grid = (int)((num_envs + kE - 1) / kE);
  if (grid > ctx->cta_mask_cap) {
    cudaStreamCaptureStatus cs;
    CUDA_TRY(cudaStreamIsCapturing((cudaStream_t)stream, &cs));
    if (cs != cudaStreamCaptureStatusNone) return fail(RL_EINVAL, "rl_reset_envs: first call at this num_envs must happen outside stream capture%s", "");
    int rc = ensure_scratch(ctx, grid);
    if (rc != RL_OK) return rc;
  }
  KArgs a;
  RlStepOut o;
  memset(&o, 0, sizeof(o));
  o.done_bits = const_cast<uint8_t*>(done_bits);
  if (log) o.reset_log = *log;
  int frc = fill_args(ctx, a, num_envs, nullptr, mdp, &o, rnd, RL_PHASE_RESET, 0);
  if (frc != RL_OK) return frc;
  a.has_ids = 1; a.env_ids = env_ids; a.n_env_ids = n_env_ids;
  return dispatch_step<0>(ctx, a, (int)num_envs, (cudaStream_t)stream);
}

int rl_term_eval(RlCtx* ctx, int64_t num_envs, const RlRewardTerm* term, const RlStateView* state, const RlMdpState* mdp,
                 const uint8_t* terminated, float* out, void* stream) {
  if (!ctx || !term || !state || !mdp || !out) return fail(RL_EINVAL, "rl_term_eval: null argument%s", "");
  if (num_envs <= 0) return RL_OK;
  if (term->type <= RL_REW_NONE || term->type >= RL_REW_TYPE_COUNT) return fail(RL_EINVAL, "rl_term_eval: unknown term type%s %lld", "", term->type);
  if (term->n_idx < 0 || term->n_idx > RL_MAX_IDX) return fail(RL_EINVAL, "rl_term_eval: n_idx out of range%s", "");
  if (!state->root_quat_w.ptr || !state->root_lin_vel_w.ptr || !state->root_ang_vel_w.ptr || !state->root_pos_w.ptr ||
      !state->joint_pos.ptr || !state->joint_vel.ptr || !state->joint_acc.ptr || !state->applied_torque.ptr ||
      !mdp->command.ptr || !mdp->action.ptr || !mdp->prev_action.ptr || !mdp->episode_length.ptr)
    return fail(RL_EINVAL, "rl_term_eval: state fields missing%s", "");
  DeviceGuard guard(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  // rotate through a small ring of device copies so that back-to-back async calls do not race
  static thread_local int ring = 0;
  RlRewardTerm* dev = ctx->adhoc_dev + (ring++ & 63);
  CUDA_TRY(cudaMemcpyAsync(dev, term, sizeof(RlRewardTerm), cudaMemcpyHostToDevice, st));
  KArgs a;
  int frc = fill_args(ctx, a, num_envs, state, mdp, nullptr, nullptr, 0, 1);
  if (frc != RL_OK) return frc;
  a.adhoc = dev; a.ext_terminated = terminated; a.term_out = out; a.use_pdl = 0;
  return dispatch_step<1>(ctx, a, (int)num_envs, st);
}

}  // extern "C"
