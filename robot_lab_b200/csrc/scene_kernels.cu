// scene_kernels.cu - the neighbours of the MDP step (SURVEY.md 8(f) rows 3 and 4), hand-written for sm_100a, behind
// the same C-ABI (include/rl_mdp_step.h):
//
//   rl_actuator_step         Articulation._apply_actuator_model [IL] with the IdealPD / Implicit / DCMotor models the
//                            reference selects per robot (assets/unitree.py:55-63, 107-115, 504-575)
//   rl_is_robot_on_terrain   is_robot_on_terrain (V/mdp/utils.py:73-127)
//   rl_command_pit_restrict  tail of UniformThresholdVelocityCommand._update_command (V/mdp/commands.py:61-85)
//   rl_height_scan_cast      grid-pattern RayCaster [IL] (V/velocity_env_cfg.py:70-77) over a height-field terrain
//   rl_interval_push         EventManager.reset / apply("interval") [IL] with push_by_setting_velocity [IL]
//                            (randomize_push_robot, V/velocity_env_cfg.py:366-371)
//
// All of them are per-env maps over a few hundred bytes per env: HBM / L2 bound elementwise work, no tensor cores.
// Index order follows the layout of the tensor being written so that SoA [C][N] and IsaacLab-shaped AoS [N][C]
// tensors both coalesce. Built with -fmad=false like mdp_step.cu: the reference is eager PyTorch, every op rounds.

#include "rl_common.cuh"

#include <math.h>

namespace {

__device__ __forceinline__ float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }

// ---------------------------------------------------------------------------------------------------
// Actuator models [IL] (isaaclab/actuators/actuator_pd.py): one thread per (env, joint).
// ---------------------------------------------------------------------------------------------------
struct ActuatorArgs {
  int N, J;
  RlField tgt, vtgt, etgt, jpos, jvel, applied, computed;
  RlActuatorCfg cfg;
};

__global__ void __launch_bounds__(256) actuator_kernel(const __grid_constant__ ActuatorArgs a) {
  const int total = a.N * a.J;   // < 2^31, checked by the host
  const bool env_major = (a.applied.env_stride == 1);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int env, j;
    if (env_major) { env = i % a.N; j = i / a.N; } else { j = i % a.J; env = i / a.J; }
    const int type = a.cfg.type[j];
    if (type == RL_ACT_NONE) continue;
    const float q = ld_f(a.jpos, env, j), qd = ld_f(a.jvel, env, j);
    const float pt = ld_f(a.tgt, env, j);
    const float vt = a.vtgt.ptr ? ld_f(a.vtgt, env, j) : 0.f;
    const float et = a.etgt.ptr ? ld_f(a.etgt, env, j) : 0.f;
    // IdealPDActuator.compute [IL]: stiffness * error_pos + damping * error_vel + feed-forward effort
    const float error_pos = pt - q, error_vel = vt - qd;
    const float computed = (a.cfg.stiffness[j] * error_pos + a.cfg.damping[j] * error_vel) + et;
    const float lim = a.cfg.effort_limit[j];
    float lo = -lim, hi = lim;
    if (type == RL_ACT_DC_MOTOR) {
      // DCMotor._clip_effort [IL]: four-quadrant torque-speed curve
      const float sat = a.cfg.saturation_effort[j], vlim = a.cfg.velocity_limit[j];
      const float vel_at_effort_lim = vlim * (1.f + lim / sat);
      const float vel = clampf(qd, -vel_at_effort_lim, vel_at_effort_lim);
      const float top = sat * (1.f - vel / vlim);
      const float bottom = sat * (-1.f - vel / vlim);
      hi = fminf(top, lim);
      lo = fmaxf(bottom, -lim);
    }
    const float applied = fminf(fmaxf(computed, lo), hi);   // torch.clip(x, min, max) = min(max(x, min), max)
    if (a.computed.ptr) st_f(a.computed, env, j, computed);
    st_f(a.applied, env, j, applied);
  }
}

// ---------------------------------------------------------------------------------------------------
// Terrain queries (V/mdp/utils.py:73-127) and the pit branch of the command term (V/mdp/commands.py:61-85).
// The terrain origins (x, y of every grid cell) are staged in shared memory once per CTA; a group of 8 lanes scans
// them for one env and reduces to the first minimum in flat row-major order, like torch.argmin.
// The distance is sqrt(dx^2 + dy^2) as torch.cdist defines it (the reference's matmul-based cdist path differs
// from it only in rounding, i.e. for robots within ~1e-4 m of a cell boundary).
// ---------------------------------------------------------------------------------------------------
constexpr int kMaxTerrainCells = 4096;   // 32 KB of shared memory for (x, y)

struct TerrainArgs {
  int N;
  RlField pos;
  RlTerrainGrid grid;
  // rl_is_robot_on_terrain
  uint8_t* out;
  // rl_command_pit_restrict
  RlField cmd, head, ishead, isstand;
  uint8_t* was_on_pit;
  RlRandom rnd;
  RlCommandCfg cc;
};

__device__ __forceinline__ void stage_origins(float* s_xy, const RlTerrainGrid& g) {
  const int cells = g.num_rows * g.num_cols;
  for (int i = threadIdx.x; i < cells; i += blockDim.x) {
    s_xy[2 * i] = g.terrain_origins[3 * i];
    s_xy[2 * i + 1] = g.terrain_origins[3 * i + 1];
  }
  __syncthreads();
}

// kLanesPerEnv lanes share one env: lane l scans cells l, l + kLanesPerEnv, ... and keeps ITS first minimum; the
// group then reduces to the smallest distance, ties to the smallest flat index - exactly the first minimum of the
// whole scan. sqrt is monotone, so a cell whose squared distance is not below the running best cannot win: the IEEE
// square root is only taken for the few candidates that pass that filter (a smaller squared distance can still round
// to the same distance - then the earlier index stays, as in torch.argmin over the rounded distances).
// Tolerance against the reference (advisor note): `torch.cdist` switches to the matmul form |x|^2 + |y|^2 - 2 x.y when
// either operand has more than 25 rows - every terrain grid here - which rounds differently from the direct
// sqrt(dx^2 + dy^2) used below (and by the CPU restatement the tests check against). A robot within rounding distance
// of the bisector between two cell centres can therefore resolve to the other cell than in the reference; the decision
// (pit column or not) differs only if those two cells lie on different sides of the pit columns' edge. The golden
// fixtures (tests/test_pit_terrain_golden.py) keep robots away from bisectors; everywhere else the argmin is the same.
constexpr int kLanesPerEnv = 8;

__device__ __forceinline__ bool on_terrain(const float* s_xy, const RlTerrainGrid& g, float x, float y, int sub) {
  const int cells = g.num_rows * g.num_cols;
  float best = INFINITY, best2 = INFINITY;
  int arg = 0x7fffffff;
  for (int i = sub; i < cells; i += kLanesPerEnv) {
    const float dx = x - s_xy[2 * i], dy = y - s_xy[2 * i + 1];
    const float d2 = dx * dx + dy * dy;
    if (d2 < best2) {
      const float d = sqrtf(d2);
      if (d < best) { best = d; best2 = d2; arg = i; }
    }
  }
#pragma unroll
  for (int off = 1; off < kLanesPerEnv; off <<= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, off);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, off);
    if (ob < best || (ob == best && oa < arg)) { best = ob; arg = oa; }
  }
  if (arg == 0x7fffffff) arg = 0;   // nothing compared below +inf (NaN position): torch.argmin returns index 0
  const int col = arg % g.num_cols;
  return (col >= g.col_start) && (col < g.col_end);
}

template <bool RESTRICT>
__global__ void __launch_bounds__(128) terrain_kernel(const __grid_constant__ TerrainArgs a) {
  extern __shared__ float s_xy[];
  stage_origins(s_xy, a.grid);
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int sub = gid % kLanesPerEnv;
  const int env_raw = gid / kLanesPerEnv;
  const int env = min(env_raw, a.N - 1);       // whole lane groups stay converged for the shuffles
  const bool on = on_terrain(s_xy, a.grid, ld_f(a.pos, env, 0), ld_f(a.pos, env, 1), sub);
  if (env_raw >= a.N || sub != 0) return;
  if constexpr (!RESTRICT) {
    a.out[env] = on ? 1 : 0;
  } else {
    const bool was = a.was_on_pit[env] != 0;
    const RlCommandCfg& cc = a.cc;
    if (was && !on) {
      // UniformVelocityCommand._resample_command [IL] + the small-command threshold (V/mdp/commands.py:43-47)
      float u[RL_NUM_CMD_UNIFORMS];
      if (a.rnd.cmd_uniforms != nullptr) {
#pragma unroll
        for (int i = 1; i < RL_NUM_CMD_UNIFORMS; ++i) u[i] = a.rnd.cmd_uniforms[(long long)i * a.N + env];
      } else {
        const RandState rs = rl_rand_state(a.rnd);
        const uint4 r0 = rl_philox(rs, env, RL_STREAM_PIT_RESAMPLE, 0), r1 = rl_philox(rs, env, RL_STREAM_PIT_RESAMPLE, 1);
        u[1] = u01(r0.y); u[2] = u01(r0.z); u[3] = u01(r0.w);
        u[4] = u01(r1.x); u[5] = u01(r1.y); u[6] = u01(r1.z);
      }
      float c0 = u[1] * (cc.lin_vel_x_hi - cc.lin_vel_x_lo) + cc.lin_vel_x_lo;
      float c1 = u[2] * (cc.lin_vel_y_hi - cc.lin_vel_y_lo) + cc.lin_vel_y_lo;
      const float c2 = u[3] * (cc.ang_vel_z_hi - cc.ang_vel_z_lo) + cc.ang_vel_z_lo;
      if (cc.heading_command) {
        st_f(a.head, env, 0, u[4] * (cc.heading_hi - cc.heading_lo) + cc.heading_lo);
        static_cast<uint8_t*>(a.ishead.ptr)[(long long)env * a.ishead.env_stride] = (u[5] <= cc.rel_heading_envs) ? 1 : 0;
      }
      static_cast<uint8_t*>(a.isstand.ptr)[(long long)env * a.isstand.env_stride] = (u[6] <= cc.rel_standing_envs) ? 1 : 0;
      const float keep = (sqrtf(c0 * c0 + c1 * c1) > cc.small_cmd_threshold) ? 1.f : 0.f;
      c0 *= keep; c1 *= keep;
      st_f(a.cmd, env, 0, c0); st_f(a.cmd, env, 1, c1); st_f(a.cmd, env, 2, c2);
    }
    if (on) {
      // forward only, 0.3 .. 0.6 m/s, no lateral / yaw command, heading target 0 (V/mdp/commands.py:72-82)
      const float c0 = ld_f(a.cmd, env, 0);
      st_f(a.cmd, env, 0, clampf(fabsf(c0), 0.3f, 0.6f));
      st_f(a.cmd, env, 1, 0.f);
      st_f(a.cmd, env, 2, 0.f);
      if (cc.heading_command) st_f(a.head, env, 0, 0.f);
    }
    a.was_on_pit[env] = on ? 1 : 0;
  }
}

// ---------------------------------------------------------------------------------------------------
// Height-scan ray caster over a height field. One warp per env: every lane evaluates the yaw rotation of its env once
// (not once per ray), then the lanes stride over the env's rays - neighbouring rays read neighbouring vertices (same
// L1 lines) and the hit row [R] is written coalesced. The height field (1201 x 2001 vertices = 9.6 MB for the default
// rough terrain) stays L2-resident; 8 envs per CTA, grid = N / 8.
// isaaclab.utils.math [IL]: yaw_quat, quat_apply.
// ---------------------------------------------------------------------------------------------------
struct CastArgs {
  int N;
  RlHeightField hf;
  RlField pos, quat, hits, sensor_z;
};

__global__ void __launch_bounds__(256) height_scan_kernel(const __grid_constant__ CastArgs a) {
  const int R = a.hf.num_rays;
  const int lane = threadIdx.x & 31;
  const int warps_per_grid = (gridDim.x * blockDim.x) >> 5;
  for (int env = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; env < a.N; env += warps_per_grid) {
    const float px = ld_f(a.pos, env, 0), py = ld_f(a.pos, env, 1);
    const float qw = ld_f(a.quat, env, 0), qx = ld_f(a.quat, env, 1), qy = ld_f(a.quat, env, 2), qz = ld_f(a.quat, env, 3);
    if (lane == 0 && a.sensor_z.ptr) st_f(a.sensor_z, env, 0, ld_f(a.pos, env, 2));
    // yaw_quat [IL]
    const float yaw = atan2f(2.f * (qw * qz + qx * qy), 1.f - 2.f * (qy * qy + qz * qz));
    float yw = cosf(yaw / 2.f), yz = sinf(yaw / 2.f);
    const float nrm = fmaxf(sqrtf(yw * yw + yz * yz), 1e-9f);
    yw = yw / nrm; yz = yz / nrm;
    // batches of kRaysPerLane rays per lane: all vertex loads of a batch are issued before the first interpolation,
    // so the L2 round trips of the batch overlap instead of queueing behind each other (187 rays = one batch)
    constexpr int kRaysPerLane = 6;
    for (int base = 0; base < R; base += 32 * kRaysPerLane) {
      float fx[kRaysPerLane], fy[kRaysPerLane], h00[kRaysPerLane], h01[kRaysPerLane], h10[kRaysPerLane], h11[kRaysPerLane];
      bool inside[kRaysPerLane];
#pragma unroll
      for (int k = 0; k < kRaysPerLane; ++k) {
        const int r = min(base + k * 32 + lane, R - 1);
        // quat_apply [IL] with xyz = (0, 0, yz): t = 2 * (xyz x v); v + w * t + xyz x t
        const float vx = __ldg(a.hf.ray_starts + 3 * r), vy = __ldg(a.hf.ray_starts + 3 * r + 1);
        const float tx = (0.f - yz * vy) * 2.f, ty = (yz * vx - 0.f) * 2.f;
        const float cx = 0.f - yz * ty, cy = yz * tx - 0.f;
        const float wx = ((vx + yw * tx) + cx) + px, wy = ((vy + yw * ty) + cy) + py;
        // cell of the height-field mesh under (wx, wy)
        const float gx = (wx - a.hf.x0) / a.hf.horizontal_scale, gy = (wy - a.hf.y0) / a.hf.horizontal_scale;
        inside[k] = gx >= 0.f && gy >= 0.f && gx <= (float)(a.hf.num_x - 1) && gy <= (float)(a.hf.num_y - 1);
        const int ix = inside[k] ? min((int)gx, a.hf.num_x - 2) : 0, iy = inside[k] ? min((int)gy, a.hf.num_y - 2) : 0;
        fx[k] = gx - (float)ix; fy[k] = gy - (float)iy;
        const float* h = a.hf.heights + (long long)ix * a.hf.num_y + iy;
        h00[k] = __ldg(h); h01[k] = __ldg(h + 1); h10[k] = __ldg(h + a.hf.num_y); h11[k] = __ldg(h + a.hf.num_y + 1);
      }
#pragma unroll
      for (int k = 0; k < kRaysPerLane; ++k) {
        const int r = base + k * 32 + lane;
        // triangle (v00, v11, v01) above the diagonal, (v00, v10, v11) below it
        const float za = (h00[k] + fx[k] * (h11[k] - h01[k])) + fy[k] * (h01[k] - h00[k]);
        const float zb = (h00[k] + fx[k] * (h10[k] - h00[k])) + fy[k] * (h11[k] - h10[k]);
        const float z = inside[k] ? ((fy[k] >= fx[k]) ? za : zb) : INFINITY;
        if (r < R) st_f(a.hits, env, r, z);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Derived articulation views [IL] (ArticulationData properties that Python term functions read: V/mdp/rewards.py:34,
// 226 and 28 more uses): projected_gravity_b, root_lin_vel_b (= root_com_lin_vel_b), root_ang_vel_b, heading_w.
// One thread per env; same arithmetic, same operand order as make_ctx / command_update of the step kernels
// (isaaclab.utils.math.quat_apply_inverse / quat_apply [IL]).
// ---------------------------------------------------------------------------------------------------
struct DerivedArgs {
  int N;
  RlField quat, lin, ang;
  RlField grav_b, lin_b, ang_b, heading;
};
struct D3 { float x, y, z; };
__device__ __forceinline__ D3 d_cross(D3 a, D3 b) { return D3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
__device__ __forceinline__ D3 d_rot(float w, D3 q, D3 v, float sign) {   // sign -1: quat_apply_inverse, +1: quat_apply
  D3 t = d_cross(q, v);
  t.x *= 2.f; t.y *= 2.f; t.z *= 2.f;
  const D3 c = d_cross(q, t);
  const float sw = sign * w;
  return D3{(v.x + sw * t.x) + c.x, (v.y + sw * t.y) + c.y, (v.z + sw * t.z) + c.z};
}
__global__ void __launch_bounds__(256) derived_views_kernel(const __grid_constant__ DerivedArgs a) {
  for (int env = blockIdx.x * blockDim.x + threadIdx.x; env < a.N; env += gridDim.x * blockDim.x) {
    const float w = ld_f(a.quat, env, 0);
    const D3 q{ld_f(a.quat, env, 1), ld_f(a.quat, env, 2), ld_f(a.quat, env, 3)};
    if (a.grav_b.ptr) {
      const D3 g = d_rot(w, q, D3{0.f, 0.f, -1.f}, -1.f);
      st_f(a.grav_b, env, 0, g.x); st_f(a.grav_b, env, 1, g.y); st_f(a.grav_b, env, 2, g.z);
    }
    if (a.lin_b.ptr) {
      const D3 v = d_rot(w, q, D3{ld_f(a.lin, env, 0), ld_f(a.lin, env, 1), ld_f(a.lin, env, 2)}, -1.f);
      st_f(a.lin_b, env, 0, v.x); st_f(a.lin_b, env, 1, v.y); st_f(a.lin_b, env, 2, v.z);
    }
    if (a.ang_b.ptr) {
      const D3 v = d_rot(w, q, D3{ld_f(a.ang, env, 0), ld_f(a.ang, env, 1), ld_f(a.ang, env, 2)}, -1.f);
      st_f(a.ang_b, env, 0, v.x); st_f(a.ang_b, env, 1, v.y); st_f(a.ang_b, env, 2, v.z);
    }
    if (a.heading.ptr) {
      const D3 f = d_rot(w, q, D3{1.f, 0.f, 0.f}, 1.f);
      st_f(a.heading, env, 0, atan2f(f.y, f.x));
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Interval push event [IL]: EventManager._prepare_terms / reset / apply("interval") for one non-global interval term
// (isaaclab/managers/event_manager.py) and its function push_by_setting_velocity (isaaclab/envs/mdp/events.py). One
// thread per env (step form) or per listed id (reset form): a few bytes per env, no reuse. The pushed ids leave through
// one atomic per warp (ballot + prefix popcount), so their order within the list is unspecified.
// ---------------------------------------------------------------------------------------------------
struct IntervalArgs {
  int N;
  float dt;
  RlIntervalEventCfg cfg;
  float* time_left;
  RlField lin, ang;
  const uint8_t* terminated;
  const uint8_t* truncated;
  const int32_t* env_ids;
  const int32_t* n_env_ids;
  int32_t* pushed_ids;
  int32_t* n_pushed;
  RlRandom rnd;
  const float* uniforms;   // [8][N] or NULL: timer on reset, timer on fire, velocity x, y, z, roll, pitch, yaw
};

// torch.rand(n) * (upper - lower) + lower [IL], the interval sample of _prepare_terms, reset and apply
__device__ __forceinline__ float interval_sample(const RlIntervalEventCfg& c, float u) {
  return u * (c.interval_hi - c.interval_lo) + c.interval_lo;
}

__device__ __forceinline__ float interval_reset_uniform(const IntervalArgs& a, long long env) {
  if (a.uniforms) return a.uniforms[env];
  return u01(rl_philox_inline(rl_rand_state(a.rnd), env, RL_STREAM_INTERVAL_RESET, 0).x);
}

__global__ void __launch_bounds__(256) interval_reset_kernel(const __grid_constant__ IntervalArgs a) {
  const int n = *a.n_env_ids;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const long long env = a.env_ids[i];
    a.time_left[env] = interval_sample(a.cfg, interval_reset_uniform(a, env));
  }
}

__global__ void __launch_bounds__(256) interval_step_kernel(const __grid_constant__ IntervalArgs a) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  bool fire = false;
  if (env < a.N) {
    float t = a.time_left[env];
    // EventManager.reset(env_ids) [IL] of the envs reset at stage 6 of this step
    if ((a.terminated && a.terminated[env]) || (a.truncated && a.truncated[env])) t = interval_sample(a.cfg, interval_reset_uniform(a, env));
    // apply("interval"): time_left -= dt; time_left < 1e-6 (fp32 tensor against a python scalar: compared in fp32)
    t = t - a.dt;
    fire = t < 1e-6f;
    if (fire) {
      float u[7];
      if (a.uniforms) {
#pragma unroll
        for (int q = 0; q < 7; ++q) u[q] = a.uniforms[(long long)(q + 1) * a.N + env];
      } else {
        const RandState rs = rl_rand_state(a.rnd);
        const uint4 r0 = rl_philox_inline(rs, env, RL_STREAM_INTERVAL_PUSH, 0), r1 = rl_philox_inline(rs, env, RL_STREAM_INTERVAL_PUSH, 1);
        u[0] = u01(r0.x); u[1] = u01(r0.y); u[2] = u01(r0.z); u[3] = u01(r0.w);
        u[4] = u01(r1.x); u[5] = u01(r1.y); u[6] = u01(r1.z);
      }
      t = interval_sample(a.cfg, u[0]);
      // push_by_setting_velocity [IL]: root_vel_w += sample_uniform(ranges[:, 0], ranges[:, 1]) = rand * (hi - lo) + lo
      const RlIntervalEventCfg& c = a.cfg;
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        st_f(a.lin, env, q, ld_f(a.lin, env, q) + (u[1 + q] * (c.vel_hi[q] - c.vel_lo[q]) + c.vel_lo[q]));
        st_f(a.ang, env, q, ld_f(a.ang, env, q) + (u[4 + q] * (c.vel_hi[3 + q] - c.vel_lo[3 + q]) + c.vel_lo[3 + q]));
      }
    }
    a.time_left[env] = t;
  }
  const unsigned m = __ballot_sync(0xffffffffu, fire);   // whole warps reach this point (no early exit above)
  if (m) {
    const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(a.n_pushed, __popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (fire) a.pushed_ids[base + __popc(m & ((1u << lane) - 1u))] = env;
  }
}

}  // namespace

extern "C" {

int rl_actuator_step(RlCtx* ctx, int64_t num_envs, const RlActuatorCfg* cfg, const RlField* joint_pos_target,
                     const RlField* joint_vel_target, const RlField* joint_effort_target, const RlStateView* state,
                     const RlField* computed_torque, void* stream) {
  if (!ctx || !cfg || !joint_pos_target || !state) return rl_fail(RL_EINVAL, "rl_actuator_step: null argument%s", "");
  if (num_envs <= 0) return RL_OK;
  const RlStepSpec* s = rl_ctx_spec_of(ctx);
  if (cfg->num_joints != s->num_joints)
    return rl_fail(RL_EINVAL, "rl_actuator_step: cfg has %s%lld joints, the context's spec %lld", "", cfg->num_joints, s->num_joints);
  if (!joint_pos_target->ptr || !state->joint_pos.ptr || !state->joint_vel.ptr || !state->applied_torque.ptr)
    return rl_fail(RL_EINVAL, "rl_actuator_step: joint_pos_target, joint_pos, joint_vel and applied_torque are required%s", "");
  for (int j = 0; j < cfg->num_joints; ++j) {
    const int t = cfg->type[j];
    if (t < RL_ACT_NONE || t > RL_ACT_DC_MOTOR) return rl_fail(RL_EINVAL, "rl_actuator_step: joint %s%lld has an unknown actuator type", "", j);
    if (t == RL_ACT_DC_MOTOR && !(cfg->saturation_effort[j] > 0.f && cfg->velocity_limit[j] > 0.f))
      return rl_fail(RL_EINVAL, "rl_actuator_step: DC motor joint %s%lld needs positive saturation_effort and velocity_limit", "", j);
  }
  const long long total = num_envs * (long long)cfg->num_joints;
  if (total >= (1ll << 31)) return rl_fail(RL_EINVAL, "rl_actuator_step: num_envs * num_joints must stay below 2^31%s", "");
  ActuatorArgs a;
  memset(&a, 0, sizeof(a));
  a.N = (int)num_envs; a.J = cfg->num_joints;
  a.tgt = *joint_pos_target;
  if (joint_vel_target) a.vtgt = *joint_vel_target;
  if (joint_effort_target) a.etgt = *joint_effort_target;
  a.jpos = state->joint_pos; a.jvel = state->joint_vel; a.applied = state->applied_torque;
  if (computed_torque) a.computed = *computed_torque;
  a.cfg = *cfg;
  RlDeviceGuard guard(rl_ctx_device_of(ctx));
  const int threads = 256;
  const int blocks = (int)((total + threads - 1) / threads);
  actuator_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  return RL_OK;
}

static int check_grid(const char* who, const RlTerrainGrid* g) {
  if (!g->terrain_origins || g->num_rows <= 0 || g->num_cols <= 0)
    return rl_fail(RL_EINVAL, "%s: terrain_origins with positive num_rows / num_cols required", who);
  if ((long long)g->num_rows * g->num_cols > kMaxTerrainCells)
    return rl_fail(RL_EUNSUPPORTED, "%s: more than %lld terrain cells", who, kMaxTerrainCells);
  return RL_OK;
}

int rl_is_robot_on_terrain(RlCtx* ctx, int64_t num_envs, const RlField* root_pos_w, const RlTerrainGrid* grid,
                           uint8_t* out, void* stream) {
  if (!ctx || !root_pos_w || !grid || !out) return rl_fail(RL_EINVAL, "rl_is_robot_on_terrain: null argument%s", "");
  if (num_envs <= 0) return RL_OK;
  if (!root_pos_w->ptr) return rl_fail(RL_EINVAL, "rl_is_robot_on_terrain: root_pos_w required%s", "");
  if (int rc = check_grid("rl_is_robot_on_terrain", grid)) return rc;
  if (num_envs >= (1ll << 27)) return rl_fail(RL_EINVAL, "rl_is_robot_on_terrain: too many envs%s", "");
  TerrainArgs a;
  memset(&a, 0, sizeof(a));
  a.N = (int)num_envs; a.pos = *root_pos_w; a.grid = *grid; a.out = out;
  RlDeviceGuard guard(rl_ctx_device_of(ctx));
  const int threads = 128;
  const size_t smem = sizeof(float) * 2 * (size_t)grid->num_rows * grid->num_cols;
  const long long work = num_envs * kLanesPerEnv;
  terrain_kernel<false><<<(int)((work + threads - 1) / threads), threads, smem, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  return RL_OK;
}

int rl_command_pit_restrict(RlCtx* ctx, int64_t num_envs, const RlField* root_pos_w, const RlTerrainGrid* grid,
                            const RlMdpState* mdp, uint8_t* was_on_pit, const RlRandom* rnd, void* stream) {
  if (!ctx || !root_pos_w || !grid || !mdp || !was_on_pit || !rnd)
    return rl_fail(RL_EINVAL, "rl_command_pit_restrict: null argument%s", "");
  if (num_envs <= 0) return RL_OK;
  if (int rc = check_grid("rl_command_pit_restrict", grid)) return rc;
  if (num_envs >= (1ll << 27)) return rl_fail(RL_EINVAL, "rl_command_pit_restrict: too many envs%s", "");
  const RlStepSpec* s = rl_ctx_spec_of(ctx);
  if (!root_pos_w->ptr || !mdp->command.ptr || !mdp->is_standing_env.ptr ||
      (s->command.heading_command && (!mdp->heading_target.ptr || !mdp->is_heading_env.ptr)))
    return rl_fail(RL_EINVAL, "rl_command_pit_restrict: root_pos_w and the command state fields are required%s", "");
  TerrainArgs a;
  memset(&a, 0, sizeof(a));
  a.N = (int)num_envs; a.pos = *root_pos_w; a.grid = *grid;
  a.cmd = mdp->command; a.head = mdp->heading_target; a.ishead = mdp->is_heading_env; a.isstand = mdp->is_standing_env;
  a.was_on_pit = was_on_pit; a.rnd = *rnd; a.cc = s->command;
  RlDeviceGuard guard(rl_ctx_device_of(ctx));
  const int threads = 128;
  const size_t smem = sizeof(float) * 2 * (size_t)grid->num_rows * grid->num_cols;
  const long long work = num_envs * kLanesPerEnv;
  terrain_kernel<true><<<(int)((work + threads - 1) / threads), threads, smem, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  return RL_OK;
}

int rl_height_scan_cast(RlCtx* ctx, int64_t num_envs, const RlHeightField* hf, const RlStateView* state, void* stream) {
  if (!ctx || !hf || !state) return rl_fail(RL_EINVAL, "rl_height_scan_cast: null argument%s", "");
  if (num_envs <= 0) return RL_OK;
  const RlStepSpec* s = rl_ctx_spec_of(ctx);
  if (hf->num_rays != s->num_rays) return rl_fail(RL_EINVAL, "rl_height_scan_cast: %s%lld rays, the context's spec has %lld", "", hf->num_rays, s->num_rays);
  if (hf->num_rays <= 0) return RL_OK;
  if (!hf->heights || !hf->ray_starts || hf->num_x < 2 || hf->num_y < 2 || !(hf->horizontal_scale > 0.f))
    return rl_fail(RL_EINVAL, "rl_height_scan_cast: heights (>= 2 x 2), ray_starts and a positive horizontal_scale are required%s", "");
  if (!state->root_pos_w.ptr || !state->root_quat_w.ptr || !state->ray_hits_z.ptr)
    return rl_fail(RL_EINVAL, "rl_height_scan_cast: root_pos_w, root_quat_w and ray_hits_z are required%s", "");
  CastArgs a;
  memset(&a, 0, sizeof(a));
  a.N = (int)num_envs; a.hf = *hf;
  a.pos = state->root_pos_w; a.quat = state->root_quat_w; a.hits = state->ray_hits_z; a.sensor_z = state->ray_sensor_pos_z;
  RlDeviceGuard guard(rl_ctx_device_of(ctx));
  const int threads = 256;   // 8 warps = 8 envs per CTA
  const long long want = (num_envs + 7) / 8;
  const int blocks = (int)(want < (1ll << 20) ? want : (1ll << 20));
  height_scan_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  return RL_OK;
}

int rl_derived_views(RlCtx* ctx, int64_t num_envs, const RlStateView* state, const RlField* projected_gravity_b,
                     const RlField* root_lin_vel_b, const RlField* root_ang_vel_b, const RlField* heading_w, void* stream) {
  if (!ctx || !state) return rl_fail(RL_EINVAL, "rl_derived_views: null argument%s", "");
  if (num_envs <= 0) return RL_OK;
  if (!state->root_quat_w.ptr) return rl_fail(RL_EINVAL, "rl_derived_views: root_quat_w is required%s", "");
  if ((root_lin_vel_b && root_lin_vel_b->ptr && !state->root_lin_vel_w.ptr) || (root_ang_vel_b && root_ang_vel_b->ptr && !state->root_ang_vel_w.ptr))
    return rl_fail(RL_EINVAL, "rl_derived_views: the world-frame velocity of a requested base-frame velocity is missing%s", "");
  DerivedArgs a;
  memset(&a, 0, sizeof(a));
  a.N = (int)num_envs;
  a.quat = state->root_quat_w; a.lin = state->root_lin_vel_w; a.ang = state->root_ang_vel_w;
  if (projected_gravity_b) a.grav_b = *projected_gravity_b;
  if (root_lin_vel_b) a.lin_b = *root_lin_vel_b;
  if (root_ang_vel_b) a.ang_b = *root_ang_vel_b;
  if (heading_w) a.heading = *heading_w;
  RlDeviceGuard guard(rl_ctx_device_of(ctx));
  const int threads = 256;
  const int blocks = (int)((num_envs + threads - 1) / threads);
  derived_views_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  return RL_OK;
}

int rl_interval_push(RlCtx* ctx, int64_t num_envs, const RlIntervalEventCfg* cfg, float dt, float* time_left,
                     const RlStateView* state, const uint8_t* terminated, const uint8_t* truncated,
                     const int32_t* env_ids, const int32_t* n_env_ids, int32_t* pushed_ids, int32_t* n_pushed,
                     const RlRandom* rnd, const float* uniforms, void* stream) {
  if (!ctx || !cfg || !time_left || !rnd) return rl_fail(RL_EINVAL, "rl_interval_push: null argument%s", "");
  if (!(cfg->interval_lo <= cfg->interval_hi))
    return rl_fail(RL_EINVAL, "rl_interval_push: interval_range_s needs lo <= hi%s", "");
  for (int q = 0; q < 6; ++q)
    if (!(cfg->vel_lo[q] <= cfg->vel_hi[q]))
      return rl_fail(RL_EINVAL, "rl_interval_push: velocity_range component %s%lld needs lo <= hi", "", q);
  if (num_envs >= (1ll << 31)) return rl_fail(RL_EINVAL, "rl_interval_push: num_envs must stay below 2^31%s", "");
  IntervalArgs a;
  memset(&a, 0, sizeof(a));
  a.N = (int)(num_envs > 0 ? num_envs : 0); a.dt = dt; a.cfg = *cfg; a.time_left = time_left;
  a.rnd = *rnd; a.uniforms = uniforms;
  RlDeviceGuard guard(rl_ctx_device_of(ctx));
  const int threads = 256;
  const int blocks = (int)((num_envs + threads - 1) / threads);
  if (env_ids || n_env_ids) {   // reset form
    if (!env_ids || !n_env_ids) return rl_fail(RL_EINVAL, "rl_interval_push: env_ids and n_env_ids go together%s", "");
    if (num_envs <= 0) return RL_OK;
    a.env_ids = env_ids; a.n_env_ids = n_env_ids;
    interval_reset_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(a);
    CUDA_TRY(cudaGetLastError());
    return RL_OK;
  }
  if (!state || !state->root_lin_vel_w.ptr || !state->root_ang_vel_w.ptr)
    return rl_fail(RL_EINVAL, "rl_interval_push: root_lin_vel_w and root_ang_vel_w are required%s", "");
  if (!terminated && !truncated) return rl_fail(RL_EINVAL, "rl_interval_push: env_ids or the done masks are required%s", "");
  if (!pushed_ids || !n_pushed) return rl_fail(RL_EINVAL, "rl_interval_push: pushed_ids and n_pushed are required%s", "");
  if (!(dt > 0.f)) return rl_fail(RL_EINVAL, "rl_interval_push: dt must be positive%s", "");
  CUDA_TRY(cudaMemsetAsync(n_pushed, 0, sizeof(int32_t), (cudaStream_t)stream));   // a graph node: defined on every replay
  if (num_envs <= 0) return RL_OK;
  a.lin = state->root_lin_vel_w; a.ang = state->root_ang_vel_w;
  a.terminated = terminated; a.truncated = truncated; a.pushed_ids = pushed_ids; a.n_pushed = n_pushed;
  interval_step_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  return RL_OK;
}

}  // extern "C"
