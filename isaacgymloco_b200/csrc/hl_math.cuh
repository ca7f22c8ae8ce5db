// Per-environment math of the post-physics path, shared by the fused kernel (shared-memory
// view, one lane per env) and the generic stage kernel (global view, one warp per env).
// Every function cites the reference lines it restates (LR = legged_robot.py).
#pragma once
#include "hl_common.cuh"

// Where one env's records live (shared-memory slab or global memory; generic pointers).
struct EnvView {
  const float* root;     // 13: pos3 quat_xyzw4 lin3 ang3
  const float* dof;      // 24: (pos, vel) interleaved
  const float* cf;       // B*3 contact forces
  const float* fpos[4];  // world position (3) of foot f
  const float* fvel[4];  // world linear velocity (3) of foot f
  const float* act;      // 12 each
  const float* lact;
  const float* llact;
  const float* ldp;      // last_dof_pos   (only read by dof_pos_dif)
  const float* ldv;      // last_dof_vel
  const float* tq;
  const float* ltq;      // last_torques   (only read by torques_dif)
  __device__ __forceinline__ float dof_pos(int d) const { return dof[2 * d]; }
  __device__ __forceinline__ float dof_vel(int d) const { return dof[2 * d + 1]; }
};

struct EnvScalars {
  float blv[3], bav[3], pg[3];  // base_lin_vel, base_ang_vel, projected_gravity
  float cmd[4];
  float air[4];                 // feet_air_time
  float base_h;                 // _get_base_heights()
  int feet_shift;               // how many times _reward_foot_clearance_terrain did `feet_pos += border`
  long long ep_len, terrain_level, gid;
  unsigned contact, cfilt, last_contact;  // bit f = foot f
  bool time_out, reset;
};

// body-state record (13 floats) of foot f of env e: from the packed (N,4,13) tensor when given, else
// rigid_body_states[e, feet_idx[f]] (LR:203-204)
__device__ __forceinline__ const float* hl_foot_rec(const HlCfg& c, const HlEnvBuffers& b, long long e, int f) {
  return b.foot_records ? b.foot_records + (e * 4 + f) * 13 : b.rigid_body_states + (e * c.num_bodies + c.feet_idx[f]) * 13;
}

// ----------------------------------------------------------------------------- frame
// isaacgym.torch_utils.quat_rotate_inverse: a - b + c with a = v(2w^2-1), b = 2w(q_v x v),
// c = 2 q_v (q_v . v)   (used at LR:198-200,1616,1691-1692)
__device__ __forceinline__ void hl_quat_rotate_inverse(const float* q, float vx, float vy, float vz, float* o) {
  const float x = q[0], y = q[1], z = q[2], w = q[3];
  const float s = 2.0f * w * w - 1.0f;
  const float cx = y * vz - z * vy, cy = z * vx - x * vz, cz = x * vy - y * vx;
  const float d = x * vx + y * vy + z * vz;
  o[0] = vx * s - cx * w * 2.0f + x * d * 2.0f;
  o[1] = vy * s - cy * w * 2.0f + y * d * 2.0f;
  o[2] = vz * s - cz * w * 2.0f + z * d * 2.0f;
}

__device__ __forceinline__ void hl_frame(const EnvView& v, EnvScalars& s) {  // LR:197-200
  const float* q = v.root + 3;
  hl_quat_rotate_inverse(q, v.root[7], v.root[8], v.root[9], s.blv);
  hl_quat_rotate_inverse(q, v.root[10], v.root[11], v.root[12], s.bav);
  hl_quat_rotate_inverse(q, 0.0f, 0.0f, -1.0f, s.pg);
}

// LR:616-620 with quat_apply(q,(1,0,0)) expanded and wrap_to_pi of utils/math.py:45-48.
__device__ __forceinline__ float hl_heading_command(const float* q, float cmd_heading) {
  const float x = q[0], y = q[1], z = q[2], w = q[3];
  const float ty = 2.0f * z, tz = -2.0f * y;           // t = 2 (q_v x e_x) = (0, 2z, -2y)
  const float fx = 1.0f + (y * tz - z * ty);           // b + w t + q_v x t
  const float fy = w * ty + (-x * tz);
  const float heading = atan2f(fy, fx);
  const float two_pi = 6.283185307179586f, pi = 3.141592653589793f;
  float a = hl_pymod(cmd_heading - heading, two_pi);
  a -= two_pi * (a > pi ? 1.0f : 0.0f);
  return hl_clampf(0.5f * a, -2.0f, 2.0f);
}

__device__ __forceinline__ void hl_contacts(const HlCfg& c, const EnvView& v, unsigned last, EnvScalars& s) {
  unsigned ct = 0;                                      // LR:207-209
#pragma unroll
  for (int f = 0; f < 4; ++f) ct |= (v.cf[c.feet_idx[f] * 3 + 2] > 1.0f ? 1u : 0u) << f;
  s.contact = ct;
  s.cfilt = ct | last;
  s.last_contact = ct;
}

// ----------------------------------------------------------------------------- height scan
// Yaw-only unit quaternion exactly as quat_apply_yaw builds it (utils/math.py:38-42 +
// torch_utils.normalize): norm over (0,0,z,w) = sqrt(rn(rn(z^2)+rn(w^2))) -- the rounding eager
// torch produces on both devices (the squares are rounded separately, see DESIGN.md).
__device__ __forceinline__ void hl_yaw_quat(const float* q, float& qz, float& qw) {
  const float z = q[2], w = q[3];
  float n = __fsqrt_rn(__fadd_rn(__fmul_rn(z, z), __fmul_rn(w, w)));
  n = fmaxf(n, 1e-9f);
  qz = __fdiv_rn(z, n);
  qw = __fdiv_rn(w, n);
}

// Per-axis terms of quat_apply(q_yaw, (bx,by,0)) in the reference's op order, each product
// rounded on its own (never contracted):  t = 2 (q_v x b);  out = (b + w t) + q_v x t.
//   x: rn(rn(bx + AX(by)) + CX(bx)),  AX = rn(qw * tx), tx = -2 rn(qz by),  CX = -rn(qz ty)
//   y: rn(rn(by + AY(bx)) + CY(by)),  AY = rn(qw * ty), ty =  2 rn(qz bx),  CY =  rn(qz tx)
struct ScanAxis {
  float a, c;
};
__device__ __forceinline__ ScanAxis hl_scan_axis_x(float qz, float qw, float bx) {  // indexed by i (x grid)
  const float ty = 2.0f * __fmul_rn(qz, bx);
  ScanAxis r;
  r.a = __fmul_rn(qw, ty);   // AY_i
  r.c = -__fmul_rn(qz, ty);  // CX_i
  return r;
}
__device__ __forceinline__ ScanAxis hl_scan_axis_y(float qz, float qw, float by) {  // indexed by j (y grid)
  const float tx = -2.0f * __fmul_rn(qz, by);
  ScanAxis r;
  r.a = __fmul_rn(qw, tx);  // AX_j
  r.c = __fmul_rn(qz, tx);  // CY_j
  return r;
}

// world point -> clipped cell index: `points += border; (points / hscale).long(); clip`
// (LR:1342-1347).  torch CUDA turns `tensor / python_scalar` into a multiply by the fp32
// reciprocal; torch CPU divides.
__device__ __forceinline__ int hl_cell(const HlCfg& c, float world, int hi) {
  const float p = __fadd_rn(world, c.border_size);
  const float g = (c.index_math == HL_INDEX_MATH_TORCH_CPU) ? __fdiv_rn(p, c.horizontal_scale)
                                                            : __fmul_rn(p, c.inv_horizontal_scale);
  long long i = (long long)g;  // truncation toward zero, like Tensor.long()
  i = i < 0 ? 0 : (i > hi ? hi : i);
  return (int)i;
}

__device__ __forceinline__ int hl_sample_min3(const HlCfg& c, const HlEnvBuffers& b, int px, int py) {
  if (b.height_min3) return (int)__ldg(b.height_min3 + (size_t)px * (c.terrain_cols - 1) + py);
  const int16_t* h = b.height_samples + (size_t)px * c.terrain_cols + py;  // LR:1349-1353
  const int h1 = __ldg(h), h2 = __ldg(h + c.terrain_cols), h3 = __ldg(h + 1);
  return min(min(h1, h2), h3);
}

// raw (int16 units) height under body-frame point (bxv, byv) of an env at (posx, posy)
__device__ __forceinline__ int hl_scan_point(const HlCfg& c, const HlEnvBuffers& b, float posx, float posy,
                                             float bxv, float byv, ScanAxis ax_i, ScanAxis ax_j, int* pxo,
                                             int* pyo) {
  const float rx = __fadd_rn(__fadd_rn(bxv, ax_j.a), ax_i.c);
  const float ry = __fadd_rn(__fadd_rn(byv, ax_i.a), ax_j.c);
  const int px = hl_cell(c, __fadd_rn(rx, posx), c.terrain_rows - 2);
  const int py = hl_cell(c, __fadd_rn(ry, posy), c.terrain_cols - 2);
  if (pxo) { *pxo = px; *pyo = py; }
  return hl_sample_min3(c, b, px, py);
}

// ----------------------------------------------------------------------------- termination
__device__ __forceinline__ float hl_norm3(const float* p) { return sqrtf(p[0] * p[0] + p[1] * p[1] + p[2] * p[2]); }

__device__ __forceinline__ void hl_check_termination(const HlCfg& c, const EnvView& v, EnvScalars& s) {  // LR:249-286
  bool r = false;
  for (int k = 0; k < c.n_term_contact; ++k) r |= hl_norm3(v.cf + c.term_contact_idx[k] * 3) > 1.0f;
  s.time_out = s.ep_len > c.max_episode_length;
  r |= s.time_out;
  if (c.term_base_vel_violate) {
    const float err = s.blv[0] - s.cmd[0];
    bool viol = ((err > 2.0f) && (s.cmd[0] < 0.0f)) || ((err < -2.0f) && (s.cmd[0] > 0.0f));
    r |= viol && (s.terrain_level > 3);
  }
  if (c.term_out_of_border) {  // terrain.py:220-227
    const float x = v.root[0], y = v.root[1];
    r |= !((x >= 0.0f) && (y >= 0.0f) && (x < c.x_limit) && (y < c.y_limit));
  }
  if (c.term_fall_down) r |= v.root[9] < -5.0f;
  s.reset = r;
}

// ----------------------------------------------------------------------------- reward terms
__device__ __forceinline__ float hl_sq(float x) { return x * x; }
__device__ __forceinline__ float hl_up(const EnvScalars& s) { return hl_clampf(-s.pg[2], 0.0f, 1.0f); }
__device__ __forceinline__ float hl_cmd_norm(const EnvScalars& s) { return sqrtf(s.cmd[0] * s.cmd[0] + s.cmd[1] * s.cmd[1]); }

__device__ __forceinline__ float hl_pose(const HlCfg& c, const EnvView& v, int j) {  // LR:1662-1679
  float a = 0.0f;
#pragma unroll
  for (int leg = 0; leg < 4; ++leg) a += fabsf(v.dof_pos(leg * 3 + j) - c.default_dof_pos[leg * 3 + j]);
  return a;
}

// foot f position / velocity relative to the base, rotated into the body frame (LR:1612-1616,1685-1692)
__device__ __forceinline__ void hl_foot_body(const EnvView& v, int f, bool vel, float* o) {
  const float* p = vel ? v.fvel[f] : v.fpos[f];
  const int ro = vel ? 7 : 0;
  hl_quat_rotate_inverse(v.root + 3, p[0] - v.root[ro], p[1] - v.root[ro + 1], p[2] - v.root[ro + 2], o);
}

__device__ __forceinline__ float hl_stumble(const HlCfg& c, const EnvView& v, const EnvScalars& s, float factor) {  // LR:1589-1608
  bool any = false;
#pragma unroll
  for (int f = 0; f < 4; ++f) {
    const float* p = v.cf + c.feet_idx[f] * 3;
    any |= sqrtf(p[0] * p[0] + p[1] * p[1]) > factor * fabsf(p[2]);
  }
  const bool in_slice = (s.gid >= c.stairsup_start && s.gid < c.stairsup_end) || (s.gid >= c.pit_start && s.gid < c.gap_end);
  return (any && s.terrain_level > 3 && in_slice) ? 1.0f : 0.0f;
}

__device__ __forceinline__ float hl_var12(const float* x) {  // torch.var(dim=1), unbiased
  float m = 0.0f;
#pragma unroll
  for (int d = 0; d < 12; ++d) m += x[d];
  m *= (1.0f / 12.0f);
  float q = 0.0f;
#pragma unroll
  for (int d = 0; d < 12; ++d) q += hl_sq(x[d] - m);
  return q / 11.0f;
}

__device__ float hl_foot_clearance_terrain(const HlCfg& c, const HlEnvBuffers& b, const EnvView& v, EnvScalars& s) {  // LR:1717-1743
  float acc = 0.0f;
  if (c.mesh_type != 0) s.feet_shift += 1;  // in-place `points += border` on self.feet_pos
#pragma unroll
  for (int f = 0; f < 4; ++f) {
    float fh;
    if (c.mesh_type == 0) {
      fh = v.fpos[f][2];
    } else {
      // the shifted feet_pos is what gets divided (no second +border: the in-place add already
      // happened); coordinates may have been shifted by an earlier foot_clearance_terrain* term
      float sx = v.fpos[f][0], sy = v.fpos[f][1], sz = v.fpos[f][2];
      for (int k = 0; k < s.feet_shift; ++k) {
        sx = __fadd_rn(sx, c.border_size);
        sy = __fadd_rn(sy, c.border_size);
        sz = __fadd_rn(sz, c.border_size);
      }
      const float gx = (c.index_math == HL_INDEX_MATH_TORCH_CPU) ? __fdiv_rn(sx, c.horizontal_scale) : __fmul_rn(sx, c.inv_horizontal_scale);
      const float gy = (c.index_math == HL_INDEX_MATH_TORCH_CPU) ? __fdiv_rn(sy, c.horizontal_scale) : __fmul_rn(sy, c.inv_horizontal_scale);
      long long ix = (long long)gx, iy = (long long)gy;
      ix = ix < 0 ? 0 : (ix > c.terrain_rows - 2 ? c.terrain_rows - 2 : ix);
      iy = iy < 0 ? 0 : (iy > c.terrain_cols - 2 ? c.terrain_cols - 2 : iy);
      fh = sz - __fmul_rn((float)hl_sample_min3(c, b, (int)ix, (int)iy), c.vertical_scale);   // LR:1741: `heights * vertical_scale` rounded before the subtraction
    }
    const float lat = sqrtf(hl_sq(v.fvel[f][0]) + hl_sq(v.fvel[f][1]));
    acc += lat * hl_sq(fh - c.foot_height_target_terrain);
  }
  return acc;
}

// One `_reward_<name>()` value for this env (formulas: SURVEY.md A.4 / LR:1444-1770).
// (forceinline: with a compile-time `id` the switch folds to the one case -- see reward_fast in hl_persist_kernel.inc)
__device__ __forceinline__ float hl_eval_term(int id, const HlCfg& c, const HlEnvBuffers& b, const EnvView& v, EnvScalars& s) {
  float r = 0.0f;
  switch (id) {
    case T_action_rate:
      for (int d = 0; d < 12; ++d) r += hl_sq(v.lact[d] - v.act[d]);
      break;
    case T_ang_vel_xy:
    case T_ang_vel_xy_up:
      r = hl_sq(s.bav[0]) + hl_sq(s.bav[1]);
      if (id == T_ang_vel_xy_up) r *= hl_up(s);
      break;
    case T_base_height:
    case T_base_height_up:
      r = hl_sq(s.base_h - c.base_height_target);
      if (id == T_base_height_up) r *= hl_up(s);
      break;
    case T_calf_pose: r = hl_pose(c, v, 2); break;
    case T_calf_pose_up: r = hl_pose(c, v, 2) * hl_up(s); break;
    case T_thigh_pose: r = hl_pose(c, v, 1); break;
    case T_thigh_pose_up: r = hl_pose(c, v, 1) * hl_up(s); break;
    case T_hip_pos: r = hl_pose(c, v, 0); break;
    case T_hip_pos_up: r = hl_pose(c, v, 0) * hl_up(s); break;
    case T_collision:
    case T_collision_up:
      for (int k = 0; k < c.n_penalised; ++k) r += hl_norm3(v.cf + c.penalised_idx[k] * 3) > 0.1f ? 1.0f : 0.0f;
      if (id == T_collision_up) r *= hl_up(s);
      break;
    case T_dof_acc:
    {  // LR:1513-1515: ((last_dof_vel - dof_vel) / dt)^2; x * (1/dt) differs from x / dt by at most 1 ulp (12 IEEE
       // divisions were 8 % of the scalar chain)
      const float inv_dt = 1.0f / c.dt;
      for (int d = 0; d < 12; ++d) r += hl_sq((v.ldv[d] - v.dof_vel(d)) * inv_dt);
      break;
    }
    case T_dof_pos_dif:
      for (int d = 0; d < 12; ++d) r += hl_sq(v.ldp[d] - v.dof_pos(d));
      break;
    case T_dof_pos_limits:
      for (int d = 0; d < 12; ++d)
        r += -fminf(v.dof_pos(d) - c.dof_pos_lo[d], 0.0f) + fmaxf(v.dof_pos(d) - c.dof_pos_hi[d], 0.0f);
      break;
    case T_dof_vel:
      for (int d = 0; d < 12; ++d) r += hl_sq(v.dof_vel(d));
      break;
    case T_dof_vel_limits:
      for (int d = 0; d < 12; ++d)
        r += hl_clampf(fabsf(v.dof_vel(d)) - c.dof_vel_limits[d] * c.soft_dof_vel_limit, 0.0f, 1.0f);
      break;
    case T_feet_air_time: {  // LR:1459-1470; stateful; sees the already-updated last_contacts
      const unsigned filt = s.contact | s.last_contact;
      s.last_contact = s.contact;
#pragma unroll
      for (int f = 0; f < 4; ++f) {
        const bool fc = (filt >> f) & 1u;
        const bool first = (s.air[f] > 0.0f) && fc;
        s.air[f] += c.dt;
        r += (s.air[f] - 0.5f) * (first ? 1.0f : 0.0f);
        s.air[f] *= fc ? 0.0f : 1.0f;
      }
      r *= hl_cmd_norm(s) > 0.1f ? 1.0f : 0.0f;
    } break;
    case T_feet_contact_forces:
      for (int f = 0; f < 4; ++f) r += fmaxf(hl_norm3(v.cf + c.feet_idx[f] * 3) - c.max_contact_force, 0.0f);
      break;
    case T_feet_mirror:
    case T_feet_mirror_up: {
      const float d1 = hl_sq(v.dof_pos(1) - v.dof_pos(10)) + hl_sq(v.dof_pos(2) - v.dof_pos(11));
      const float d2 = hl_sq(v.dof_pos(4) - v.dof_pos(7)) + hl_sq(v.dof_pos(5) - v.dof_pos(8));
      r = 0.5f * (d1 + d2);
      if (id == T_feet_mirror_up) r *= hl_up(s);
    } break;
    case T_feet_slide:
    case T_feet_slide_up:
      for (int f = 0; f < 4; ++f) {
        float o[3];
        hl_foot_body(v, f, true, o);
        r += (((s.cfilt >> f) & 1u) ? 1.0f : 0.0f) * sqrtf(hl_sq(o[0]) + hl_sq(o[1]));
      }
      if (id == T_feet_slide_up) r *= hl_up(s);
      break;
    case T_feet_stumble: r = hl_stumble(c, v, s, 5.0f); break;
    case T_feet_stumble_up: r = hl_stumble(c, v, s, 4.0f) * hl_up(s); break;
    case T_foot_clearance_base:
    case T_foot_clearance_base_up:
      for (int f = 0; f < 4; ++f) {
        float p[3], o[3];
        hl_foot_body(v, f, false, p);
        hl_foot_body(v, f, true, o);
        r += hl_sq(p[2] - c.foot_height_target_base) * sqrtf(hl_sq(o[0]) + hl_sq(o[1]));
      }
      if (id == T_foot_clearance_base_up) r *= hl_up(s);
      break;
    case T_foot_clearance_terrain: r = hl_foot_clearance_terrain(c, b, v, s); break;
    case T_foot_clearance_terrain_up: r = hl_foot_clearance_terrain(c, b, v, s) * hl_up(s); break;
    case T_has_contact:
      r = (hl_cmd_norm(s) < 0.1f ? 1.0f : 0.0f) * (float)__popc(s.cfilt & 0xFu) / 4.0f;
      break;
    case T_hip_action_magnitude:
      for (int leg = 0; leg < 4; ++leg) r += hl_sq(fmaxf(fabsf(v.act[leg * 3]) - 1.0f, 0.0f));
      break;
    case T_joint_power:
      for (int d = 0; d < 12; ++d) r += fabsf(v.dof_vel(d)) * fabsf(v.tq[d]);
      break;
    case T_lin_vel_z: r = hl_sq(s.blv[2]); break;
    case T_lin_vel_z_up: r = hl_sq(s.blv[2]) * hl_up(s); break;
    case T_orientation: r = hl_sq(s.pg[0]) + hl_sq(s.pg[1]); break;
    case T_orientation_up: r = (hl_sq(s.pg[0]) + hl_sq(s.pg[1])) * hl_up(s); break;
    case T_power:
      for (int d = 0; d < 12; ++d) r += fabsf(v.tq[d] * v.dof_vel(d));
      break;
    case T_power_distribution: {
      float x[12];
      for (int d = 0; d < 12; ++d) x[d] = fabsf(v.tq[d] * v.dof_vel(d));
      r = hl_var12(x);
    } break;
    case T_smoothness:
      for (int d = 0; d < 12; ++d) r += hl_sq(v.act[d] - v.lact[d] - v.lact[d] + v.llact[d]);
      break;
    case T_stand_nice:
    case T_stand_still:
      for (int d = 0; d < 12; ++d) r += fabsf(v.dof_pos(d) - c.default_dof_pos[d]);
      r *= hl_cmd_norm(s) < 0.1f ? 1.0f : 0.0f;
      if (id == T_stand_nice) r *= 1.0f - s.pg[2];
      break;
    case T_stuck: r = (fabsf(s.blv[0]) < 0.1f && fabsf(s.cmd[0]) > 0.1f) ? 1.0f : 0.0f; break;
    case T_termination: r = (s.reset && !s.time_out) ? 1.0f : 0.0f; break;
    case T_torque_limits:
      for (int d = 0; d < 12; ++d) r += fmaxf(fabsf(v.tq[d]) - c.torque_limits[d] * c.soft_torque_limit, 0.0f);
      break;
    case T_torques:
      for (int d = 0; d < 12; ++d) r += hl_sq(v.tq[d]);
      break;
    case T_torques_dif:
      for (int d = 0; d < 12; ++d) r += hl_sq(v.tq[d] - v.ltq[d]);
      break;
    case T_torques_distribution: {
      float x[12];
      for (int d = 0; d < 12; ++d) x[d] = fabsf(v.tq[d]);
      r = hl_var12(x);
    } break;
    case T_tracking_ang_vel: r = expf(-hl_sq(s.cmd[2] - s.bav[2]) / c.tracking_sigma); break;
    case T_tracking_lin_vel: {
      const float keep = hl_cmd_norm(s) < 0.1f ? 0.0f : 1.0f;
      r = expf(-(hl_sq(s.cmd[0] * keep - s.blv[0]) + hl_sq(s.cmd[1] * keep - s.blv[1])) / c.tracking_sigma);
    } break;
    case T_upward: r = 1.0f - s.pg[2]; break;
    default: break;
  }
  return r;
}

// compute_reward() for one env (LR:363-380).  `sums` points at this env's column of the (R, n)
// episode-sums matrix (row stride n).
// `write` = this thread owns the stores.
template <typename IndexT>
__device__ __forceinline__ float hl_compute_reward(const HlCfg& c, const HlEnvBuffers& b, const EnvView& v, EnvScalars& s,
                                                   float* sums, IndexT n, bool write) {
  float rew = 0.0f;
  const bool acc = write && sums;
  for (int k = 0; k < c.n_terms; ++k) {
    const float r = hl_eval_term(c.term_id[k], c, b, v, s) * c.term_scale[k];
    rew += r;
    if (acc) sums[(IndexT)k * n] += r;
  }
  if (c.only_positive_rewards) rew = fmaxf(rew, 0.0f);
  if (c.has_termination_term) {
    const float r = ((s.reset && !s.time_out) ? 1.0f : 0.0f) * c.termination_scale;
    rew += r;
    if (acc) sums[(IndexT)c.n_terms * n] += r;
  }
  return rew;
}

__device__ __forceinline__ float4 hl_lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }

// ----------------------------------------------------------------------------- compile-time reward lists
__host__ __device__ constexpr unsigned long long hl_tbit(int t) { return 1ull << t; }
constexpr unsigned long long HL_MASK_COMMON =
    hl_tbit(T_action_rate) | hl_tbit(T_ang_vel_xy) | hl_tbit(T_base_height) | hl_tbit(T_calf_pose) | hl_tbit(T_dof_acc) | hl_tbit(T_feet_air_time) |
    hl_tbit(T_feet_contact_forces) | hl_tbit(T_feet_slide) | hl_tbit(T_hip_pos) | hl_tbit(T_joint_power) | hl_tbit(T_lin_vel_z) |
    hl_tbit(T_orientation) | hl_tbit(T_stand_still) | hl_tbit(T_stuck) | hl_tbit(T_thigh_pose) | hl_tbit(T_torques) | hl_tbit(T_tracking_ang_vel) |
    hl_tbit(T_tracking_lin_vel);
// aliengo flat / AMP (aliengo_config.py:217-256): 21 terms
constexpr unsigned long long HL_MASK_FLAT = HL_MASK_COMMON | hl_tbit(T_feet_mirror) | hl_tbit(T_foot_clearance_base) | hl_tbit(T_smoothness);
// aliengo_stairs (aliengo_stairs_config.py:171-210): 20 terms (+ termination, added after the loop)
constexpr unsigned long long HL_MASK_STAIRS = HL_MASK_COMMON | hl_tbit(T_collision) | hl_tbit(T_feet_stumble);
__host__ __device__ constexpr int hl_popc64(unsigned long long x) { int c = 0; while (x) { x &= x - 1; ++c; } return c; }

// compute_reward() (LR:363-380) for one env with the active terms known at compile time: no
// dispatch, the per-DOF terms share one pass over the rows (128-bit shared-memory loads), the rest is
// hl_eval_term with a constant id.  Same per-term op order as hl_eval_term; same alphabetical
// accumulation.  `es` = this env's column of the (R, N) episode sums (row stride n) or NULL: each scaled term
// is added by a fire-and-forget red.global.add.f32 -- one IEEE add per element per step by a single thread, so the
// result is the same `sum += term` (LR:371) without a load, a register or a wait.
template <unsigned long long M>
__device__ __forceinline__ float hl_reward_fast(const HlCfg& c, const HlEnvBuffers& b, const EnvView& v, EnvScalars& s, float* es, long long n) {
#define HAS(t) ((M >> (t)) & 1ull)
  float a_rate = 0.f, a_acc = 0.f, a_pow = 0.f, a_smooth = 0.f, a_tq = 0.f, a_pose0 = 0.f, a_pose1 = 0.f, a_pose2 = 0.f, a_stand = 0.f;
  {
    const float inv_dt = 1.0f / c.dt;
#pragma unroll
    for (int g = 0; g < 3; ++g) {
      const float4 d0 = hl_lds4(v.dof + 8 * g), d1 = hl_lds4(v.dof + 8 * g + 4);
      const float q[4] = {d0.x, d0.z, d1.x, d1.z}, qd[4] = {d0.y, d0.w, d1.y, d1.w};
      float a[4] = {0.f, 0.f, 0.f, 0.f}, la[4] = {0.f, 0.f, 0.f, 0.f}, lla[4] = {0.f, 0.f, 0.f, 0.f}, lv[4] = {0.f, 0.f, 0.f, 0.f},
            tq[4] = {0.f, 0.f, 0.f, 0.f};
      if (HAS(T_action_rate) || HAS(T_smoothness)) {
        const float4 x = hl_lds4(v.act + 4 * g), y = hl_lds4(v.lact + 4 * g);
        a[0] = x.x; a[1] = x.y; a[2] = x.z; a[3] = x.w;
        la[0] = y.x; la[1] = y.y; la[2] = y.z; la[3] = y.w;
      }
      if (HAS(T_smoothness)) {
        const float4 x = hl_lds4(v.llact + 4 * g);
        lla[0] = x.x; lla[1] = x.y; lla[2] = x.z; lla[3] = x.w;
      }
      if (HAS(T_dof_acc)) {
        const float4 x = hl_lds4(v.ldv + 4 * g);
        lv[0] = x.x; lv[1] = x.y; lv[2] = x.z; lv[3] = x.w;
      }
      if (HAS(T_joint_power) || HAS(T_torques)) {
        const float4 x = hl_lds4(v.tq + 4 * g);
        tq[0] = x.x; tq[1] = x.y; tq[2] = x.z; tq[3] = x.w;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int d = 4 * g + i;
        if (HAS(T_action_rate)) a_rate += hl_sq(la[i] - a[i]);
        if (HAS(T_dof_acc)) a_acc += hl_sq((lv[i] - qd[i]) * inv_dt);
        if (HAS(T_joint_power)) a_pow += fabsf(qd[i]) * fabsf(tq[i]);
        if (HAS(T_smoothness)) a_smooth += hl_sq(a[i] - la[i] - la[i] + lla[i]);
        if (HAS(T_torques)) a_tq += hl_sq(tq[i]);
        const float dev = fabsf(q[i] - c.default_dof_pos[d]);
        if (HAS(T_stand_still) || HAS(T_stand_nice)) a_stand += dev;
        if (d % 3 == 0) { if (HAS(T_hip_pos) || HAS(T_hip_pos_up)) a_pose0 += dev; }
        else if (d % 3 == 1) { if (HAS(T_thigh_pose) || HAS(T_thigh_pose_up)) a_pose1 += dev; }
        else { if (HAS(T_calf_pose) || HAS(T_calf_pose_up)) a_pose2 += dev; }
      }
    }
  }
  float rew = 0.0f;
#define EMIT(t, val)                                            \
  if (HAS(t)) {                                                 \
    constexpr int k_ = hl_popc64(M & (hl_tbit(t) - 1ull));            \
    const float r_ = (val) * c.term_scale[k_];                  \
    rew += r_;                                                  \
    if (es) atomicAdd(es + (long long)k_ * n, r_);              \
  }
#define EVAL(t) EMIT(t, hl_eval_term(t, c, b, v, s))
  EMIT(T_action_rate, a_rate)
  EVAL(T_ang_vel_xy) EVAL(T_ang_vel_xy_up) EVAL(T_base_height) EVAL(T_base_height_up)
  EMIT(T_calf_pose, a_pose2)
  EMIT(T_calf_pose_up, a_pose2 * hl_up(s))
  EVAL(T_collision) EVAL(T_collision_up)
  EMIT(T_dof_acc, a_acc)
  EVAL(T_dof_pos_dif) EVAL(T_dof_pos_limits) EVAL(T_dof_vel) EVAL(T_dof_vel_limits) EVAL(T_feet_air_time)
  EVAL(T_feet_contact_forces) EVAL(T_feet_mirror) EVAL(T_feet_mirror_up) EVAL(T_feet_slide) EVAL(T_feet_slide_up)
  EVAL(T_feet_stumble) EVAL(T_feet_stumble_up) EVAL(T_foot_clearance_base) EVAL(T_foot_clearance_base_up)
  EVAL(T_foot_clearance_terrain) EVAL(T_foot_clearance_terrain_up) EVAL(T_has_contact) EVAL(T_hip_action_magnitude)
  EMIT(T_hip_pos, a_pose0)
  EMIT(T_hip_pos_up, a_pose0 * hl_up(s))
  EMIT(T_joint_power, a_pow)
  EVAL(T_lin_vel_z) EVAL(T_lin_vel_z_up) EVAL(T_orientation) EVAL(T_orientation_up) EVAL(T_power) EVAL(T_power_distribution)
  EMIT(T_smoothness, a_smooth)
  EMIT(T_stand_nice, a_stand * (hl_cmd_norm(s) < 0.1f ? 1.0f : 0.0f) * (1.0f - s.pg[2]))
  EMIT(T_stand_still, a_stand * (hl_cmd_norm(s) < 0.1f ? 1.0f : 0.0f))
  EVAL(T_stuck)
  EMIT(T_thigh_pose, a_pose1)
  EMIT(T_thigh_pose_up, a_pose1 * hl_up(s))
  EVAL(T_torque_limits)
  EMIT(T_torques, a_tq)
  EVAL(T_torques_dif) EVAL(T_torques_distribution) EVAL(T_tracking_ang_vel) EVAL(T_tracking_lin_vel) EVAL(T_upward)
#undef EVAL
#undef EMIT
#undef HAS
  if (c.only_positive_rewards) rew = fmaxf(rew, 0.0f);
  if (c.has_termination_term) {
    const float r = ((s.reset && !s.time_out) ? 1.0f : 0.0f) * c.termination_scale;
    rew += r;
    if (es) atomicAdd(es + (long long)hl_popc64(M) * n, r);
  }
  return rew;
}


__device__ __forceinline__ bool hl_needs_base_height(const HlCfg& c) {
  bool need = false;
  for (int k = 0; k < c.n_terms; ++k) need |= (c.term_id[k] == T_base_height) | (c.term_id[k] == T_base_height_up);
  return need;
}

// ----------------------------------------------------------------------------- observations
// element k (0..44) of the one-step observation before noise (LR:385-391)
__device__ __forceinline__ float hl_obs45(const HlCfg& c, const EnvView& v, const EnvScalars& s, int k) {
  if (k < 3) return s.cmd[k] * c.commands_scale[k];
  if (k < 6) return s.bav[k - 3] * c.obs_ang_vel;
  if (k < 9) return s.pg[k - 6];
  if (k < 21) return (v.dof_pos(k - 9) - c.default_dof_pos[k - 9]) * c.obs_dof_pos;
  if (k < 33) return v.dof_vel(k - 21) * c.obs_dof_vel;
  return v.act[k - 33];
}
// element p of the height part (LR:399-400), u = U[0,1) draw
__device__ __forceinline__ float hl_obs_height(const HlCfg& c, float root_z, float mh, float u) {
  float h = hl_clampf(root_z - 0.5f - mh, -1.0f, 1.0f) * c.obs_height;
  if (c.add_noise) h += (2.0f * u - 1.0f) * c.noise_height;
  return h;
}
__device__ __forceinline__ float hl_add_noise45(const HlCfg& c, float x, float u, int k) {  // LR:394
  return c.add_noise ? x + (2.0f * u - 1.0f) * c.noise45[k] : x;
}
