// Post-physics kernels (sm_100a): PD torques, the fused post-physics step, the generic
// per-stage kernel behind the individual drop-in methods, reset-id compaction, terminal rows.
// Reference: legged_gym/legged_gym/envs/base/legged_robot.py (LR) -- see include/himloco_b200.h.
#include <stdarg.h>
#include <stdio.h>

#include "hl_math.cuh"

// ----------------------------------------------------------------------------- error string
static thread_local char g_err[512] = "";
void hl_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* hl_last_error(void) { return g_err; }
bool hl_pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("HL_PDL");
    return !(e && e[0] == '0');
  }();
  return on;
}
extern "C" int hl_version(void) { return HL_VERSION; }
extern "C" int hl_sizeof_cfg(void) { return (int)sizeof(HlCfg); }
extern "C" int hl_sizeof_env_buffers(void) { return (int)sizeof(HlEnvBuffers); }

static int check_cfg(const HlCfg* c, const HlEnvBuffers* b) {
  if (!c || c->struct_bytes != (int)sizeof(HlCfg)) {
    hl_set_error("HlCfg size mismatch (binding %d vs library %d)", c ? c->struct_bytes : -1, (int)sizeof(HlCfg));
    return HL_E_INVALID;
  }
  if (b && b->struct_bytes != (int)sizeof(HlEnvBuffers)) {
    hl_set_error("HlEnvBuffers size mismatch (binding %d vs library %d)", b->struct_bytes, (int)sizeof(HlEnvBuffers));
    return HL_E_INVALID;
  }
  if (c->n_terms < 0 || c->n_terms > HL_MAX_TERMS || c->n_px > HL_MAX_PTS || c->n_py > HL_MAX_PTS ||
      c->n_px * c->n_py > 256 || c->n_bx * c->n_by > 256 || c->num_bodies < 1 || c->n_penalised > HL_MAX_BODIES_IDX ||
      c->n_term_contact > HL_MAX_BODIES_IDX) {
    hl_set_error("HlCfg out of range");
    return HL_E_INVALID;
  }
  return HL_OK;
}

// ============================================================================= a1: PD torques
// LR:658-688.  Three threads per env (one float4 of every 12-wide row each).
struct PdCfg {
  float action_scale, hip_reduction, sim_dt;
  int control_type;
  float p_gains[12], d_gains[12], torque_limits[12], default_dof_pos[12];
};
__device__ __forceinline__ float pd_one(const PdCfg& c, int d, float action, float ms, float pos, float vel, float kp,
                                        float kd, float last_vel, float* target) {
  float scaled = (ms * action) * c.action_scale;
  if (d % 3 == 0) scaled *= c.hip_reduction;  // columns [0,3,6,9]
  *target = c.default_dof_pos[d] + scaled;
  float tq;
  if (c.control_type == 0) tq = c.p_gains[d] * kp * (*target - pos) - c.d_gains[d] * kd * vel;
  else if (c.control_type == 1) tq = c.p_gains[d] * (scaled - vel) - c.d_gains[d] * (vel - last_vel) / c.sim_dt;
  else tq = scaled;
  return hl_clampf(tq, -c.torque_limits[d], c.torque_limits[d]);
}
__global__ void __launch_bounds__(192) hl_pd_torque_vec_kernel(PdCfg c, const float* __restrict__ actions, long long a_stride,
                                                               const float4* __restrict__ dof_state,
                                                               const float4* __restrict__ motor_strength,
                                                               const float* __restrict__ kp, const float* __restrict__ kd,
                                                               const float4* __restrict__ last_dof_vel, float4* __restrict__ out,
                                                               float4* __restrict__ target_out, long long n) {
  // three threads per env, one leg-and-a-third (4 dofs = one float4 of every 12-wide row) each:
  // 5 independent 128-bit loads in flight per thread, 196,608 threads for 65,536 envs
  hl_pdl_enter();
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * 3) return;
  const long long e = t / 3;
  const int j = (int)(t - e * 3);
  const float4 a = __ldg(reinterpret_cast<const float4*>(actions + e * a_stride) + j);
  const float4 m = __ldg(motor_strength + t);
  const float4 dv0 = __ldg(dof_state + 2 * t), dv1 = __ldg(dof_state + 2 * t + 1);
  const float4 lv = c.control_type == 1 ? __ldg(last_dof_vel + t) : make_float4(0.f, 0.f, 0.f, 0.f);
  const float kpe = __ldg(kp + e), kde = __ldg(kd + e);
  const float af[4] = {a.x, a.y, a.z, a.w}, mf[4] = {m.x, m.y, m.z, m.w}, lf[4] = {lv.x, lv.y, lv.z, lv.w};
  const float pos[4] = {dv0.x, dv0.z, dv1.x, dv1.z}, vel[4] = {dv0.y, dv0.w, dv1.y, dv1.w};
  float tq[4], tg[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    // dof d = 4j + i; its constants picked with selects on j (uniform constant-bank operands)
    float r;
    if (j == 0) r = pd_one(c, i, af[i], mf[i], pos[i], vel[i], kpe, kde, lf[i], &tg[i]);
    else if (j == 1) r = pd_one(c, 4 + i, af[i], mf[i], pos[i], vel[i], kpe, kde, lf[i], &tg[i]);
    else r = pd_one(c, 8 + i, af[i], mf[i], pos[i], vel[i], kpe, kde, lf[i], &tg[i]);
    tq[i] = r;
  }
  out[t] = make_float4(tq[0], tq[1], tq[2], tq[3]);
  if (target_out) target_out[t] = make_float4(tg[0], tg[1], tg[2], tg[3]);
}
// fallback for unaligned / oddly strided action views: one thread per (env, dof)
__global__ void __launch_bounds__(256) hl_pd_torque_kernel(PdCfg c, const float* __restrict__ actions, long long a_stride,
                                                           const float2* __restrict__ dof_state,
                                                           const float* __restrict__ motor_strength,
                                                           const float* __restrict__ kp, const float* __restrict__ kd,
                                                           const float* __restrict__ last_dof_vel,
                                                           float* __restrict__ out, float* __restrict__ target_out,
                                                           long long total) {
  hl_pdl_enter();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long e = i / 12;
  const int d = (int)(i - e * 12);
  const float2 pv = dof_state[i];
  float tg;
  out[i] = pd_one(c, d, actions[e * a_stride + d], motor_strength[i], pv.x, pv.y, kp[e], kd[e],
                  c.control_type == 1 ? last_dof_vel[i] : 0.0f, &tg);
  if (target_out) target_out[i] = tg;
}

extern "C" int hl_pd_torque(const HlCfg* cfg, const float* actions, int64_t a_stride, const float* dof_state,
                            const float* motor_strength, const float* kp, const float* kd, const float* last_dof_vel,
                            float* torques_out, float* target_out, int64_t n, void* stream) {
  if (int r = check_cfg(cfg, nullptr)) return r;
  HL_CHECK_ARG(actions && dof_state && motor_strength && kp && kd && torques_out, "null pointer");
  HL_CHECK_ARG(cfg->control_type != 1 || last_dof_vel, "control_type V needs last_dof_vel");
  if (n <= 0) return HL_OK;
  PdCfg pc;
  pc.action_scale = cfg->action_scale;
  pc.hip_reduction = cfg->hip_reduction;
  pc.sim_dt = cfg->sim_dt;
  pc.control_type = cfg->control_type;
  for (int d = 0; d < 12; ++d) {
    pc.p_gains[d] = cfg->p_gains[d];
    pc.d_gains[d] = cfg->d_gains[d];
    pc.torque_limits[d] = cfg->torque_limits[d];
    pc.default_dof_pos[d] = cfg->default_dof_pos[d];
  }
  auto al16 = [](const void* p) { return ((uintptr_t)p & 15) == 0; };
  const bool vec = al16(actions) && (a_stride % 4 == 0) && al16(dof_state) && al16(motor_strength) && al16(torques_out) &&
                   (!target_out || al16(target_out)) && (!last_dof_vel || al16(last_dof_vel));
  if (vec) {
    hl_launch(hl_pd_torque_vec_kernel, dim3((unsigned)((n * 3 + 191) / 192)), dim3(192), 0, (cudaStream_t)stream,
        pc, actions, a_stride, (const float4*)dof_state, (const float4*)motor_strength, kp, kd, (const float4*)last_dof_vel,
        (float4*)torques_out, (float4*)target_out, n);
  } else {
    const long long total = n * 12;
    hl_launch(hl_pd_torque_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, (cudaStream_t)stream,
        pc, actions, a_stride, (const float2*)dof_state, motor_strength, kp, kd, last_dof_vel, torques_out, target_out, total);
  }
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= terrain min3 table
__global__ void hl_terrain_min3_kernel(const int16_t* __restrict__ h, int rows, int cols, int16_t* __restrict__ out) {
  const int y = blockIdx.x * blockDim.x + threadIdx.x, x = blockIdx.y;
  if (y >= cols - 1 || x >= rows - 1) return;
  const int a = h[(size_t)x * cols + y], b = h[(size_t)(x + 1) * cols + y], c = h[(size_t)x * cols + y + 1];
  out[(size_t)x * (cols - 1) + y] = (int16_t)min(min(a, b), c);
}
extern "C" int hl_terrain_prepare(const int16_t* hs, int32_t rows, int32_t cols, int16_t* out, void* stream) {
  HL_CHECK_ARG(hs && out && rows >= 2 && cols >= 2, "bad terrain");
  dim3 grid((cols - 1 + 255) / 256, rows - 1);
  hl_terrain_min3_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(hs, rows, cols, out);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

__global__ void hl_terrain_min3f_kernel(const int16_t* __restrict__ h, int rows, int cols, float vs, float* __restrict__ out) {
  const int y = blockIdx.x * blockDim.x + threadIdx.x, x = blockIdx.y;
  if (y >= cols - 1 || x >= rows - 1) return;
  const int a = h[(size_t)x * cols + y], b = h[(size_t)(x + 1) * cols + y], c = h[(size_t)x * cols + y + 1];
  out[(size_t)x * (cols - 1) + y] = __fmul_rn((float)min(min(a, b), c), vs);   // LR:1355 `heights * vertical_scale`
}
extern "C" int hl_terrain_prepare_f32(const int16_t* hs, int32_t rows, int32_t cols, float vertical_scale, float* out, void* stream) {
  HL_CHECK_ARG(hs && out && rows >= 2 && cols >= 2, "bad terrain");
  dim3 grid((cols - 1 + 255) / 256, rows - 1);
  hl_terrain_min3f_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(hs, rows, cols, vertical_scale, out);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// SM count of the current device (cached per device id)
static int device_sms() {
  static int cache[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  int v = cache[dev];
  if (!v) {
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    cache[dev] = v;   // benign race: every thread computes the same value
  }
  return v;
}

// ============================================================================= shared pieces
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Height-scan noise: one Philox block per lane per pass = the uniforms of THAT lane's points in
// iterations 4*pass .. 4*pass+3 (point 32*it + lane takes component it&3 of block pass*32+lane).
struct HeightNoise {
  uint4 blk;
  __device__ __forceinline__ void refill(const HlEnvBuffers& b, uint64_t step, unsigned long long genv, int pass, int lane, unsigned stream) {
    blk = hl_noise_block(b.philox_seed, step, genv, (unsigned)(pass * 32 + lane), stream);
  }
  __device__ __forceinline__ float get(int it, int /*lane*/) const {
    const int cpt = it & 3;
    return hl_u01(cpt == 0 ? blk.x : (cpt == 1 ? blk.y : (cpt == 2 ? blk.z : blk.w)));
  }
};

// Warp-cooperative scans for one env.  `root` = the env's 13-float root record.
// Writes measured_heights (and optionally the height part of privileged_obs + debug indices);
// returns _get_base_heights() when want_base.
struct ScanOut {
  float* measured;     // row of measured_heights or nullptr
  float* priv_heights; // &privileged_obs[e][51] or nullptr
  int32_t* idx;        // debug (P,2) or nullptr
  const float* u187;   // pre-drawn noise row or nullptr
  bool clip;
  float* keep;         // optional: lane-private copy of this lane's heights, keep[it]
};

// it_mod / it_rem: this warp only handles the 32-point iterations with it % it_mod == it_rem (the
// post-reset fix-up spreads one env over several warps); 1 / 0 = all of them.  `step`: the Philox step key.
__device__ __forceinline__ float hl_warp_scan_env(const HlCfg& c, const HlEnvBuffers& b, uint64_t step, const float* root,
                                                  unsigned long long genv, int lane, bool do_heights, bool want_base,
                                                  const ScanOut& o, unsigned noise_stream, int it_mod = 1, int it_rem = 0) {
  float qz, qw;
  hl_yaw_quat(root + 3, qz, qw);
  const float posx = root[0], posy = root[1], posz = root[2];
  float base_h = 0.0f;
  if (do_heights) {
    const int P = c.n_px * c.n_py;
    if (c.mesh_type == 0) {  // plane: zeros (LR:1331-1332)
      HeightNoise hn;
      for (int it = 0; it * 32 < P; ++it) {
        const int p = it * 32 + lane;
        if (o.priv_heights && !o.u187 && (it & 3) == 0) hn.refill(b, step, genv, it >> 2, lane, noise_stream);
        float u = 0.5f;
        if (o.priv_heights && c.add_noise) u = o.u187 ? (p < P ? o.u187[p] : 0.5f) : hn.get(it, lane);
        if (p < P) {
          if (o.measured) o.measured[p] = 0.0f;
          if (o.keep) o.keep[it] = 0.0f;
          if (o.priv_heights) {
            float hv = hl_obs_height(c, posz, 0.0f, u);
            if (o.clip) hv = hl_clampf(hv, -c.clip_obs, c.clip_obs);
            o.priv_heights[p] = hv;
          }
        }
      }
    } else {
      const ScanAxis axi = hl_scan_axis_x(qz, qw, c.px[lane < c.n_px ? lane : 0]);
      const ScanAxis axj = hl_scan_axis_y(qz, qw, c.py[lane < c.n_py ? lane : 0]);
      HeightNoise hn;
      // pass 1: every gather of the env in flight (P <= 256 -> at most 8 per lane); pass 2: outputs
      int hraw[8], pxs[8], pys[8];
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        hraw[it] = 0; pxs[it] = 0; pys[it] = 0;
        if (it * 32 < P && (it % it_mod) == it_rem) {   // warp-uniform
          const int p = it * 32 + lane;
          const int pc = p < P ? p : P - 1;
          const int i = pc / c.n_py, j = pc - i * c.n_py;
          ScanAxis ai, aj;
          ai.a = __shfl_sync(0xffffffffu, axi.a, i);
          ai.c = __shfl_sync(0xffffffffu, axi.c, i);
          aj.a = __shfl_sync(0xffffffffu, axj.a, j);
          aj.c = __shfl_sync(0xffffffffu, axj.c, j);
          hraw[it] = hl_scan_point(c, b, posx, posy, c.px[i], c.py[j], ai, aj, &pxs[it], &pys[it]);
        }
      }
      int pass = -1;
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        if (it * 32 >= P) break;
        if ((it % it_mod) != it_rem) continue;
        const int p = it * 32 + lane;
        const float mh = (float)hraw[it] * c.vertical_scale;
        if (o.priv_heights && !o.u187 && (it >> 2) != pass) { pass = it >> 2; hn.refill(b, step, genv, pass, lane, noise_stream); }
        float u = 0.5f;
        if (o.priv_heights && c.add_noise) u = o.u187 ? (p < P ? o.u187[p] : 0.5f) : hn.get(it, lane);
        if (p < P) {
          if (o.measured) o.measured[p] = mh;
          if (o.keep) o.keep[it] = mh;
          if (o.idx) { o.idx[2 * p] = pxs[it]; o.idx[2 * p + 1] = pys[it]; }
          if (o.priv_heights) {
            float hv = hl_obs_height(c, posz, mh, u);
            if (o.clip) hv = hl_clampf(hv, -c.clip_obs, c.clip_obs);
            o.priv_heights[p] = hv;
          }
        }
      }
    }
  }
  if (want_base) {  // LR:1357-1398
    if (c.mesh_type == 0) {
      base_h = posz;
    } else {
      const int P = c.n_bx * c.n_by;
      const ScanAxis axi = hl_scan_axis_x(qz, qw, c.bx[lane < c.n_bx ? lane : 0]);
      const ScanAxis axj = hl_scan_axis_y(qz, qw, c.by[lane < c.n_by ? lane : 0]);
      float acc = 0.0f;
      for (int it = 0; it * 32 < P; ++it) {
        const int p = it * 32 + lane;
        const int pc = p < P ? p : P - 1;
        const int i = pc / c.n_by, j = pc - i * c.n_by;
        ScanAxis ai, aj;
        ai.a = __shfl_sync(0xffffffffu, axi.a, i);
        ai.c = __shfl_sync(0xffffffffu, axi.c, i);
        aj.a = __shfl_sync(0xffffffffu, axj.a, j);
        aj.c = __shfl_sync(0xffffffffu, axj.c, j);
        const int hraw = hl_scan_point(c, b, posx, posy, c.bx[i], c.by[j], ai, aj, nullptr, nullptr);
        if (p < P) acc += posz - __fmul_rn((float)hraw, c.vertical_scale);   // LR:1396: `heights * vertical_scale` rounded before the subtraction (no FMA)
      }
      base_h = warp_sum(acc) / (float)P;
    }
  }
  return base_h;
}

__device__ __forceinline__ int hl_priv_dim(const HlCfg& c) { return 51 + (c.measure_heights ? c.n_px * c.n_py : 0); }

// ============================================================================= generic stage kernel
// One warp per env (optionally per listed env id); scalars are computed redundantly by all lanes,
// vector work (scan, obs rows) is lane-parallel.  Serves the individual drop-in methods and the
// post-reset fix-up; the hot path is hl_post_physics_fused_kernel below.
// Per-warp staging of one env's records: lane-parallel, coalesced loads that are all in flight
// together (one DRAM round trip), then the per-env math reads shared memory.  Layout (floats):
// root 13 | dof 24 | feet 4 x (pos3, vel3) | act, lact, llact, ldp, ldv, tq, ltq 7 x 12 | cf B*3
constexpr int WS_ROOT = 0, WS_DOF = 13, WS_FEET = 37, WS_A = 61, WS_CF = 145;
__host__ __device__ inline int hl_warp_stage_floats(int num_bodies) { return (WS_CF + num_bodies * 3 + 3) & ~3; }

__device__ __forceinline__ void hl_stage_env(float* st, const HlCfg& c, const HlEnvBuffers& b, long long e, int lane,
                                             bool zero_last, EnvView& v) {
  const int B = c.num_bodies;
  const float r_root = (lane < 13 && b.root_states) ? b.root_states[e * 13 + lane] : 0.0f;
  const float r_dof = (lane < 24 && b.dof_state) ? b.dof_state[e * 24 + lane] : 0.0f;
  float r_feet = 0.0f;
  if (lane < 24 && (b.rigid_body_states || b.foot_records)) {
    const int f = lane / 6, k = lane - f * 6;
    r_feet = hl_foot_rec(c, b, e, f)[k < 3 ? k : k + 4];
  }
  const float* a_src[7] = {b.actions, b.last_actions, b.last_last_actions, b.last_dof_pos, b.last_dof_vel, b.torques, b.last_torques};
  float r_a[7];
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    const bool last = j == 1 || j == 2 || j == 3 || j == 4 || j == 6;   // zeroed by reset_idx (LR:323-329)
    r_a[j] = (lane < 12 && a_src[j] && !(zero_last && last)) ? a_src[j][e * 12 + lane] : 0.0f;
  }
  float r_cf[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) r_cf[j] = (lane + 32 * j < B * 3 && b.contact_forces) ? b.contact_forces[e * B * 3 + lane + 32 * j] : 0.0f;
  if (lane < 13) st[WS_ROOT + lane] = r_root;
  if (lane < 24) st[WS_DOF + lane] = r_dof;
  if (lane < 24) st[WS_FEET + lane] = r_feet;
#pragma unroll
  for (int j = 0; j < 7; ++j)
    if (lane < 12) st[WS_A + 12 * j + lane] = r_a[j];
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (lane + 32 * j < B * 3) st[WS_CF + lane + 32 * j] = r_cf[j];
  for (int i = lane + 128; i < B * 3; i += 32) st[WS_CF + i] = b.contact_forces ? b.contact_forces[e * B * 3 + i] : 0.0f;
  __syncwarp();
  v.root = st + WS_ROOT;
  v.dof = st + WS_DOF;
  v.cf = st + WS_CF;
  for (int f = 0; f < 4; ++f) {
    v.fpos[f] = st + WS_FEET + 6 * f;
    v.fvel[f] = v.fpos[f] + 3;
  }
  v.act = st + WS_A;
  v.lact = st + WS_A + 12;
  v.llact = st + WS_A + 24;
  v.ldp = st + WS_A + 36;
  v.ldv = st + WS_A + 48;
  v.tq = st + WS_A + 60;
  v.ltq = st + WS_A + 72;
}

// ============================================================================= reset_idx re-draws (SURVEY.md §8f rank 2)
// u[k] of one env: column k of its uniform vector (include/himloco_b200.h: HL_RESET_NU).  Philox mode: lane l
// computes block l (four uniforms) of stream `stream`, keyed by (seed, step, global env id); a shuffle hands
// column k to every lane.
struct ResetUniforms {
  uint4 blk;
  const float* row;   // pre-drawn row or nullptr
  __device__ __forceinline__ void init(const HlEnvBuffers& b, uint64_t step, const HlReset& r, long long e, unsigned long long genv, int lane,
                                       unsigned stream) {
    row = r.uniforms ? r.uniforms + e * HL_RESET_NU : nullptr;
    blk = make_uint4(0u, 0u, 0u, 0u);
    if (!row && lane < (HL_RESET_NU + 3) / 4) blk = hl_noise_block(b.philox_seed, step, genv, (unsigned)lane, stream);
  }
  __device__ __forceinline__ float get(int k) const {   // warp-uniform k; every lane of the warp must call
    const unsigned x = __shfl_sync(0xffffffffu, hl_pick(blk, k & 3), k >> 2);
    return row ? row[k] : hl_u01(x);
  }
  __device__ __forceinline__ float range(int k, const float* lohi) const {   // torch_rand_float(lo, hi): (hi - lo) * u + lo
    return (lohi[1] - lohi[0]) * get(k) + lohi[0];
  }
};

// The command ranges of a HlReset as 8 floats (lin_vel_x, lin_vel_y, ang_vel_yaw, heading; lo, hi) in `slot` (shared
// memory): from the device copy when reset.cmd_ranges is set (read after griddepcontrol.wait), else the by-value fields.
// Thread 0 stores; the caller's next __syncthreads publishes them to the CTA.
__device__ __forceinline__ void hl_cmd_ranges_cta(const HlReset& r, float* slot) {
  if (threadIdx.x != 0) return;
  if (r.cmd_ranges) {
#pragma unroll
    for (int k = 0; k < 8; ++k) slot[k] = (float)r.cmd_ranges[k];
  } else {
    slot[0] = r.cmd_lin_vel_x[0]; slot[1] = r.cmd_lin_vel_x[1];
    slot[2] = r.cmd_lin_vel_y[0]; slot[3] = r.cmd_lin_vel_y[1];
    slot[4] = r.cmd_ang_vel_yaw[0]; slot[5] = r.cmd_ang_vel_yaw[1];
    slot[6] = r.cmd_heading[0]; slot[7] = r.cmd_heading[1];
  }
}

// _resample_commands for one env (LR:634-656); lane 0 stores.  cr: the CTA's command ranges (hl_cmd_ranges_cta)
__device__ __forceinline__ void hl_resample_env(const HlReset& r, const float* cr, const ResetUniforms& ru, long long e, long long gid, int lane) {
  float c0 = (1.0f - (-1.0f)) * ru.get(36) + (-1.0f);            // LR:641
  float c1 = ru.range(37, cr + 2);                                 // LR:642
  const float c3 = ru.range(38, r.heading_command ? cr + 6 : cr + 4);   // LR:643-646
  const float hv = ru.range(39, cr);
  if (gid < r.high_vel_envs) {   // LR:649-653 (env_ids < num_envs * 0.2)
    c0 = hv;
    c1 *= fabsf(c0) < 1.0f ? 1.0f : 0.0f;     // norm of a 1-vector
  }
  const float keep = sqrtf(c0 * c0 + c1 * c1) > 0.2f ? 1.0f : 0.0f;   // LR:656
  c0 *= keep;
  c1 *= keep;
  if (lane == 0) {
    r.commands[e * 4 + 0] = c0;
    r.commands[e * 4 + 1] = c1;
    r.commands[e * 4 + (r.heading_command ? 3 : 2)] = c3;
  }
}

// reset_idx for env e, the part that draws: terrain curriculum, dofs, root state, commands, gain factors
// (LR:301-320,336-341).  Warp-cooperative: lanes 0-11 own one dof each, lane 0 the scalars.
__device__ __forceinline__ void hl_reset_draw_env(const HlCfg& c, const HlEnvBuffers& b, uint64_t step, const HlReset& r, const float* cr,
                                                  long long e, int lane) {
  const long long gid = e + c.env_id_offset;
  ResetUniforms ru;
  ru.init(b, step, r, e, (unsigned long long)gid, lane, 3u);
  const unsigned parts = r.parts ? (unsigned)r.parts : 0xffffffffu;
  // ---- _update_terrain_curriculum (LR:845-866): pre-reset root position and commands
  if ((parts & HL_RESET_CURRICULUM) && r.terrain_curriculum && r.terrain_origins && r.terrain_types) {
    const float dx = r.root_states[e * 13 + 0] - r.env_origins[e * 3 + 0], dy = r.root_states[e * 13 + 1] - r.env_origins[e * 3 + 1];
    const float dist = sqrtf(dx * dx + dy * dy);
    const float cx = r.commands[e * 4 + 0], cy = r.commands[e * 4 + 1];
    const bool up = dist > r.env_length / 2.0f;
    const bool down = (dist < sqrtf(cx * cx + cy * cy) * r.max_episode_length_s * 0.5f) && !up;
    long long lvl = r.terrain_levels[e] + (up ? 1 : 0) - (down ? 1 : 0);
    const float ul = ru.get(43);
    if (lvl >= r.max_terrain_level) {
      long long rl = (long long)(ul * (float)r.max_terrain_level);   // torch.randint_like(levels, max_terrain_level)
      lvl = rl < r.max_terrain_level ? rl : r.max_terrain_level - 1;
    } else if (lvl < 0) {
      lvl = 0;
    }
    __syncwarp();
    if (lane == 0) r.terrain_levels[e] = lvl;
    if (lane < 3) r.env_origins[e * 3 + lane] = r.terrain_origins[(lvl * r.n_terrain_types + r.terrain_types[e]) * 3 + lane];
    __syncwarp();
  }
  // ---- _reset_dofs (LR:690-716)
  if (parts & HL_RESET_DOFS) {
    float ratio = 1.0f, vel = 0.0f;
#pragma unroll
    for (int d = 0; d < 12; ++d) {
      const float ud = ru.get(d), uv = ru.get(12 + d);
      if (lane == d) {
        if (r.randomize_dof_pos) ratio = (r.dof_pos_ratio[1] - r.dof_pos_ratio[0]) * ud + r.dof_pos_ratio[0];
        if (r.randomize_dof_vel) vel = uv * fabsf(r.dof_vel_range[1] - r.dof_vel_range[0]) + fminf(r.dof_vel_range[0], r.dof_vel_range[1]);
      }
    }
    if (lane < 12) {
      r.dof_state[e * 24 + 2 * lane] = c.default_dof_pos[lane] * ratio;
      r.dof_state[e * 24 + 2 * lane + 1] = vel;
    }
  }
  // ---- _reset_root_states (LR:718-820)
  if (parts & HL_RESET_ROOT) {
    float px = r.base_init_state[0] + r.env_origins[e * 3 + 0], py = r.base_init_state[1] + r.env_origins[e * 3 + 1],
          pz = r.base_init_state[2] + r.env_origins[e * 3 + 2];
    const float ux = ru.get(24), uy = ru.get(25), uz = ru.get(26);
    if (r.custom_origins) {
      if (r.has_pos_range) {
        px += (r.pos_range[1] - r.pos_range[0]) * ux + r.pos_range[0];
        py += (r.pos_range[3] - r.pos_range[2]) * uy + r.pos_range[2];
        pz += (r.pos_range[5] - r.pos_range[4]) * uz + r.pos_range[4];
      } else {
        px += (1.0f - (-1.0f)) * ux + (-1.0f);
        py += (1.0f - (-1.0f)) * uy + (-1.0f);
      }
    }
    float q[4] = {r.base_init_state[3], r.base_init_state[4], r.base_init_state[5], r.base_init_state[6]};
    const float ur = ru.get(27), up_ = ru.get(28), uyw = ru.get(29);
    if (r.has_rot_range) {   // quat_from_euler_xyz(roll, pitch, yaw) (isaacgym.torch_utils)
      const float roll = (r.rot_range[1] - r.rot_range[0]) * ur + r.rot_range[0], pitch = (r.rot_range[3] - r.rot_range[2]) * up_ + r.rot_range[2],
                  yaw = (r.rot_range[5] - r.rot_range[4]) * uyw + r.rot_range[4];
      const float cy = cosf(yaw * 0.5f), sy = sinf(yaw * 0.5f), cr = cosf(roll * 0.5f), sr = sinf(roll * 0.5f), cp = cosf(pitch * 0.5f),
                  sp = sinf(pitch * 0.5f);
      q[0] = cy * sr * cp - sy * cr * sp;
      q[1] = cy * cr * sp + sy * sr * cp;
      q[2] = sy * cr * cp - cy * sr * sp;
      q[3] = cy * cr * cp + sy * sr * sp;
    }
    float vel6 = 0.0f;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const float u = ru.get(30 + k);
      const float* lohi = r.vel_range_is_dict ? r.vel_range + 2 * k : r.vel_range;
      if (lane == k) vel6 = (lohi[1] - lohi[0]) * u + lohi[0];
    }
    if (lane == 0) {
      float* rs = r.root_states + e * 13;
      rs[0] = px; rs[1] = py; rs[2] = pz;
      rs[3] = q[0]; rs[4] = q[1]; rs[5] = q[2]; rs[6] = q[3];
    }
    if (lane < 6) r.root_states[e * 13 + 7 + lane] = vel6;
  }
  // ---- _resample_commands (LR:634-656)
  if (parts & HL_RESET_COMMANDS) hl_resample_env(r, cr, ru, e, gid, lane);
  // ---- Kp / Kd / motor-strength factors (LR:336-341)
  if (parts & HL_RESET_FACTORS) {
    const float ukp = ru.get(40), ukd = ru.get(41), ums = ru.get(42);
    if (lane == 0) {
      if (r.randomize_kp && r.kp_factors) r.kp_factors[e] = (r.kp_range[1] - r.kp_range[0]) * ukp + r.kp_range[0];
      if (r.randomize_kd && r.kd_factors) r.kd_factors[e] = (r.kd_range[1] - r.kd_range[0]) * ukd + r.kd_range[0];
      if (r.randomize_motor_strength && r.motor_strength_factors)
        r.motor_strength_factors[e] = (r.motor_strength_range[1] - r.motor_strength_range[0]) * ums + r.motor_strength_range[0];
    }
  }
  __syncwarp();
}

// One env through any subset of the stages, by one warp (or, with a split, by one warp of its group: `lead` does the
// buffer resets, slot 0 / privileged_obs[0:51] and the roll, the others the height iterations it % it_mod == it_rem).
// `items`: length of the id list -- the warp that completes it finalises the episode-logging means; < 0 = the caller
// finalises them itself.  `st`: this warp's staging area (hl_warp_stage_floats floats of shared memory).  `step`: the Philox step key.
// `cr`: the CTA's command ranges (hl_cmd_ranges_cta; read with HL_ST_RESET_DRAW only).
__device__ __forceinline__ void hl_stage_one(const HlCfg& c, const HlEnvBuffers& b, const uint64_t step, const HlReset& rs, const float* cr,
                                             const unsigned stages, float* st, const long long e, const long long n, const long long items,
                                             const int lane, const bool lead, const bool scans, const int it_mod, const int it_rem) {
  const int B = c.num_bodies;
  const int P = c.n_px * c.n_py;
  const int PD = hl_priv_dim(c);
  __syncwarp();   // the previous env's staged records are no longer read
  if ((stages & HL_ST_RESET_DRAW) && lead) hl_reset_draw_env(c, b, step, rs, cr, e, lane);   // writes the env's root / dof / command rows
  EnvView v;
  hl_stage_env(st, c, b, e, lane, (stages & HL_ST_RESET_ZERO) != 0, v);
  if ((stages & HL_ST_RESET_ZERO) && lead) {  // LR:323-329,350,361
    if (lane < 12) {
      b.last_actions[e * 12 + lane] = 0.0f;
      b.last_last_actions[e * 12 + lane] = 0.0f;
      b.last_dof_pos[e * 12 + lane] = 0.0f;
      b.last_dof_vel[e * 12 + lane] = 0.0f;
      b.last_torques[e * 12 + lane] = 0.0f;
    }
    if (lane < 4) b.feet_air_time[e * 4 + lane] = 0.0f;
    if (b.episode_sums) {
      if ((stages & HL_ST_RESET_DRAW) && rs.means_out && rs.means_ws) {   // LR:346-350: the logged means, before the rows are zeroed
        const long long len = b.episode_length_buf[e] < 1 ? 1 : b.episode_length_buf[e];
        for (int k = lane; k < c.n_terms + c.has_termination_term; k += 32)
          atomicAdd(rs.means_ws + k, (double)__fdiv_rn(__fdiv_rn(b.episode_sums[(long long)k * n + e], (float)len), c.dt));
        // the warp that completes the list turns the sums into means and re-arms the workspace (graph safe)
        const int R = c.n_terms + c.has_termination_term;
        __threadfence();
        __syncwarp();
        unsigned long long done = 0;
        if (lane == 0 && items >= 0) done = atomicAdd(reinterpret_cast<unsigned long long*>(rs.means_ws + R), 1ull) + 1ull;
        done = __shfl_sync(0xffffffffu, done, 0);
        if (items >= 0 && done == (unsigned long long)items) {
          __threadfence();
          for (int k = lane; k < R; k += 32) {
            const double t = *reinterpret_cast<volatile double*>(rs.means_ws + k);
            rs.means_out[k] = (float)(t / (double)items);
            rs.means_ws[k] = 0.0;
          }
          if (lane == 0) *reinterpret_cast<unsigned long long*>(rs.means_ws + R) = 0ull;
        }
      }
      for (int k = lane; k < c.n_terms + c.has_termination_term; k += 32) b.episode_sums[(long long)k * n + e] = 0.0f;
    }
    if (lane == 0) {
      b.episode_length_buf[e] = 0;
      b.reset_buf[e] = 1;
    }
    __syncwarp();
  }
  EnvScalars s;
  s.gid = e + c.env_id_offset;
  s.feet_shift = 0;
  s.base_h = 0.0f;
  s.terrain_level = b.terrain_levels ? b.terrain_levels[e] : 0;
  s.ep_len = b.episode_length_buf[e];
  for (int k = 0; k < 4; ++k) s.cmd[k] = b.commands[e * 4 + k];
  for (int k = 0; k < 4; ++k) s.air[k] = b.feet_air_time[e * 4 + k];
  unsigned last = 0, filt = 0;
  for (int f = 0; f < 4; ++f) {
    last |= (b.last_contacts[e * 4 + f] ? 1u : 0u) << f;
    filt |= (b.contact_filt[e * 4 + f] ? 1u : 0u) << f;
  }
  s.last_contact = last;
  s.cfilt = filt;
  s.contact = 0;
#pragma unroll
  for (int f = 0; f < 4; ++f) s.contact |= (v.cf[c.feet_idx[f] * 3 + 2] > 1.0f ? 1u : 0u) << f;
  s.reset = b.reset_buf[e] != 0;
  s.time_out = b.time_out_buf[e] != 0;
  __syncwarp();

  if (!lead) goto heights_only;   // (parts > 1) the other warps of the env: height iterations only
  if (stages & HL_ST_COUNTERS) {
    s.ep_len += 1;
    if (lane == 0) b.episode_length_buf[e] = s.ep_len;
  }
  if (stages & HL_ST_FRAME) {
    hl_frame(v, s);
    if (lane < 3) {
      b.base_lin_vel[e * 3 + lane] = s.blv[lane];
      b.base_ang_vel[e * 3 + lane] = s.bav[lane];
      b.projected_gravity[e * 3 + lane] = s.pg[lane];
    }
  } else {
    for (int k = 0; k < 3; ++k) {
      s.blv[k] = b.base_lin_vel[e * 3 + k];
      s.bav[k] = b.base_ang_vel[e * 3 + k];
      s.pg[k] = b.projected_gravity[e * 3 + k];
    }
  }
  if (stages & HL_ST_CONTACTS) {
    hl_contacts(c, v, last, s);
    if (lane < 4) {
      b.contact_filt[e * 4 + lane] = (s.cfilt >> lane) & 1u;
      b.last_contacts[e * 4 + lane] = (s.last_contact >> lane) & 1u;
    }
    if (lane < 12) {
      const int f = lane / 3, k = lane % 3;
      if (b.feet_pos) b.feet_pos[e * 12 + lane] = v.fpos[f][k];
      if (b.feet_vel) b.feet_vel[e * 12 + lane] = v.fvel[f][k];
    }
  }
  if ((stages & HL_ST_HEADING) && c.heading_command) {
    s.cmd[2] = hl_heading_command(v.root + 3, s.cmd[3]);
    if (lane == 0) b.commands[e * 4 + 2] = s.cmd[2];
  }
heights_only:
  float myh[8];
  const bool do_h = (stages & HL_ST_HEIGHTS) && c.measure_heights && scans;
  const bool want_base = ((stages & HL_ST_REWARD) && hl_needs_base_height(c)) || (stages & HL_ST_BASE_HEIGHT);
  if (do_h || want_base) {
    ScanOut o;
    o.measured = b.measured_heights + e * P;
    o.priv_heights = nullptr;
    o.idx = b.height_idx_out ? b.height_idx_out + e * P * 2 : nullptr;
    o.u187 = nullptr;
    o.clip = false;
    o.keep = myh;
    s.base_h = hl_warp_scan_env(c, b, step, v.root, (unsigned long long)s.gid, lane, do_h, want_base && lead, o, 0u, it_mod, it_rem);
    if ((stages & HL_ST_BASE_HEIGHT) && b.base_height_out && lane == 0) b.base_height_out[e] = s.base_h;
  }
  if ((stages & HL_ST_TERMINATION) && lead) {
    hl_check_termination(c, v, s);
    if (lane == 0) {
      b.reset_buf[e] = s.reset;
      b.time_out_buf[e] = s.time_out;
    }
  }
  if ((stages & HL_ST_REWARD) && lead) {
    const float rew = hl_compute_reward(c, b, v, s, b.episode_sums ? b.episode_sums + e : nullptr, n, lane == 0);
    if (lane == 0) b.rew_buf[e] = rew;
    if (lane < 4) {
      b.feet_air_time[e * 4 + lane] = s.air[lane];
      b.last_contacts[e * 4 + lane] = (s.last_contact >> lane) & 1u;
    }
  }
  if (stages & HL_ST_OBS) {
    const bool clip = stages & HL_ST_OBS_CLIP;
    const float cl = c.clip_obs;
    // history first (registers), then the new slot: safe when obs_buf_out aliases obs_buf_in
    float old[8];
    if (!(stages & HL_ST_OBS_NOSHIFT) && lead) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int k = i * 32 + lane;
        old[i] = k < 225 ? b.obs_buf_in[e * 270 + k] : 0.0f;
      }
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int k = i * 32 + lane;
        if (k < 225) b.obs_buf_out[e * 270 + 45 + k] = clip ? hl_clampf(old[i], -cl, cl) : old[i];
      }
    }
    if (lead) {
      uint4 nb = make_uint4(0u, 0u, 0u, 0u);
      int cb, c0;
      hl_cur_noise_slot(P, cb, c0);
      if (c.add_noise && !b.noise_u45)
        nb = hl_noise_block(b.philox_seed, step, (unsigned long long)s.gid, (unsigned)(cb * 32 + lane), 0u);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k = lane + 32 * h;
        if (k < 45) {
          float u = 0.5f;
          if (c.add_noise) u = b.noise_u45 ? b.noise_u45[e * 45 + k] : hl_u01(hl_pick(nb, c0 + h));
          float x = hl_add_noise45(c, hl_obs45(c, v, s, k), u, k);
          if (clip) x = hl_clampf(x, -cl, cl);
          b.obs_buf_out[e * 270 + k] = x;
          b.privileged_obs_buf[e * PD + k] = x;
        }
      }
    }
    if (lane < 6 && lead) {
      float x = lane < 3 ? s.blv[lane] * c.obs_lin_vel : b.disturbance[e * B * 3 + (lane - 3)];
      if (clip) x = hl_clampf(x, -cl, cl);
      b.privileged_obs_buf[e * PD + 45 + lane] = x;
    }
    if (c.measure_heights && scans) {
      HeightNoise hn;
      const float rz = v.root[2];
      int pass = -1;
      for (int it = 0; it * 32 < P; ++it) {
        if ((it % it_mod) != it_rem) continue;
        const int p = it * 32 + lane;
        if (!b.noise_u187 && (it >> 2) != pass) { pass = it >> 2; hn.refill(b, step, (unsigned long long)s.gid, pass, lane, 0u); }
        float u = 0.5f;
        if (c.add_noise) u = b.noise_u187 ? (p < P ? b.noise_u187[e * P + p] : 0.5f) : hn.get(it, lane);
        if (p < P) {
          const float mh = do_h ? myh[it] : b.measured_heights[e * P + p];
          float hv = hl_obs_height(c, rz, mh, u);
          if (clip) hv = hl_clampf(hv, -cl, cl);
          b.privileged_obs_buf[e * PD + 51 + p] = hv;
        }
      }
    }
  }
  if ((stages & HL_ST_ROLL) && lead) {  // LR:235-241 (reads complete before writes: llact <- lact <- act)
    __syncwarp();
    float la = 0.f, a = 0.f, dp = 0.f, dv = 0.f, tq = 0.f, rv = 0.f;
    if (lane < 12) {
      la = v.lact[lane];
      a = v.act[lane];
      dp = v.dof_pos(lane);
      dv = v.dof_vel(lane);
      tq = v.tq[lane];
    }
    if (lane < 6) rv = v.root[7 + lane];
    __syncwarp();
    if (lane < 12) {
      b.last_last_actions[e * 12 + lane] = la;
      b.last_actions[e * 12 + lane] = a;
      b.last_dof_pos[e * 12 + lane] = dp;
      b.last_dof_vel[e * 12 + lane] = dv;
      b.last_torques[e * 12 + lane] = tq;
    }
    if (lane < 6) b.last_root_vel[e * 6 + lane] = rv;
    if (lane < 3) b.disturbance[e * B * 3 + lane] = 0.0f;
  }
}

template <unsigned STAGES, bool SPLIT = false>  // STAGES 0 = take the mask at run time; otherwise everything else is compiled out
__global__ void __launch_bounds__(256, 3) hl_stage_kernel(HlCfg c, HlEnvBuffers b, unsigned stages_rt,
                                                       const long long* __restrict__ ids,
                                                       const int* __restrict__ n_ids, long long n, int parts, HlReset rs) {
  // parts > 1 (post-reset fix-up only): an env is spread over `parts` warps -- warp 0 ("lead") does the
  // buffer resets, slot 0 / privileged_obs[0:51] and the roll, warps 1.. the height iterations
  // it % (parts-1) == part-1 (scan + height part of privileged_obs): shorter dependent chains for the
  // few hundred reset envs of a step.
  hl_pdl_enter();
  const unsigned stages = STAGES ? STAGES : stages_rt;
  __shared__ unsigned long long s_step;
  __shared__ float s_cr[8];
  if (stages & HL_ST_RESET_DRAW) hl_cmd_ranges_cta(rs, s_cr);   // published by hl_step_key_cta's barrier
  const uint64_t step = hl_step_key_cta(b, &s_step);
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long items = ids ? (long long)*n_ids : n;
  extern __shared__ __align__(16) float stage_smem[];
  float* st = stage_smem + (threadIdx.x >> 5) * hl_warp_stage_floats(c.num_bodies);
  const int np = (SPLIT && parts > 1) ? parts : 1;   // !SPLIT: folds to the one-warp-per-env code
  for (long long w = warp0; w < items * np; w += nwarps) {
    const long long it0 = w / np;
    const int part = (int)(w - it0 * np);
    const bool lead = part == 0;                      // np == 1: the only warp of the env
    const bool scans = np == 1 || part > 0;           // does height iterations
    const int it_mod = np == 1 ? 1 : np - 1, it_rem = np == 1 ? 0 : part - 1;
    const long long e = ids ? ids[it0] : it0;
    if (e < 0 || e >= n) continue;
    hl_stage_one(c, b, step, rs, s_cr, stages, st, e, n, items, lane, lead, scans, it_mod, it_rem);
  }
}

static int launch_stage(const HlCfg* cfg, const HlEnvBuffers* bufs, unsigned stages, const int64_t* ids,
                        const int32_t* n_ids, int64_t n, void* stream, const HlReset* reset = nullptr) {
  if (int r = check_cfg(cfg, bufs)) return r;
  HlReset rs = {};
  if (stages & HL_ST_RESET_DRAW) {
    HL_CHECK_ARG(reset && reset->struct_bytes == (int)sizeof(HlReset), "HL_ST_RESET_DRAW needs a HlReset (size mismatch?)");
    HL_CHECK_ARG(reset->root_states && reset->dof_state && reset->commands && reset->env_origins, "HlReset: null state tensor");
    HL_CHECK_ARG(ids && n_ids, "HL_ST_RESET_DRAW runs on a reset id list");
    rs = *reset;
  }
  HL_CHECK_ARG((ids == nullptr) == (n_ids == nullptr), "env_ids and n_ids_dev go together");
  if (n <= 0) return HL_OK;
  long long blocks = (n * 32 + 255) / 256;
  if (ids) blocks = blocks < 148 * 8 ? blocks : 148 * 8;  // id lists are short; grid-stride covers the rest
  const size_t stage_smem = (size_t)8 * hl_warp_stage_floats(cfg->num_bodies) * sizeof(float);
  HL_CHECK_ARG(stage_smem <= 48 * 1024, "num_bodies too large for the per-warp staging area");
  static const int fix_parts_env = [] { const char* e = getenv("HL_FIX_PARTS"); return e ? atoi(e) : 4; }();
  // small shards are latency-bound (a few hundred reset envs on 148 SMs): spread each env over several
  // warps; at 65,536 envs the extra staging costs more than the shorter chains save (measured)
  // (a split env would have its scan warps read the root record while the lead warp re-draws it: no split with RESET_DRAW)
  const int fix_parts = (ids && cfg->measure_heights && cfg->mesh_type != 0 && fix_parts_env > 1 && n <= 16384 && !(stages & HL_ST_RESET_DRAW)) ? fix_parts_env : 1;
  constexpr unsigned FIX = HL_ST_HEIGHTS | HL_ST_OBS | HL_ST_OBS_NOSHIFT | HL_ST_OBS_CLIP | HL_ST_ROLL;
  const cudaStream_t st = (cudaStream_t)stream;
  if (stages == FIX)
  {
    if (fix_parts > 1) hl_launch(hl_stage_kernel<FIX, true>, dim3((unsigned)blocks), dim3(256), stage_smem, st, *cfg, *bufs, stages, (const long long*)ids, n_ids, n, fix_parts, rs);
    else hl_launch(hl_stage_kernel<FIX, false>, dim3((unsigned)blocks), dim3(256), stage_smem, st, *cfg, *bufs, stages, (const long long*)ids, n_ids, n, 1, rs);
  }
  else if (stages == (FIX | HL_ST_RESET_ZERO))
  {
    if (fix_parts > 1) hl_launch(hl_stage_kernel<FIX | HL_ST_RESET_ZERO, true>, dim3((unsigned)blocks), dim3(256), stage_smem, st, *cfg, *bufs, stages, (const long long*)ids, n_ids, n, fix_parts, rs);
    else hl_launch(hl_stage_kernel<FIX | HL_ST_RESET_ZERO, false>, dim3((unsigned)blocks), dim3(256), stage_smem, st, *cfg, *bufs, stages, (const long long*)ids, n_ids, n, 1, rs);
  }
  else if (stages == (FIX | HL_ST_RESET_ZERO | HL_ST_RESET_DRAW))
    hl_launch(hl_stage_kernel<FIX | HL_ST_RESET_ZERO | HL_ST_RESET_DRAW, false>, dim3((unsigned)blocks), dim3(256), stage_smem, st, *cfg, *bufs, stages, (const long long*)ids, n_ids, n, 1, rs);
  else
    hl_launch(hl_stage_kernel<0u, false>, dim3((unsigned)blocks), dim3(256), stage_smem, st, *cfg, *bufs, stages, (const long long*)ids, n_ids, n, 1, rs);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

extern "C" int hl_post_physics_stages(const HlCfg* cfg, const HlEnvBuffers* bufs, uint32_t stages,
                                      const int64_t* env_ids, const int32_t* n_ids_dev, int64_t n, void* stream) {
  return launch_stage(cfg, bufs, stages, env_ids, n_ids_dev, n, stream);
}

extern "C" int hl_post_reset_fixup(const HlCfg* cfg, const HlEnvBuffers* bufs, const int64_t* env_ids,
                                   const int32_t* n_ids_dev, int32_t with_reset_zero, int64_t n, void* stream) {
  HL_CHECK_ARG(env_ids && n_ids_dev, "needs the reset id list");
  return launch_stage(cfg, bufs,
                      HL_ST_HEIGHTS | HL_ST_OBS | HL_ST_OBS_NOSHIFT | HL_ST_OBS_CLIP | HL_ST_ROLL |
                          (with_reset_zero ? HL_ST_RESET_ZERO : 0u),
                      env_ids, n_ids_dev, n, stream);
}

extern "C" int hl_sizeof_reset(void) { return (int)sizeof(HlReset); }

extern "C" int hl_reset_idx(const HlCfg* cfg, const HlEnvBuffers* bufs, const HlReset* reset, const int64_t* env_ids,
                            const int32_t* n_ids_dev, int64_t n, void* stream) {
  return launch_stage(cfg, bufs, HL_ST_RESET_ZERO | HL_ST_RESET_DRAW, env_ids, n_ids_dev, n, stream, reset);
}

extern "C" int hl_reset_draw(const HlCfg* cfg, const HlEnvBuffers* bufs, const HlReset* reset, const int64_t* env_ids,
                             const int32_t* n_ids_dev, int64_t n, void* stream) {
  return launch_stage(cfg, bufs, HL_ST_RESET_DRAW, env_ids, n_ids_dev, n, stream, reset);
}

extern "C" int hl_reset_and_fixup(const HlCfg* cfg, const HlEnvBuffers* bufs, const HlReset* reset, const int64_t* env_ids,
                                  const int32_t* n_ids_dev, int64_t n, void* stream) {
  return launch_stage(cfg, bufs,
                      HL_ST_HEIGHTS | HL_ST_OBS | HL_ST_OBS_NOSHIFT | HL_ST_OBS_CLIP | HL_ST_ROLL | HL_ST_RESET_ZERO | HL_ST_RESET_DRAW,
                      env_ids, n_ids_dev, n, stream, reset);
}

// _resample_commands: one thread per candidate env.  The four uniforms are block 9 (columns 36-39) of the env's
// reset-uniform vector, so this matches hl_reset_draw_env's command part for the same (seed, offset, env, stream).
__global__ void __launch_bounds__(256) hl_resample_kernel(HlCfg c, HlEnvBuffers b, HlReset r, const long long* __restrict__ ids,
                                                          const int* __restrict__ n_ids, long long interval, long long n) {
  hl_pdl_enter();
  __shared__ unsigned long long s_step;
  __shared__ float cr[8];
  hl_cmd_ranges_cta(r, cr);                               // published by hl_step_key_cta's barrier
  const uint64_t step = hl_step_key_cta(b, &s_step);
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long e;
  if (ids) {
    if (t >= (long long)*n_ids) return;
    e = ids[t];
    if (e < 0 || e >= n) return;
  } else {
    if (t >= n) return;
    e = t;
    if (interval <= 0 || (b.episode_length_buf[e] + 1) % interval != 0) return;   // LR:612 after LR:193's increment
  }
  const long long gid = e + c.env_id_offset;
  float u[4];
  if (r.uniforms) {
#pragma unroll
    for (int k = 0; k < 4; ++k) u[k] = r.uniforms[e * HL_RESET_NU + 36 + k];
  } else {
    const uint4 q = hl_noise_block(b.philox_seed, step, (unsigned long long)gid, 9u, ids ? 3u : 2u);
    u[0] = hl_u01(q.x); u[1] = hl_u01(q.y); u[2] = hl_u01(q.z); u[3] = hl_u01(q.w);
  }
  float c0 = (1.0f - (-1.0f)) * u[0] + (-1.0f);
  float c1 = (cr[3] - cr[2]) * u[1] + cr[2];
  const float* lohi = r.heading_command ? cr + 6 : cr + 4;
  const float c3 = (lohi[1] - lohi[0]) * u[2] + lohi[0];
  if (gid < r.high_vel_envs) {
    c0 = (cr[1] - cr[0]) * u[3] + cr[0];
    c1 *= fabsf(c0) < 1.0f ? 1.0f : 0.0f;
  }
  const float keep = sqrtf(c0 * c0 + c1 * c1) > 0.2f ? 1.0f : 0.0f;
  r.commands[e * 4 + 0] = c0 * keep;
  r.commands[e * 4 + 1] = c1 * keep;
  r.commands[e * 4 + (r.heading_command ? 3 : 2)] = c3;
}

extern "C" int hl_resample_commands(const HlCfg* cfg, const HlEnvBuffers* bufs, const HlReset* reset, const int64_t* env_ids,
                                    const int32_t* n_ids_dev, int64_t interval, int64_t n, void* stream) {
  if (int r = check_cfg(cfg, bufs)) return r;
  HL_CHECK_ARG(reset && reset->struct_bytes == (int)sizeof(HlReset) && reset->commands, "needs a HlReset with the commands tensor");
  HL_CHECK_ARG((env_ids == nullptr) == (n_ids_dev == nullptr), "env_ids and n_ids_dev go together");
  HL_CHECK_ARG(env_ids || bufs->episode_length_buf, "the pre-step form needs episode_length_buf");
  if (n <= 0) return HL_OK;
  hl_launch(hl_resample_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, *cfg, *bufs, *reset,
            (const long long*)env_ids, n_ids_dev, (long long)interval, (long long)n);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// update_command_curriculum (LR:868-880) on the device ranges: one CTA, a grid-stride float64 sum over the reset ids, then
// thread 0 decides and moves the ranges.  It runs once per max_episode_length steps: a multi-CTA reduction is not worth it.
__global__ void __launch_bounds__(256) hl_command_curriculum_kernel(const float* __restrict__ sums, const long long* __restrict__ ids,
                                                                    const int* __restrict__ n_ids, double threshold, long long max_len,
                                                                    double max_backward, double max_forward, double max_lat,
                                                                    double* ranges, double* ranges_log, long long n) {
  hl_pdl_enter();
  __shared__ double part[8];
  const int tid = threadIdx.x;
  const long long cnt = *n_ids;
  double s = 0.0;
  for (long long i = tid; i < cnt; i += blockDim.x) {
    const long long e = ids[i];
    if (e >= 0 && e < n) s += (double)sums[e];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((tid & 31) == 0) part[tid >> 5] = s;
  __syncthreads();
  if (tid != 0) return;
  double tot = 0.0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += part[w];
  if (cnt > 0) {   // the host returns early on an empty id list
    const float v = __fdiv_rn((float)(tot / (double)cnt), (float)max_len);   // fp32 mean, then the fp32 divide by the length
    if ((double)v > threshold) {   // np.clip(x, lo, hi) == min(max(x, lo), hi), in float64
      ranges[0] = fmin(fmax(ranges[0] - 0.1, -max_backward), 0.0);
      ranges[1] = fmin(fmax(ranges[1] + 0.1, 0.0), max_forward);
      ranges[2] = fmin(fmax(ranges[2] - 0.1, -max_lat), 0.0);
      ranges[3] = fmin(fmax(ranges[3] + 0.1, 0.0), max_lat);
    }
  }
  if (ranges_log)
    for (int k = 0; k < 8; ++k) ranges_log[k] = ranges[k];
}

extern "C" int hl_command_curriculum(const float* tracking_sums, const int64_t* env_ids, const int32_t* n_ids_dev, double threshold,
                                     int64_t max_episode_length, double max_backward, double max_forward, double max_lat,
                                     double* ranges, double* ranges_log, int64_t n, void* stream) {
  HL_CHECK_ARG(tracking_sums && env_ids && n_ids_dev && ranges, "null pointer");
  HL_CHECK_ARG(max_episode_length > 0, "max_episode_length must be positive");
  hl_launch(hl_command_curriculum_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, tracking_sums, (const long long*)env_ids,
            n_ids_dev, threshold, (long long)max_episode_length, max_backward, max_forward, max_lat, ranges, ranges_log, (long long)n);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// one env's records for the terminal rows (root 13 | dof 24 | act 12), staged per warp
constexpr int TR_FLOATS = 52;
__device__ __forceinline__ void hl_stage_rows_env(float* st, const HlEnvBuffers& b, long long e, int lane, EnvView& v) {
  const float r_root = lane < 13 ? b.root_states[e * 13 + lane] : 0.0f;
  const float r_dof = lane < 24 ? b.dof_state[e * 24 + lane] : 0.0f;
  const float r_act = lane < 12 ? b.actions[e * 12 + lane] : 0.0f;
  if (lane < 13) st[lane] = r_root;
  if (lane < 24) st[13 + lane] = r_dof;
  if (lane < 12) st[37 + lane] = r_act;
  __syncwarp();
  v.root = st;
  v.dof = st + 13;
  v.act = st + 37;
}

// ============================================================================= terminal rows
// compute_termination_observations(env_ids) + get_amp_observations()[env_ids] (LR:227-228):
// one warp per reset env, from the persisted pre-reset derived state.
__global__ void __launch_bounds__(256) hl_terminal_rows_kernel(HlCfg c, HlEnvBuffers b, const long long* __restrict__ ids,
                                                               const int* __restrict__ n_ids,
                                                               const float* __restrict__ u45,
                                                               const float* __restrict__ u187,
                                                               float* __restrict__ out_priv, float* __restrict__ out_amp,
                                                               long long n) {
  hl_pdl_enter();
  __shared__ unsigned long long s_step;
  const uint64_t step = hl_step_key_cta(b, &s_step);
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long items = *n_ids;
  const int B = c.num_bodies, P = c.n_px * c.n_py, PD = hl_priv_dim(c);
  __shared__ float tr_stage[8 * TR_FLOATS];
  float* st = tr_stage + (threadIdx.x >> 5) * TR_FLOATS;
  for (long long r = warp0; r < items; r += nwarps) {
    const long long e = ids[r];
    if (e < 0 || e >= n) continue;
    __syncwarp();
    EnvView v;
    hl_stage_rows_env(st, b, e, lane, v);
    EnvScalars s;
    s.gid = e + c.env_id_offset;
    for (int k = 0; k < 4; ++k) s.cmd[k] = b.commands[e * 4 + k];
    for (int k = 0; k < 3; ++k) {
      s.blv[k] = b.base_lin_vel[e * 3 + k];
      s.bav[k] = b.base_ang_vel[e * 3 + k];
      s.pg[k] = b.projected_gravity[e * 3 + k];
    }
    {
      uint4 nb = make_uint4(0u, 0u, 0u, 0u);
      int cb, c0;
      hl_cur_noise_slot(P, cb, c0);
      if (c.add_noise && !u45)
        nb = hl_noise_block(b.philox_seed, step, (unsigned long long)s.gid, (unsigned)(cb * 32 + lane), 1u);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k = lane + 32 * h;
        if (k < 45) {
          float u = 0.5f;
          if (c.add_noise) u = u45 ? u45[e * 45 + k] : hl_u01(hl_pick(nb, c0 + h));
          out_priv[r * PD + k] = hl_add_noise45(c, hl_obs45(c, v, s, k), u, k);
        }
      }
    }
    if (lane < 6) out_priv[r * PD + 45 + lane] = lane < 3 ? s.blv[lane] * c.obs_lin_vel : b.disturbance[e * B * 3 + (lane - 3)];
    if (c.measure_heights) {
      HeightNoise hn;
      const float rz = v.root[2];
      for (int it = 0; it * 32 < P; ++it) {
        const int p = it * 32 + lane;
        if (!u187 && (it & 3) == 0) hn.refill(b, step, (unsigned long long)s.gid, it >> 2, lane, 1u);
        float u = 0.5f;
        if (c.add_noise) u = u187 ? (p < P ? u187[e * P + p] : 0.5f) : hn.get(it, lane);
        if (p < P) out_priv[r * PD + 51 + p] = hl_obs_height(c, rz, b.measured_heights[e * P + p], u);
      }
    }
    if (out_amp && lane < 30) {  // LR:416: dof_pos 12, base_lin_vel 3, base_ang_vel 3, dof_vel 12
      float x;
      if (lane < 12) x = v.dof_pos(lane);
      else if (lane < 15) x = s.blv[lane - 12];
      else if (lane < 18) x = s.bav[lane - 15];
      else x = v.dof_vel(lane - 18);
      out_amp[r * 30 + lane] = x;
    }
  }
}

extern "C" int hl_terminal_rows(const HlCfg* cfg, const HlEnvBuffers* bufs, const int64_t* env_ids,
                                const int32_t* n_ids_dev, const float* u45, const float* u187, float* out_priv,
                                float* out_amp, int64_t n, void* stream) {
  if (int r = check_cfg(cfg, bufs)) return r;
  HL_CHECK_ARG(env_ids && n_ids_dev && out_priv, "null pointer");
  if (n <= 0) return HL_OK;
  hl_launch(hl_terminal_rows_kernel, dim3((unsigned)((n * 32 + 255) / 256 < 148 * 8 ? (n * 32 + 255) / 256 : 148 * 8)), dim3(256), 0,
            (cudaStream_t)stream, *cfg, *bufs, (const long long*)env_ids, n_ids_dev, u45, u187, out_priv, out_amp, n);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= ids + terminal rows
// One launch for LR:225-228: env_ids = reset_buf.nonzero().flatten(), then
// compute_termination_observations(env_ids) and get_amp_observations()[env_ids].
// CTA = 1024 consecutive envs: flags -> block scan -> (sum of the counts of all lower CTAs, which
// were dispatched earlier and publish right after their scan) -> ordered ids -> the CTA's warps
// write the rows of its own reset envs.  ws = {pad, done, epoch, pad, state[nblocks]}.
constexpr int SEL_ENVS = 256;   // small tiles: the rows of a CTA's ~6 reset envs go one per warp
// RESET: each warp, right after the terminal rows of a reset env (pre-reset state), also runs that env's reset_idx
// (re-draws, buffer zeroing, episode-logging sums) and post-reset fix-up (re-scan, slot 0, roll) -- LR:225-241 for the
// reset envs in ONE launch; the last CTA to finish turns the logging sums into means.
template <bool RESET>
__global__ void __launch_bounds__(256) hl_select_terminal_kernel(HlCfg c, HlEnvBuffers b, const float* __restrict__ u45,
                                                                 const float* __restrict__ u187,
                                                                 long long* __restrict__ ids_out, int* __restrict__ count_out,
                                                                 float* __restrict__ out_priv, float* __restrict__ out_amp,
                                                                 unsigned long long* ws, long long n, HlReset rs) {
  __shared__ int warp_tot[8];
  __shared__ int s_excl, s_total;
  __shared__ unsigned s_epoch;
  __shared__ int s_local[SEL_ENVS];  // local env offsets of this CTA's reset envs, ascending
  hl_pdl_enter();
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const unsigned nblocks = gridDim.x;
  unsigned* ctrl = reinterpret_cast<unsigned*>(ws);
  volatile unsigned long long* state = reinterpret_cast<volatile unsigned long long*>(ws) + 2;
  __shared__ unsigned s_vb;
  __shared__ unsigned long long s_step;
  __shared__ float s_cr[8];
  if (tid == 0) {   // virtual block id by ticket: a CTA only ever waits on CTAs that have already started
    s_vb = atomicAdd(ctrl, 1u);
    s_epoch = *reinterpret_cast<volatile unsigned*>(ctrl + 2) + 1u;
    s_step = hl_step_key(b);
  }
  if (RESET) hl_cmd_ranges_cta(rs, s_cr);
  __syncthreads();
  const unsigned vb = s_vb;
  const uint64_t step = s_step;
  const long long e0 = (long long)vb * SEL_ENVS;
  // one flag per thread
  const long long off = e0 + tid;
  const unsigned mask = (off < n && b.reset_buf[off]) ? 1u : 0u;
  const int cnt = (int)mask;
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warp_tot[wid] = incl;
  __syncthreads();
  int wbase = 0;
  for (int w = 0; w < wid; ++w) wbase += warp_tot[w];
  if (tid == 0) {
    int tot = 0;
    for (int w = 0; w < 8; ++w) tot += warp_tot[w];
    s_total = tot;
    state[vb] = ((unsigned long long)s_epoch << 32) | HL_LB_AGG | (unsigned long long)(unsigned)tot;  // publish early
    __threadfence();
  }
  int pos = wbase + incl - cnt;
  if (mask) s_local[pos] = tid;
  __syncthreads();
  // warps 1..7 stage the records of their first reset env while warp 0 does the look-back
  __shared__ float tr_stage[8 * TR_FLOATS];
  float* st = tr_stage + wid * TR_FLOATS;
  EnvView v;
  bool staged = false;
  if (out_priv && wid != 0 && wid < s_total) {
    hl_stage_rows_env(st, b, e0 + s_local[wid], lane, v);
    staged = true;
  }
  if (wid == 0) {  // exclusive prefix: nearest earlier CTA with an inclusive prefix + the aggregates in between
    const unsigned ep = s_epoch;
    int acc = 0;
    long long t = (long long)vb - 1;
    while (t >= 0) {
      const long long idx = t - lane;
      unsigned long long w = ((unsigned long long)ep << 32) | HL_LB_PREFIX;
      if (idx >= 0) {
        w = state[idx];
        while ((unsigned)(w >> 32) != ep) w = state[idx];
      }
      const unsigned pm = __ballot_sync(0xffffffffu, (w & HL_LB_PREFIX) != 0ull);
      const int first = pm ? (__ffs(pm) - 1) : 31;
      int val = lane <= first ? (int)(w & HL_LB_VALUE) : 0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) val += __shfl_xor_sync(0xffffffffu, val, o);
      acc += val;
      if (pm) break;
      t -= 32;
    }
    if (lane == 0) {
      s_excl = acc;
      state[vb] = ((unsigned long long)ep << 32) | HL_LB_PREFIX | (unsigned long long)(unsigned)(acc + s_total);
      if (vb == nblocks - 1) *count_out = acc + s_total;
    }
  }
  __syncthreads();
  const int excl = s_excl, total = s_total;
  for (int i = tid; i < total; i += 256) ids_out[excl + i] = e0 + s_local[i];
  // rows: one warp per reset env of this CTA
  const int B = c.num_bodies, P = c.n_px * c.n_py, PD = hl_priv_dim(c);
  if (out_priv) {
    int cb, c0;
    hl_cur_noise_slot(P, cb, c0);
    for (int i = wid; i < total; i += 8) {
      const long long e = e0 + s_local[i], r = excl + i;
      if (!(staged && i == wid)) {
        __syncwarp();
        hl_stage_rows_env(st, b, e, lane, v);
      }
      EnvScalars s;
      s.gid = e + c.env_id_offset;
      for (int k = 0; k < 4; ++k) s.cmd[k] = b.commands[e * 4 + k];
      for (int k = 0; k < 3; ++k) {
        s.blv[k] = b.base_lin_vel[e * 3 + k];
        s.bav[k] = b.base_ang_vel[e * 3 + k];
        s.pg[k] = b.projected_gravity[e * 3 + k];
      }
      uint4 nb = make_uint4(0u, 0u, 0u, 0u);
      if (c.add_noise && !u45) nb = hl_noise_block(b.philox_seed, step, (unsigned long long)s.gid, (unsigned)(cb * 32 + lane), 1u);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k = lane + 32 * h;
        if (k < 45) {
          float u = 0.5f;
          if (c.add_noise) u = u45 ? u45[e * 45 + k] : hl_u01(hl_pick(nb, c0 + h));
          out_priv[r * PD + k] = hl_add_noise45(c, hl_obs45(c, v, s, k), u, k);
        }
      }
      if (lane < 6) out_priv[r * PD + 45 + lane] = lane < 3 ? s.blv[lane] * c.obs_lin_vel : b.disturbance[e * B * 3 + (lane - 3)];
      if (c.measure_heights) {
        HeightNoise hn;
        const float rz = v.root[2];
        float mh[8];
#pragma unroll
        for (int it = 0; it < 8; ++it) mh[it] = (it * 32 + lane < P) ? b.measured_heights[e * P + it * 32 + lane] : 0.0f;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          if (it * 32 >= P) break;
          const int p = it * 32 + lane;
          if (!u187 && (it & 3) == 0) hn.refill(b, step, (unsigned long long)s.gid, it >> 2, lane, 1u);
          float u = 0.5f;
          if (c.add_noise) u = u187 ? (p < P ? u187[e * P + p] : 0.5f) : hn.get(it, lane);
          if (p < P) out_priv[r * PD + 51 + p] = hl_obs_height(c, rz, mh[it], u);
        }
      }
      if (out_amp && lane < 30) {
        float x;
        if (lane < 12) x = v.dof_pos(lane);
        else if (lane < 15) x = s.blv[lane - 12];
        else if (lane < 18) x = s.bav[lane - 15];
        else x = v.dof_vel(lane - 18);
        out_amp[r * 30 + lane] = x;
      }
      if (RESET) {   // the terminal rows are out: this env may now be reset (same warp, program order)
        extern __shared__ __align__(16) float sel_stage[];
        __syncwarp();
        hl_stage_one(c, b, step, rs, s_cr, HL_ST_HEIGHTS | HL_ST_OBS | HL_ST_OBS_NOSHIFT | HL_ST_OBS_CLIP | HL_ST_ROLL | HL_ST_RESET_ZERO | HL_ST_RESET_DRAW,
                     sel_stage + wid * hl_warp_stage_floats(c.num_bodies), e, n, -1, lane, true, true, 1, 0);
        staged = false;
      }
    }
  }
  __syncthreads();
  if (tid == 0) {  // last CTA re-arms the workspace (graph safe)
    __threadfence();
    if (atomicAdd(ctrl + 1, 1u) == nblocks - 1) {
      if (RESET && rs.means_out && rs.means_ws && b.episode_sums) {   // every CTA's logging sums are in: LR:346-350 means
        __threadfence();
        const int total = *reinterpret_cast<volatile int*>(count_out);
        const int R = c.n_terms + c.has_termination_term;
        for (int k = 0; k < R; ++k) {
          const double t = *reinterpret_cast<volatile double*>(rs.means_ws + k);
          if (total > 0) rs.means_out[k] = (float)(t / (double)total);
          rs.means_ws[k] = 0.0;
        }
      }
      ctrl[0] = 0u;
      ctrl[1] = 0u;
      ctrl[2] = s_epoch;
      __threadfence();
    }
  }
}

extern "C" int64_t hl_select_terminal_workspace_bytes(int64_t n) { return (int64_t)(((n + SEL_ENVS - 1) / SEL_ENVS) + 2) * 8; }
extern "C" int hl_select_and_terminal(const HlCfg* cfg, const HlEnvBuffers* bufs, const float* u45, const float* u187,
                                      int64_t* ids_out, int32_t* count_out, float* out_priv, float* out_amp,
                                      void* workspace, int64_t n, void* stream) {
  if (int r = check_cfg(cfg, bufs)) return r;
  HL_CHECK_ARG(ids_out && count_out && workspace && bufs->reset_buf, "null pointer");
  if (n <= 0) return HL_OK;
  HlReset none = {};
  hl_launch(hl_select_terminal_kernel<false>, dim3((unsigned)((n + SEL_ENVS - 1) / SEL_ENVS)), dim3(256), 0, (cudaStream_t)stream,
            *cfg, *bufs, u45, u187, (long long*)ids_out, count_out, out_priv, out_amp, (unsigned long long*)workspace, n, none);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

extern "C" int hl_select_terminal_reset(const HlCfg* cfg, const HlEnvBuffers* bufs, const HlReset* reset, const float* u45,
                                        const float* u187, int64_t* ids_out, int32_t* count_out, float* out_priv, float* out_amp,
                                        void* workspace, int64_t n, void* stream) {
  if (int r = check_cfg(cfg, bufs)) return r;
  HL_CHECK_ARG(ids_out && count_out && workspace && bufs->reset_buf && out_priv, "null pointer");
  HL_CHECK_ARG(reset && reset->struct_bytes == (int)sizeof(HlReset), "needs a HlReset (size mismatch?)");
  HL_CHECK_ARG(reset->root_states && reset->dof_state && reset->commands && reset->env_origins, "HlReset: null state tensor");
  if (n <= 0) return HL_OK;
  const size_t smem = (size_t)8 * hl_warp_stage_floats(cfg->num_bodies) * sizeof(float);
  HL_CHECK_ARG(smem <= 40 * 1024, "num_bodies too large for the per-warp staging area");
  hl_launch(hl_select_terminal_kernel<true>, dim3((unsigned)((n + SEL_ENVS - 1) / SEL_ENVS)), dim3(256), smem, (cudaStream_t)stream,
            *cfg, *bufs, u45, u187, (long long*)ids_out, count_out, out_priv, out_amp, (unsigned long long*)workspace, n, *reset);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= episode logging of reset_idx
// One CTA per reward row; threads stride over the reset id list, float64 partials, block reduce.
__global__ void __launch_bounds__(256) hl_episode_means_kernel(float* __restrict__ sums, const long long* __restrict__ ep_len,
                                                               const long long* __restrict__ ids, const int* __restrict__ n_ids,
                                                               long long n, float dt, int zero_rows, float* __restrict__ out) {
  hl_pdl_enter();
  __shared__ double part[8];
  const int k = blockIdx.x, tid = threadIdx.x;
  const int cnt = *n_ids;
  float* row = sums + (long long)k * n;
  double acc = 0.0;
  for (int i = tid; i < cnt; i += 256) {
    const long long e = ids[i];
    if (e < 0 || e >= n) continue;
    const long long len = ep_len[e] < 1 ? 1 : ep_len[e];
    acc += (double)__fdiv_rn(__fdiv_rn(row[e], (float)len), dt);   // LR:349 op order, each division rounded
    if (zero_rows) row[e] = 0.0f;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((tid & 31) == 0) part[tid >> 5] = acc;
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += part[w];
    if (cnt > 0) out[k] = (float)(t / (double)cnt);   // no reset: reset_idx returns early (LR:298-299), the logged value stays
  }
}

extern "C" int hl_episode_means(float* episode_sums, const int64_t* episode_length_buf, const int64_t* env_ids,
                                const int32_t* n_ids_dev, int32_t n_rows, int64_t n, float dt, int32_t zero_rows,
                                float* means_out, void* stream) {
  HL_CHECK_ARG(episode_sums && episode_length_buf && env_ids && n_ids_dev && means_out, "null pointer");
  HL_CHECK_ARG(dt > 0.0f, "dt must be positive");
  if (n_rows <= 0 || n <= 0) return HL_OK;
  hl_launch(hl_episode_means_kernel, dim3((unsigned)n_rows), dim3(256), 0, (cudaStream_t)stream, episode_sums,
            (const long long*)episode_length_buf, (const long long*)env_ids, n_ids_dev, (long long)n, dt, (int)zero_rows, means_out);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= a13: AMP observations
__global__ void __launch_bounds__(256) hl_amp_obs_kernel(const float* __restrict__ dof, const float* __restrict__ blv,
                                                         const float* __restrict__ bav, float* __restrict__ out,
                                                         long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long e = i / 30;
  const int k = (int)(i - e * 30);
  float x;
  if (k < 12) x = dof[e * 24 + 2 * k];
  else if (k < 15) x = blv[e * 3 + (k - 12)];
  else if (k < 18) x = bav[e * 3 + (k - 15)];
  else x = dof[e * 24 + 2 * (k - 18) + 1];
  out[i] = x;
}
extern "C" int hl_amp_observations(const float* dof_state, const float* blv, const float* bav, float* out, int64_t n,
                                   void* stream) {
  HL_CHECK_ARG(dof_state && blv && bav && out, "null pointer");
  if (n <= 0) return HL_OK;
  const long long total = n * 30;
  hl_amp_obs_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(dof_state, blv, bav, out, total);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= a10: reset ids
// env_ids = reset_buf.nonzero().flatten() (LR:225): ordered stream compaction.  One CTA walks the
// flags 16 KB at a time (uint4 per thread), warp-shuffle scan inside, running offset across
// chunks.  N bytes of input: ~4 chunks at 65,536 envs.
__global__ void __launch_bounds__(1024) hl_select_ids_kernel(const uint8_t* __restrict__ flags, long long n,
                                                             long long* __restrict__ ids, int* __restrict__ count) {
  __shared__ int warp_tot[32];
  __shared__ int running_s;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) running_s = 0;
  __syncthreads();
  const bool aligned = ((uintptr_t)flags & 15) == 0;
  for (long long base = 0; base < n; base += 1024 * 16) {
    const long long off = base + (long long)tid * 16;
    unsigned mask = 0;
    if (off + 16 <= n && aligned) {
      const uint4 q = *reinterpret_cast<const uint4*>(flags + off);
      const unsigned w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int j = 0; j < 4; ++j) mask |= (((w[k] >> (8 * j)) & 0xffu) ? 1u : 0u) << (4 * k + j);
    } else {
      for (int j = 0; j < 16; ++j)
        if (off + j < n && flags[off + j]) mask |= 1u << j;
    }
    const int cnt = __popc(mask);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const int running = running_s;   // read before the barrier: warp 0 overwrites it right after
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      int wt = warp_tot[lane], wi = wt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, wi, o);
        if (lane >= o) wi += t;
      }
      warp_tot[lane] = wi - wt;  // exclusive prefix of warp totals
      if (lane == 31) running_s = running + wi;
    }
    __syncthreads();
    int pos = running + warp_tot[wid] + incl - cnt;
    while (mask) {
      const int j = __ffs(mask) - 1;
      mask &= mask - 1;
      ids[pos++] = off + j;
    }
    __syncthreads();
  }
  if (tid == 0) *count = running_s;
}
extern "C" int64_t hl_select_workspace_bytes(int64_t) { return 256; }
extern "C" int hl_select_reset_ids(const uint8_t* reset_buf, int64_t n, int64_t* ids_out, int32_t* count_out, void*,
                                   void* stream) {
  HL_CHECK_ARG(reset_buf && ids_out && count_out && n >= 0, "null pointer");
  hl_select_ids_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(reset_buf, n, (long long*)ids_out, count_out);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= the fused step
// One CTA (8 warps) = EPB consecutive envs (tile sizes 64 / 52 / 32, see pick_tile).
//   phase 0  128-bit coalesced slab loads of every AoS record into shared memory (odd row strides
//            => conflict-free one-lane-per-env reads); only pos/vel of the 4 foot records are
//            fetched from rigid_body_states.
//   phase 1  warp-specialised, concurrently:
//              warps 0-1  one lane per env: frame, contacts, heading, termination, one-step obs
//                         (+noise), then -- after the base heights arrive (named barrier) -- the
//                         reward terms and episode sums;
//              warps 2-7  height scans, one warp per env: 63-point base grid first (-> base
//                         height), then the 187-point grid -> measured_heights + the height part
//                         of privileged_obs (noise, scale, clip fused).  Each lane owns fixed grid
//                         points (coordinates in registers); every op of the index path is
//                         rounded on its own in the reference's order.
//   phase 2  coalesced stores: obs history shift (register-staged, in-place safe), slot 0,
//            privileged_obs[0:51], the last_* roll (skipped for envs that reset: the post-reset
//            fix-up redoes it after reset_idx).
constexpr int S13 = 13, SA = 12, SDOF = 24, SFOOT = 25, SCUR = 57;   // shared-memory row strides (floats)

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// cell index of one coordinate, fused path (int32 is enough: cvt saturates exactly where the
// reference's clip would land; NaN -> 0 either way)
template <bool CPU_MATH>
__device__ __forceinline__ int cell32(float world, float border, float hs, float inv_hs, int hi) {
  const float p = __fadd_rn(world, border);
  const float g = CPU_MATH ? __fdiv_rn(p, hs) : __fmul_rn(p, inv_hs);
  return (int)min(__float2uint_rz(g), (unsigned)hi);   // cvt.rzi.u32 saturates: negatives and NaN -> 0
}

// raw min-of-3 height (int16 units) under body-frame point (bx,by): quat_apply_yaw + translate +
// border + scale + trunc + clip (LR:1339-1347) in the reference's op order, every product and sum
// rounded on its own with the non-contractable __fmul_rn/__fadd_rn (see hl_scan_axis_* in
// hl_math.cuh for the derivation).  NOTE: packed FFMA2 arithmetic was tried here and rejected:
// ptxas contracts packed mul->add chains into single-rounding FFMA2s even from explicit
// fma.rn.f32x2 and with -fmad=false, which breaks the one-rounding-per-op guarantee.
template <bool CPU_MATH>
__device__ __forceinline__ int scan_gather(const HlCfg& c, const int16_t* __restrict__ min3, int pitch, float qz, float qw,
                                           float posx, float posy, float bx, float by) {
  const float ty = 2.0f * __fmul_rn(qz, bx), tx = -2.0f * __fmul_rn(qz, by);
  const float ay = __fmul_rn(qw, ty), cx = -__fmul_rn(qz, ty);
  const float ax = __fmul_rn(qw, tx), cy = __fmul_rn(qz, tx);
  const float rx = __fadd_rn(__fadd_rn(bx, ax), cx);
  const float ry = __fadd_rn(__fadd_rn(by, ay), cy);
  const int ix = cell32<CPU_MATH>(__fadd_rn(rx, posx), c.border_size, c.horizontal_scale, c.inv_horizontal_scale, c.terrain_rows - 2);
  const int iy = cell32<CPU_MATH>(__fadd_rn(ry, posy), c.border_size, c.horizontal_scale, c.inv_horizontal_scale, c.terrain_cols - 2);
#ifdef HL_EXP_NO_GATHER
  return ix + iy;
#else
  return (int)__ldg(min3 + (unsigned)(ix * pitch + iy));
#endif
}

// same cell arithmetic; the table already holds metres (hl_terrain_prepare_f32)
template <bool CPU_MATH>
__device__ __forceinline__ float scan_gather_f(const HlCfg& c, const float* __restrict__ min3f, int pitch, float qz, float qw,
                                               float posx, float posy, float bx, float by) {
  const float ty = 2.0f * __fmul_rn(qz, bx), tx = -2.0f * __fmul_rn(qz, by);
  const float ay = __fmul_rn(qw, ty), cx = -__fmul_rn(qz, ty);
  const float ax = __fmul_rn(qw, tx), cy = __fmul_rn(qz, tx);
  const float rx = __fadd_rn(__fadd_rn(bx, ax), cx);
  const float ry = __fadd_rn(__fadd_rn(by, ay), cy);
  const int ix = cell32<CPU_MATH>(__fadd_rn(rx, posx), c.border_size, c.horizontal_scale, c.inv_horizontal_scale, c.terrain_rows - 2);
  const int iy = cell32<CPU_MATH>(__fadd_rn(ry, posy), c.border_size, c.horizontal_scale, c.inv_horizontal_scale, c.terrain_cols - 2);
#ifdef HL_PKX_NO_GATHER
  return (float)(ix + iy);
#else
  return __ldg(min3f + (unsigned)(ix * pitch + iy));
#endif
}

struct FusedArgs {
  int cf_stride, need_ldp, need_ltq, want_base;
  long long rs_interval;  // > 0: resample the commands of envs whose incremented episode length hits the interval (LR:612-613)
  int rs_heading;
  long long rs_hi_envs;   // HlReset::high_vel_envs (LR:649)
  float rs_lin_vel_x[2], rs_lin_vel_y[2], rs_third[2];   // third = heading range (heading_command) or yaw-rate range
  const float* rs_uniforms;   // (N, HL_RESET_NU) or nullptr => Philox stream 2
  const double* rs_ranges;    // HlReset::cmd_ranges (device) or nullptr => the by-value rs_* ranges above
  int hist_pf;            // bulk-prefetch the tile's obs-history slab into L2 (obs_buf_in 16-B aligned)
  int tma_ok;             // every dense slab of a full tile is 16-B aligned with a 16-B multiple size (n % 4 == 0, aligned bases)
  int sums_aligned;       // episode_sums rows are 16-B aligned per block (n % 4 == 0, base aligned)
  int compact;            // emit reset ids / count / terminal rows from this launch (decoupled look-back)
  int hist_clipped;       // obs history is known to be within +-clip_obs already (every step after the first)
  HlPhiloxKeys keys;      // Philox round keys of bufs.philox_seed (host-computed: constant-bank operands)
};

// _resample_commands for the lane's env inside the fused step (same arithmetic and uniform columns as hl_resample_kernel)
__device__ __forceinline__ void hl_fused_resample(const FusedArgs& fa, const HlEnvBuffers& b, uint64_t step, long long ge, long long gid, float* cmd) {
  float u[4];
  if (fa.rs_uniforms) {
#pragma unroll
    for (int k = 0; k < 4; ++k) u[k] = fa.rs_uniforms[ge * HL_RESET_NU + 36 + k];
  } else {
    const uint4 q = hl_noise_block(b.philox_seed, step, (unsigned long long)gid, 9u, 2u);
    u[0] = hl_u01(q.x); u[1] = hl_u01(q.y); u[2] = hl_u01(q.z); u[3] = hl_u01(q.w);
  }
  // the ranges: by value, or from the device copy (this branch runs after the kernel's griddepcontrol.wait)
  float x0 = fa.rs_lin_vel_x[0], x1 = fa.rs_lin_vel_x[1], y0 = fa.rs_lin_vel_y[0], y1 = fa.rs_lin_vel_y[1], t0 = fa.rs_third[0],
        t1 = fa.rs_third[1];
  if (fa.rs_ranges) {
    const double* q = fa.rs_ranges;
    const int o = fa.rs_heading ? 6 : 4;
    x0 = (float)q[0]; x1 = (float)q[1]; y0 = (float)q[2]; y1 = (float)q[3]; t0 = (float)q[o]; t1 = (float)q[o + 1];
  }
  float c0 = (1.0f - (-1.0f)) * u[0] + (-1.0f);
  float c1 = (y1 - y0) * u[1] + y0;
  const float c3 = (t1 - t0) * u[2] + t0;
  if (gid < fa.rs_hi_envs) {
    c0 = (x1 - x0) * u[3] + x0;
    c1 *= fabsf(c0) < 1.0f ? 1.0f : 0.0f;
  }
  const float keep = sqrtf(c0 * c0 + c1 * c1) > 0.2f ? 1.0f : 0.0f;
  cmd[0] = c0 * keep;
  cmd[1] = c1 * keep;
  cmd[fa.rs_heading ? 3 : 2] = c3;
}

// tile sizes: 64 (default), 52 (65,536 envs = 1261 CTAs = 2.84 waves of 444 instead of 2.31 -> 3
// waves of 52 instead of 64 envs), 32 (small shards: more CTAs than SMs sooner)
#define FK_NS fk64
#define FK_EPB 64
#define FK_SCALAR_WARPS 2
#define FK_GENERIC 1   // also the any-grid / clipped-heights fallback
#define FK_COMPACT 1
#include "hl_fused_kernel.inc"
#undef FK_NS
#undef FK_EPB
#undef FK_SCALAR_WARPS
#undef FK_GENERIC
#undef FK_COMPACT
#define FK_NS fk52
#ifdef HL_EXP_TILE
#define FK_EPB HL_EXP_TILE
#else
#define FK_EPB 52
#endif
#define FK_SCALAR_WARPS 2
#ifdef HL_EXP_T288
#define FK_THREADS 288
#endif
#define FK_GENERIC 0
#define FK_COMPACT 1
#include "hl_fused_kernel.inc"
#undef FK_NS
#undef FK_EPB
#undef FK_SCALAR_WARPS
#undef FK_GENERIC
#undef FK_COMPACT
#define FK_NS fk32
#define FK_EPB 32
#define FK_SCALAR_WARPS 1
#define FK_GENERIC 0
#define FK_COMPACT 1
#include "hl_fused_kernel.inc"
#undef FK_NS
#undef FK_EPB
#undef FK_SCALAR_WARPS
#undef FK_GENERIC
#undef FK_COMPACT

#include "hl_persist_kernel.inc"

// Envs per CTA that minimises (waves x tile cost) for this shard on this device: a wave is
// SMs x 3 resident CTAs; the cost of a tile is ~ a fixed part (loads, barriers) + its envs.
static int pick_tile(int64_t n) {
  const int sms = device_sms();
  const char* fe = getenv("HL_FUSED_EPB");  // dev/test knob, read per call
  const int forced = fe ? atoi(fe) : 0;
  if (forced == 64 || forced == 52 || forced == 32) return forced;
  const int cand[3] = {64, 52, 32};
  int best = 64;
  double best_cost = 1e30;
  for (int k = 0; k < 3; ++k) {
    const int64_t ctas = (n + cand[k] - 1) / cand[k];
    const int64_t waves = (ctas + (int64_t)sms * 3 - 1) / ((int64_t)sms * 3);
    const double cost = (double)waves * (10.0 + cand[k]);
    if (cost < best_cost) { best_cost = cost; best = cand[k]; }
  }
  return best;
}

static thread_local int g_fused_last_impl = -1;
extern "C" int hl_fused_last_impl(void) { return g_fused_last_impl; }

extern "C" int64_t hl_fused_workspace_bytes(int64_t n) { return (int64_t)(((n + 16 - 1) / 16) + 2) * 8; }  // sized for tiles of >= 16 envs

extern "C" int hl_post_physics_fused(const HlCfg* cfg, const HlEnvBuffers* bufs, int64_t n, void* stream) {
  if (int r = check_cfg(cfg, bufs)) return r;
  const HlEnvBuffers& b = *bufs;
  HL_CHECK_ARG(b.root_states && b.dof_state && b.contact_forces && (b.rigid_body_states || b.foot_records) && b.actions && b.last_actions &&
                   b.last_last_actions && b.last_dof_pos && b.last_dof_vel && b.torques && b.last_torques &&
                   b.last_root_vel && b.commands && b.episode_length_buf && b.last_contacts && b.contact_filt &&
                   b.feet_air_time && b.disturbance && b.base_lin_vel && b.base_ang_vel && b.projected_gravity &&
                   b.measured_heights && b.reset_buf && b.time_out_buf && b.rew_buf && b.obs_buf_in && b.obs_buf_out &&
                   b.privileged_obs_buf,
               "null buffer");
  HL_CHECK_ARG(cfg->mesh_type == 0 || b.height_min3, "the fused step needs the min3 terrain table (hl_terrain_prepare)");
  HL_CHECK_ARG(cfg->measure_heights, "the fused step needs measure_heights (privileged obs carries the scan)");
  {
    const void* al[] = {b.root_states, b.dof_state, b.contact_forces, b.actions, b.last_actions, b.last_last_actions,
                        b.last_dof_pos, b.last_dof_vel, b.torques, b.last_torques, b.last_root_vel, b.commands,
                        b.feet_air_time, b.last_contacts, b.contact_filt};
    for (const void* q : al) HL_CHECK_ARG(((uintptr_t)q & 15) == 0, "state tensors must be 16-byte aligned");
  }
  if (n <= 0) return HL_OK;
  const int cf_stride = cfg->num_bodies * 3;   // dense slab
  int need_ldp = 0, need_ltq = 0, want_base = 0;
  for (int k = 0; k < cfg->n_terms; ++k) {
    need_ldp |= cfg->term_id[k] == T_dof_pos_dif;
    need_ltq |= cfg->term_id[k] == T_torques_dif;
    want_base |= cfg->term_id[k] == T_base_height || cfg->term_id[k] == T_base_height_up;
  }
  const int P = cfg->n_px * cfg->n_py, PB = cfg->n_bx * cfg->n_by;
  const bool cpu = cfg->index_math == HL_INDEX_MATH_TORCH_CPU;
  const cudaStream_t st = (cudaStream_t)stream;
  // |height obs| <= obs_height + noise: the +-clip_obs clip of step() is compiled out when it cannot bind
  const bool hclip = (cfg->obs_height + (cfg->add_noise ? cfg->noise_height : 0.0f)) > cfg->clip_obs;
  FusedArgs fa;
  fa.cf_stride = cf_stride;
  fa.need_ldp = need_ldp;
  fa.need_ltq = need_ltq;
  fa.want_base = want_base;
  fa.sums_aligned = (n % 4 == 0) && (((uintptr_t)b.episode_sums & 15) == 0);
  fa.hist_clipped = (int)(b.flags & HL_BUF_HISTORY_CLIPPED);
  fa.compact = b.reset_ids_out != nullptr;
  HL_CHECK_ARG(!fa.compact || (b.n_reset_out && b.term_priv_out && b.fused_ws), "single-launch mode needs n_reset_out, term_priv_out, fused_ws");
  fa.tma_ok = 0;
  fa.hist_pf = 0;
  {
    uint32_t x = (uint32_t)b.philox_seed, y = (uint32_t)(b.philox_seed >> 32);
    for (int r = 0; r < 10; ++r) {
      fa.keys.kx[r] = x;
      fa.keys.ky[r] = y;
      x += 0x9E3779B9u;
      y += 0xBB67AE85u;
    }
  }
  const bool fast = P > 160 && P <= 192 && PB <= 64 && !hclip;
  {
    bool ok = (n % 4 == 0) && (!b.episode_sums || ((uintptr_t)b.episode_sums & 15) == 0);
    fa.tma_ok = ok;
    fa.rs_interval = 0;
    fa.rs_uniforms = nullptr;
    fa.rs_ranges = nullptr;
    if (b.resample_host && b.resample_interval > 0) {
      const HlReset* r = b.resample_host;
      HL_CHECK_ARG(r->struct_bytes == (int)sizeof(HlReset), "resample_host: HlReset size mismatch");
      fa.rs_interval = b.resample_interval;
      fa.rs_heading = r->heading_command;
      fa.rs_hi_envs = (long long)r->high_vel_envs;
      fa.rs_lin_vel_x[0] = r->cmd_lin_vel_x[0]; fa.rs_lin_vel_x[1] = r->cmd_lin_vel_x[1];
      fa.rs_lin_vel_y[0] = r->cmd_lin_vel_y[0]; fa.rs_lin_vel_y[1] = r->cmd_lin_vel_y[1];
      const float* third = r->heading_command ? r->cmd_heading : r->cmd_ang_vel_yaw;
      fa.rs_third[0] = third[0]; fa.rs_third[1] = third[1];
      fa.rs_uniforms = r->uniforms;
      fa.rs_ranges = r->cmd_ranges;
    }
    const char* pf = getenv("HL_PK_HIST_PF");   // experiment knob
    fa.hist_pf = (((uintptr_t)b.obs_buf_in & 15) == 0) && !(pf && pf[0] == '0');
  }
  // HL_FUSED_IMPL=persist selects the persistent role-pipelined kernel (hl_persist_kernel.inc)
  const char* impl = getenv("HL_FUSED_IMPL");
  if (fast && impl && impl[0] == 'p') {
    const int prc = pk::run(cfg, bufs, n, fa, cpu, device_sms(), st);
    if (prc != HL_E_UNSUPPORTED) {
      if (prc) return prc;
      HL_CHECK_LAUNCH();
      g_fused_last_impl = 1;
      return HL_OK;
    }
  }
  HL_CHECK_ARG(!fa.compact || b.fused_ws, "single-launch mode needs fused_ws");
  {  // the tiled kernel stages its slabs with LDG.128 -> STS.128 by default: the TMA bulk-copy form (HL_FUSED_TMA=1) measured
     // 104.5 vs 102.2 us at 65,536 envs -- phase 0 is bound by the load round trip, not by the staging instructions
    const char* t = getenv("HL_FUSED_TMA");
    if (!(t && t[0] == '1')) fa.tma_ok = 0;
  }
  unsigned long long rmask = 0ull;   // active reward terms as a bit set (0 when not in sorted order: the generic loop keeps the caller's order)
  for (int k = 0; k < cfg->n_terms; ++k) {
    if (cfg->term_id[k] < 0 || cfg->term_id[k] >= T_COUNT || (k > 0 && cfg->term_id[k] <= cfg->term_id[k - 1])) {
      rmask = 0ull;
      break;
    }
    rmask |= 1ull << cfg->term_id[k];
  }
  { const char* g = getenv("HL_FUSED_GENERIC_REWARD"); if (g && g[0] == '1') rmask = 0ull; }   // A/B knob
  const int tile = pick_tile(n);
  int rc = HL_E_UNSUPPORTED;
  if (tile == 52) rc = fk52::run(cfg, bufs, n, fa, fast, cpu, rmask, st);
  else if (tile == 32) rc = fk32::run(cfg, bufs, n, fa, fast, cpu, rmask, st);
  if (rc == HL_E_UNSUPPORTED) rc = fk64::run(cfg, bufs, n, fa, fast, cpu, rmask, st);
  if (rc) return rc;
  HL_CHECK_LAUNCH();
  g_fused_last_impl = 0;
  return HL_OK;
}
