// Keyed domain randomisation (sm_100a): the action delay of step() (LR:133-138, with step()'s clip) and the interval
// disturbance (LR:838-844) / push (LR:822-828) draws, from Philox streams 4-6 keyed by (seed, step, global env id)
// like every other in-kernel draw, so they depend on neither the launch mode nor the sharding; and HIMPPO.act's action
// sampling (him_ppo.py:90) from stream 7.  See include/himloco_b200.h for the ABI.
#include "hl_common.cuh"

static int check_structs(const HlCfg* c, const HlEnvBuffers* b) {
  if (!c || c->struct_bytes != (int)sizeof(HlCfg)) {
    hl_set_error("HlCfg size mismatch (binding %d vs library %d)", c ? c->struct_bytes : -1, (int)sizeof(HlCfg));
    return HL_E_INVALID;
  }
  if (!b || b->struct_bytes != (int)sizeof(HlEnvBuffers)) {
    hl_set_error("HlEnvBuffers size mismatch (binding %d vs library %d)", b ? b->struct_bytes : -1, (int)sizeof(HlEnvBuffers));
    return HL_E_INVALID;
  }
  return HL_OK;
}

// ============================================================================= clip + action delay
// CTA = DL_ENVS envs.  Phase 1: the tile's actions are clipped (written out and kept in shared memory with last_actions)
// and one thread per env takes its delay.  Phase 2: the tile's (DL_ENVS, decimation, 12) slab of delayed_actions, one
// contiguous run of stores.  Each element is read and written by the same thread, so actions_out may alias actions_in.
constexpr int DL_ENVS = 64, DL_THREADS = 256;

__global__ void __launch_bounds__(DL_THREADS) hl_delay_actions_kernel(HlEnvBuffers b, long long env_off, const float* a_in,
                                                                    float* a_out, float* __restrict__ delayed, int dec, int draw,
                                                                    float clip, const long long* __restrict__ delay_in,
                                                                    long long n) {
  __shared__ float s_act[DL_ENVS * HL_NUM_DOF], s_last[DL_ENVS * HL_NUM_DOF];
  __shared__ int s_d[DL_ENVS];
  hl_pdl_enter();
  const int tid = threadIdx.x;
  const long long e0 = (long long)blockIdx.x * DL_ENVS;
  const int cnt = (int)((n - e0) < DL_ENVS ? (n - e0) : DL_ENVS);
  const long long base = e0 * HL_NUM_DOF;
  for (int i = tid; i < cnt * HL_NUM_DOF; i += DL_THREADS) {
    const float x = a_in[base + i];
    const float c = isnan(x) ? x : fminf(fmaxf(x, -clip), clip);   // torch.clamp: NaN passes through (hl_clampf drops it)
    a_out[base + i] = c;
    s_act[i] = c;
    if (draw) s_last[i] = b.last_actions[base + i];
  }
  if (draw && tid < cnt) {
    int d;
    if (delay_in) {
      const long long v = delay_in[e0 + tid];                       // host-checked to lie in [0, decimation)
      d = v < 0 ? 0 : (v > dec ? dec : (int)v);
    } else {
      const uint4 q = hl_noise_block(b.philox_seed, hl_step_key(b), (unsigned long long)(e0 + tid + env_off), 0u, 4u);
      d = (int)__umulhi(q.x, (unsigned)dec);                          // floor(x * dec / 2^32): uniform on [0, dec)
    }
    s_d[tid] = d;
  }
  __syncthreads();
  const int per = dec * HL_NUM_DOF;
  float* __restrict__ out = delayed + e0 * per;
  for (int i = tid; i < cnt * per; i += DL_THREADS) {
    const int le = i / per, r = i - le * per, k = r / HL_NUM_DOF, j = r - k * HL_NUM_DOF;
    const float act = s_act[le * HL_NUM_DOF + j];
    float v = act;
    if (draw) {
      // _delay_actions: last + (actions - last) * mask, each op rounded on its own as the three torch launches do
      const float last = s_last[le * HL_NUM_DOF + j];
      const float m = k >= s_d[le] ? 1.0f : 0.0f;
      v = __fadd_rn(last, __fmul_rn(__fsub_rn(act, last), m));
    }
    out[i] = v;
  }
}

extern "C" int hl_delay_actions(const HlCfg* cfg, const HlEnvBuffers* bufs, const float* actions_in, float* actions_out,
                                float* delayed_out, int32_t decimation, int32_t delay, float clip_actions,
                                const int64_t* delay_in, int64_t n_envs, void* stream) {
  if (int rc = check_structs(cfg, bufs)) return rc;
  HL_CHECK_ARG(actions_in && actions_out && delayed_out, "null actions");
  HL_CHECK_ARG(decimation >= 1 && decimation <= 16, "decimation must lie in [1, 16]");
  HL_CHECK_ARG(!delay || bufs->last_actions, "the delay needs bufs->last_actions");
  HL_CHECK_ARG(n_envs >= 0, "negative n_envs");
  if (n_envs == 0) return HL_OK;
  hl_launch(hl_delay_actions_kernel, dim3((unsigned)((n_envs + DL_ENVS - 1) / DL_ENVS)), dim3(DL_THREADS), 0,
            (cudaStream_t)stream, *bufs, (long long)cfg->env_id_offset, actions_in, actions_out, delayed_out, (int)decimation,
            delay ? 1 : 0, clip_actions, (const long long*)delay_in, (long long)n_envs);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= uniform rows (disturbance, push)
// One thread per env: `cols` uniforms from one Philox block (or the pre-drawn row), scaled as torch_rand_float does.
__global__ void __launch_bounds__(256) hl_uniform_rows_kernel(HlEnvBuffers b, long long env_off, float* __restrict__ dst,
                                                              long long row_stride, int cols, float scale, float lo,
                                                              const float* __restrict__ u_in, unsigned stream_id, long long n) {
  hl_pdl_enter();
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  float u[4];
  if (u_in) {
    for (int c = 0; c < cols; ++c) u[c] = u_in[e * cols + c];
  } else {
    const uint4 q = hl_noise_block(b.philox_seed, hl_step_key(b), (unsigned long long)(e + env_off), 0u, stream_id);
    u[0] = hl_u01(q.x);
    u[1] = hl_u01(q.y);
    u[2] = hl_u01(q.z);
    u[3] = hl_u01(q.w);
  }
  for (int c = 0; c < cols; ++c) dst[e * row_stride + c] = __fadd_rn(__fmul_rn(scale, u[c]), lo);
}

extern "C" int hl_uniform_rows(const HlCfg* cfg, const HlEnvBuffers* bufs, float* dst, int64_t row_stride, int32_t cols,
                               double lo, double hi, const float* u_in, int32_t stream_id, int64_t n_envs, void* stream) {
  if (int rc = check_structs(cfg, bufs)) return rc;
  HL_CHECK_ARG(dst, "null dst");
  HL_CHECK_ARG(cols >= 1 && cols <= 4, "cols must lie in [1, 4]");
  HL_CHECK_ARG(row_stride >= cols, "row_stride must be at least cols");
  HL_CHECK_ARG(stream_id >= 4 && stream_id <= 255, "stream_id must lie in [4, 255] (streams 0-3 belong to other draws)");
  HL_CHECK_ARG(n_envs >= 0, "negative n_envs");
  if (n_envs == 0) return HL_OK;
  // torch_rand_float(lo, hi): (hi - lo) is a Python float, rounded to fp32 once by the tensor multiply
  hl_launch(hl_uniform_rows_kernel, dim3((unsigned)((n_envs + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, *bufs,
            (long long)cfg->env_id_offset, dst, (long long)row_stride, (int)cols, (float)(hi - lo), (float)lo, u_in,
            (unsigned)stream_id, (long long)n_envs);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= policy action sampling
// CTA = PS_ENVS envs, one thread per env.  Phase 1: the tile's means are staged in shared memory (coalesced).  Phase 2:
// each thread draws its ceil(A/4) Philox blocks (stream 7), forms sigma, the action and the log-probability terms in
// column order (the sequential sum), and leaves its actions in shared memory.  Phase 3: actions, mu and sigma are
// stored as contiguous runs.  Every op is rounded on its own, in the order of torch's Normal (no contraction).
constexpr int PS_ENVS = 128, PS_MAX_A = 16;

__global__ void __launch_bounds__(PS_ENVS) hl_policy_sample_kernel(HlEnvBuffers b, long long env_off, const float* mean,
                                                                   const float* __restrict__ std_dev, int std_rows,
                                                                   const float* __restrict__ z_in, int A, float* act_out,
                                                                   float* __restrict__ logp_out, float* mu_out,
                                                                   float* __restrict__ sigma_out, long long n) {
  __shared__ float s_mean[PS_ENVS * PS_MAX_A], s_act[PS_ENVS * PS_MAX_A];
  hl_pdl_enter();
  const int tid = threadIdx.x;
  const long long e0 = (long long)blockIdx.x * PS_ENVS;
  const int cnt = (int)((n - e0) < PS_ENVS ? (n - e0) : PS_ENVS);
  const long long base = e0 * A;
  for (int i = tid; i < cnt * A; i += PS_ENVS) s_mean[i] = mean[base + i];
  __syncthreads();
  if (tid < cnt) {
    const long long e = e0 + tid;
    const unsigned long long key = hl_step_key(b);
    const float* srow = std_rows ? std_dev + e * A : std_dev;
    float lp = 0.0f;
    for (int blk = 0; blk * 4 < A; ++blk) {
      float z[4];
      if (z_in) {
        for (int k = 0; k < 4; ++k) z[k] = (blk * 4 + k < A) ? z_in[e * A + blk * 4 + k] : 0.0f;
      } else {
        const uint4 q = hl_noise_block(b.philox_seed, key, (unsigned long long)(e + env_off), (unsigned)blk, 7u);
        // Box-Muller on (x, y) and (z, w): u1 = 1 - u lies in [2^-24, 1], so |z| <= sqrt(-2 ln 2^-24) = sqrt(48 ln 2)
        const float r0 = sqrtf(__fmul_rn(-2.0f, logf(__fsub_rn(1.0f, hl_u01(q.x)))));
        const float r1 = sqrtf(__fmul_rn(-2.0f, logf(__fsub_rn(1.0f, hl_u01(q.z)))));
        float s0, c0, s1, c1;
        sincospif(__fmul_rn(2.0f, hl_u01(q.y)), &s0, &c0);
        sincospif(__fmul_rn(2.0f, hl_u01(q.w)), &s1, &c1);
        z[0] = __fmul_rn(r0, c0);
        z[1] = __fmul_rn(r0, s0);
        z[2] = __fmul_rn(r1, c1);
        z[3] = __fmul_rn(r1, s1);
      }
      for (int k = 0; k < 4; ++k) {
        const int j = blk * 4 + k;
        if (j >= A) break;
        const float m = s_mean[tid * A + j];
        const float sig = __fadd_rn(__fmul_rn(m, 0.0f), srow[j]);          // mean*0. + std
        const float a = __fadd_rn(m, __fmul_rn(z[k], sig));                  // loc + eps * scale
        s_act[tid * A + j] = a;
        // Normal.log_prob: -((value - loc) ** 2) / (2 * var) - log(scale) - log(sqrt(2 pi))
        const float d = __fsub_rn(a, m);
        const float q = __fdiv_rn(-__fmul_rn(d, d), __fmul_rn(2.0f, __fmul_rn(sig, sig)));
        lp = __fadd_rn(lp, __fsub_rn(__fsub_rn(q, logf(sig)), (float)0.9189385332046727));
      }
    }
    logp_out[e] = lp;
  }
  __syncthreads();
  for (int i = tid; i < cnt * A; i += PS_ENVS) {
    const float m = s_mean[i];
    act_out[base + i] = s_act[i];
    if (mu_out) mu_out[base + i] = m;
    if (sigma_out) sigma_out[base + i] = __fadd_rn(__fmul_rn(m, 0.0f), std_rows ? std_dev[base + i] : std_dev[i % A]);
  }
}

extern "C" int hl_policy_sample(const HlCfg* cfg, const HlEnvBuffers* bufs, const float* mean, const float* std_dev,
                                int64_t std_row_stride, const float* z_in, int32_t act_dim, float* actions_out,
                                float* log_prob_out, float* mu_out, float* sigma_out, int64_t n_envs, void* stream) {
  if (int rc = check_structs(cfg, bufs)) return rc;
  HL_CHECK_ARG(mean && std_dev && actions_out && log_prob_out, "null mean, std, actions_out or log_prob_out");
  HL_CHECK_ARG(act_dim >= 1 && act_dim <= PS_MAX_A, "act_dim must lie in [1, 16]");
  HL_CHECK_ARG(std_row_stride == 0 || std_row_stride == act_dim, "std_row_stride must be 0 or act_dim");
  HL_CHECK_ARG(n_envs >= 0, "negative n_envs");
  if (n_envs == 0) return HL_OK;
  hl_launch(hl_policy_sample_kernel, dim3((unsigned)((n_envs + PS_ENVS - 1) / PS_ENVS)), dim3(PS_ENVS), 0,
            (cudaStream_t)stream, *bufs, (long long)cfg->env_id_offset, mean, std_dev, std_row_stride ? 1 : 0, z_in,
            (int)act_dim, actions_out, log_prob_out, mu_out == mean ? (float*)nullptr : mu_out, sigma_out,
            (long long)n_envs);
  HL_CHECK_LAUNCH();
  return HL_OK;
}
