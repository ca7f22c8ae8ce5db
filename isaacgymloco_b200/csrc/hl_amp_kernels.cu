// AMP data path (sm_100a): mocap frame interpolation, expert-pair gather, discriminator input
// assembly / reward epilogue, normaliser batch moments.
// Reference: rsl_rl/rsl_rl/datasets/motion_loader.py (ML), rsl_rl/rsl_rl/utils/utils.py (UT),
// rsl_rl/rsl_rl/algorithms/amp_discriminator.py (DISC), rsl_rl/rsl_rl/runners/hybrid_runner.py.
#include "hl_common.cuh"

// ============================================================================= a16: frame blend
// ML:231-255.  CTA = 128 samples.  Phase 1 (one lane per sample): float64 index math exactly as
// numpy does it (p = t/len; lo = floor(p n); hi = ceil(p n); blend = fp32(p n - lo)) and the
// quaternion_slerp coefficients of UT:153-186 (mask precedence zero -> one -> dist -> angle ->
// general, 1/angle scaling, no renormalisation).  Phase 2 (coalesced over the 49 columns):
// lerp `(1-b) v0 + b v1` with every op rounded separately, like the eager reference.
constexpr int BLEND_SAMPLES = 128;
struct BlendRow {
  int lo, hi;      // absolute row in the stacked frame table
  float blend;
  float c0, c1;    // quaternion: out = c0*q0 + c1*q1   (c1 carries the shortest-path sign)
};

__global__ void __launch_bounds__(BLEND_SAMPLES) hl_amp_blend_kernel(
    const float* __restrict__ frames, const int* __restrict__ clip_offset, const double* __restrict__ clip_len,
    const double* __restrict__ clip_nf, int n_clips, const long long* __restrict__ traj, const double* __restrict__ times,
    float* __restrict__ out, int* __restrict__ lo_out, int* __restrict__ hi_out, long long batch) {
  __shared__ BlendRow rows[BLEND_SAMPLES];
  const long long s0 = (long long)blockIdx.x * BLEND_SAMPLES;
  const int cnt = (int)((batch - s0) < BLEND_SAMPLES ? (batch - s0) : BLEND_SAMPLES);
  const int tid = threadIdx.x;
  if (tid < cnt) {
    const long long smp = s0 + tid;
    long long ti = traj[smp];
    ti = ti < 0 ? 0 : (ti >= n_clips ? n_clips - 1 : ti);
    const double p = times[smp] / clip_len[ti];
    const double pn = p * clip_nf[ti];
    const double flo = floor(pn), fhi = ceil(pn);
    const int lo = (int)flo, hi = (int)fhi;
    const float blend = (float)(pn - flo);
    BlendRow r;
    // times outside [0, len (n-1)/n] index past the clip (the reference raises IndexError, the host
    // wrapper does too); the reads are clamped to the clip so the kernel itself stays memory-safe
    const int last = (int)clip_nf[ti] - 1;
    r.lo = clip_offset[ti] + min(max(lo, 0), last);
    r.hi = clip_offset[ti] + min(max(hi, 0), last);
    r.blend = blend;
    if (lo_out) lo_out[smp] = lo;
    if (hi_out) hi_out[smp] = hi;
    const float* q0 = frames + (long long)r.lo * HL_AMP_FRAME + 3;
    const float* q1 = frames + (long long)r.hi * HL_AMP_FRAME + 3;
    // torch.isclose(f, 0/1): |f - t| <= 1e-8 + 1e-5 |t|
    const bool m_zero = fabsf(blend) <= 1e-8f;
    const bool m_one = fabsf(blend - 1.0f) <= (float)(1e-8 + 1e-5);
    float d = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(q0[0], q1[0]), __fmul_rn(q0[1], q1[1])), __fmul_rn(q0[2], q1[2])),
                        __fmul_rn(q0[3], q1[3]));
    const float eps = 8.881784197001252e-16f;  // np.finfo(float).eps * 4
    const bool m_dist = fabsf(fabsf(d) - 1.0f) < eps;
    const float sgn = d < 0.0f ? -1.0f : 1.0f;
    d = d < 0.0f ? -d : d;
    const float angle = acosf(d);
    const bool m_ang = fabsf(angle) < eps;
    float c0, c1;
    if (m_ang || m_dist) { c0 = 1.0f; c1 = 0.0f; }           // out = q0 (later assignments win)
    else if (m_one) { c0 = 0.0f; c1 = 1.0f; }                // out = q1 (the un-flipped one)
    else if (m_zero) { c0 = 1.0f; c1 = 0.0f; }
    else {
      const float isin = 1.0f / angle;
      c0 = __fmul_rn(sinf(__fmul_rn(__fsub_rn(1.0f, blend), angle)), isin);
      c1 = __fmul_rn(sinf(__fmul_rn(blend, angle)), isin) * sgn;
    }
    r.c0 = c0;
    r.c1 = c1;
    rows[tid] = r;
  }
  __syncthreads();
  const int total = cnt * HL_AMP_FRAME;
  for (int i = tid; i < total; i += BLEND_SAMPLES) {
    const int s = i / HL_AMP_FRAME, k = i - s * HL_AMP_FRAME;
    const BlendRow r = rows[s];
    const float v0 = __ldg(frames + (long long)r.lo * HL_AMP_FRAME + k);
    const float v1 = __ldg(frames + (long long)r.hi * HL_AMP_FRAME + k);
    float o;
    if (k >= 3 && k < 7) {
      // exact copies stay exact (c = 1/0 selects q0/q1); general case q0*c0 + (sgn q1)*c1
      o = (r.c1 == 0.0f && r.c0 == 1.0f) ? v0 : ((r.c0 == 0.0f && r.c1 == 1.0f) ? v1 : __fadd_rn(__fmul_rn(v0, r.c0), __fmul_rn(v1, r.c1)));
    } else {
      o = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, r.blend), v0), __fmul_rn(r.blend, v1));
    }
    out[(s0 + s) * HL_AMP_FRAME + k] = o;
  }
}

extern "C" int hl_amp_frame_blend(const float* frames, const int32_t* clip_offset, const double* clip_len,
                                  const double* clip_nf, int32_t n_clips, const int64_t* traj_idxs, const double* times,
                                  float* out, int32_t* lo_out, int32_t* hi_out, int64_t batch, void* stream) {
  HL_CHECK_ARG(frames && clip_offset && clip_len && clip_nf && traj_idxs && times && out && n_clips > 0, "null pointer");
  if (batch <= 0) return HL_OK;
  const unsigned blocks = (unsigned)((batch + BLEND_SAMPLES - 1) / BLEND_SAMPLES);
  hl_amp_blend_kernel<<<blocks, BLEND_SAMPLES, 0, (cudaStream_t)stream>>>(frames, clip_offset, clip_len, clip_nf, n_clips,
                                                                          (const long long*)traj_idxs, times, out, lo_out,
                                                                          hi_out, batch);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= a17: expert pairs
// ML:321-330: s = cat(pre_s[idx, 7:19], pre_s[idx, 31:49]), same for pre_s_next.
__global__ void __launch_bounds__(256) hl_amp_gather_kernel(const float* __restrict__ pre_s, const float* __restrict__ pre_sn,
                                                            long long n_pre, const long long* __restrict__ idxs,
                                                            float* __restrict__ s_out, float* __restrict__ sn_out,
                                                            long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long row = i / HL_AMP_OBS;
  const int col = (int)(i - row * HL_AMP_OBS);
  long long idx = idxs[row];
  idx = idx < 0 ? idx + n_pre : idx;
  const int src = col < 12 ? 7 + col : 31 + (col - 12);
  s_out[i] = __ldg(pre_s + idx * HL_AMP_FRAME + src);
  sn_out[i] = __ldg(pre_sn + idx * HL_AMP_FRAME + src);
}
extern "C" int hl_amp_gather_pairs(const float* pre_s, const float* pre_sn, int64_t n_pre, const int64_t* idxs,
                                   float* s_out, float* sn_out, int64_t batch, void* stream) {
  HL_CHECK_ARG(pre_s && pre_sn && idxs && s_out && sn_out && n_pre > 0, "null pointer");
  if (batch <= 0) return HL_OK;
  const long long total = batch * HL_AMP_OBS;
  hl_amp_gather_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(pre_s, pre_sn, n_pre,
                                                                                        (const long long*)idxs, s_out, sn_out, total);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= a19: disc input
// DISC:59-63 + UT:124-130 + hybrid_runner.py:191-192.  One thread per (env, column of 60).
__global__ void __launch_bounds__(256) hl_amp_disc_input_kernel(const float* __restrict__ state, const float* __restrict__ next_state,
                                                                const float* __restrict__ mean, const float* __restrict__ stdv,
                                                                float clip, const long long* __restrict__ reset_ids,
                                                                const int* __restrict__ n_reset,
                                                                const float* __restrict__ terminal,
                                                                float* __restrict__ patched, float* __restrict__ x, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long e = i / 60;
  const int col = (int)(i - e * 60);
  const int k = col < 30 ? col : col - 30;
  float v;
  if (col < 30) {
    v = state[e * 30 + k];
  } else {
    v = next_state[e * 30 + k];
    if (reset_ids) {  // next_amp_obs_with_term[reset_env_ids] = terminal_amp_states
      int lo = 0, hi = *n_reset;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (reset_ids[mid] < e) lo = mid + 1; else hi = mid;
      }
      if (lo < *n_reset && reset_ids[lo] == e) v = terminal[(long long)lo * 30 + k];
    }
    if (patched) patched[e * 30 + k] = v;
  }
  if (mean && stdv) v = hl_clampf(__fdiv_rn(__fsub_rn(v, mean[k]), stdv[k]), -clip, clip);
  x[i] = v;
}
extern "C" int hl_amp_disc_input(const float* state, const float* next_state, const float* mean, const float* std_,
                                 float clip, const int64_t* reset_ids, const int32_t* n_reset_dev,
                                 const float* terminal_states, float* patched_out, float* x_out, int64_t n, void* stream) {
  HL_CHECK_ARG(state && next_state && x_out, "null pointer");
  HL_CHECK_ARG((mean == nullptr) == (std_ == nullptr), "mean and std go together");
  HL_CHECK_ARG(!reset_ids || (n_reset_dev && terminal_states), "terminal patch needs ids, count and rows");
  if (n <= 0) return HL_OK;
  const long long total = n * 60;
  hl_amp_disc_input_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      state, next_state, mean, std_, clip, (const long long*)reset_ids, n_reset_dev, terminal_states, patched_out, x_out, total);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// DISC:64-68,70-72
__global__ void __launch_bounds__(256) hl_amp_reward_kernel(const float* __restrict__ d, const float* __restrict__ task_r,
                                                            float coef, float lerp, float* __restrict__ out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float t = __fsub_rn(d[i], 1.0f);
  float r = __fmul_rn(coef, fmaxf(__fsub_rn(1.0f, __fmul_rn(0.25f, __fmul_rn(t, t))), 0.0f));
  if (lerp > 0.0f) r = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, lerp), r), __fmul_rn(lerp, task_r[i]));
  out[i] = r;
}
extern "C" int hl_amp_reward(const float* d_logits, const float* task_reward, float coef, float lerp, float* reward_out,
                             int64_t n, void* stream) {
  HL_CHECK_ARG(d_logits && reward_out && (lerp <= 0.0f || task_reward), "null pointer");
  if (n <= 0) return HL_OK;
  hl_amp_reward_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_logits, task_reward, coef, lerp,
                                                                                    reward_out, n);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= AMP transition of one env-step
// hybrid_runner.py:184-195 minus the discriminator MLP, for a captured rollout: the next AMP observation (LR:406-416,
// hl_amp_obs_kernel's columns), the terminal patch with the count read on the device, the normalised discriminator input,
// the replay-ring insert at the device cursor (replay_buffer.py:52-68) and the carried amp_obs.  CTA = 64 envs: lane t
// of the first 64 finds env e0+t's terminal row (binary search only where reset_buf is set), then the CTA walks the
// tile's 64 x 30 columns coalesced.  cursor = {step, num_samples, CTA ticket}: every CTA reads step after
// griddepcontrol.wait; the last CTA to take a ticket advances the cursor with the reference's arithmetic and re-arms
// the ticket, so the launch is graph-safe.
constexpr int TRANS_ENVS = 64, TRANS_THREADS = 256;
__global__ void __launch_bounds__(TRANS_THREADS) hl_amp_transition_kernel(
    const float* __restrict__ dof, const float* __restrict__ blv, const float* __restrict__ bav,
    const unsigned char* __restrict__ reset_buf, const long long* __restrict__ reset_ids, const int* __restrict__ n_reset,
    const float* __restrict__ terminal, const double* __restrict__ stats, double eps, float clip, float* __restrict__ amp_obs,
    float* __restrict__ x, float* __restrict__ ring_s, float* __restrict__ ring_n, long long ring_rows,
    long long* __restrict__ cursor, long long n) {
  __shared__ float s_mean[HL_AMP_OBS], s_std[HL_AMP_OBS];
  __shared__ int s_row[TRANS_ENVS];          // terminal row of each env of the tile, -1 = none
  __shared__ long long s_step, s_nsamp;
  hl_pdl_enter();
  const int tid = threadIdx.x;
  const long long e0 = (long long)blockIdx.x * TRANS_ENVS;
  const int cnt = (int)(n - e0 < TRANS_ENVS ? n - e0 : TRANS_ENVS);
  if (tid == 0) {
    s_step = cursor[0];
    s_nsamp = cursor[1];
  }
  // Normalizer.mean_std_f32(): fp32(mean), sqrt(fp32(var + eps)) with the add in float64
  if (stats && tid < HL_AMP_OBS) {
    s_mean[tid] = (float)stats[tid];
    s_std[tid] = __fsqrt_rn((float)(stats[HL_AMP_OBS + tid] + eps));
  }
  if (tid < cnt) {
    const long long e = e0 + tid;
    int row = -1;
    if (reset_buf[e]) {       // reset_buf is set exactly for this step's ids: only these envs search
      const int m = *n_reset;
      int lo = 0, hi = m;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (reset_ids[mid] < e) lo = mid + 1; else hi = mid;
      }
      if (lo < m && reset_ids[lo] == e) row = lo;
    }
    s_row[tid] = row;
  }
  __syncthreads();
  const long long step = s_step;
  for (int i = tid; i < cnt * HL_AMP_OBS; i += TRANS_THREADS) {
    const int le = i / HL_AMP_OBS, k = i - le * HL_AMP_OBS;
    const long long e = e0 + le;
    float nx;
    if (k < 12) nx = dof[e * 24 + 2 * k];
    else if (k < 15) nx = blv[e * 3 + (k - 12)];
    else if (k < 18) nx = bav[e * 3 + (k - 15)];
    else nx = dof[e * 24 + 2 * (k - 18) + 1];
    const int row = s_row[le];
    const float nt = row >= 0 ? terminal[(long long)row * HL_AMP_OBS + k] : nx;
    const float s = amp_obs[e * HL_AMP_OBS + k];
    long long r = step + e;                  // step < ring_rows and e < n <= ring_rows
    if (r >= ring_rows) r -= ring_rows;
    ring_s[r * HL_AMP_OBS + k] = s;
    ring_n[r * HL_AMP_OBS + k] = nt;
    float a = s, b = nt;
    if (stats) {
      a = hl_clampf(__fdiv_rn(__fsub_rn(a, s_mean[k]), s_std[k]), -clip, clip);
      b = hl_clampf(__fdiv_rn(__fsub_rn(b, s_mean[k]), s_std[k]), -clip, clip);
    }
    x[e * 60 + k] = a;
    x[e * 60 + HL_AMP_OBS + k] = b;
    amp_obs[e * HL_AMP_OBS + k] = nx;        // amp_obs = next_amp_obs.clone(): the un-patched observation
  }
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    unsigned long long* ticket = reinterpret_cast<unsigned long long*>(cursor + 2);
    if (atomicAdd(ticket, 1ull) == (unsigned long long)gridDim.x - 1ull) {   // every other CTA has read the cursor
      const long long end = step + n, most = end > s_nsamp ? end : s_nsamp;
      cursor[1] = most < ring_rows ? most : ring_rows;    // min(size, max(step + N, num_samples))
      cursor[0] = end >= ring_rows ? end - ring_rows : end;   // (step + N) % size
      *ticket = 0ull;
    }
  }
}

extern "C" int hl_amp_transition(const float* dof_state, const float* base_lin_vel, const float* base_ang_vel,
                                 const uint8_t* reset_buf, const int64_t* reset_ids, const int32_t* n_reset_dev,
                                 const float* terminal_amp, const double* norm_stats, double eps, float clip, float* amp_obs,
                                 float* x_out, float* ring_states, float* ring_next, int64_t ring_rows, int64_t* cursor,
                                 int64_t n_envs, void* stream) {
  HL_CHECK_ARG(dof_state && base_lin_vel && base_ang_vel && amp_obs && x_out, "null pointer");
  HL_CHECK_ARG(reset_buf && reset_ids && n_reset_dev && terminal_amp, "terminal patch needs reset_buf, ids, count and rows");
  HL_CHECK_ARG(ring_states && ring_next && cursor, "null ring or cursor");
  HL_CHECK_ARG(ring_rows > 0 && n_envs <= ring_rows, "n_envs must not exceed the ring's rows");
  if (n_envs <= 0) return HL_OK;
  const unsigned blocks = (unsigned)((n_envs + TRANS_ENVS - 1) / TRANS_ENVS);
  hl_launch(hl_amp_transition_kernel, dim3(blocks), dim3(TRANS_THREADS), 0, (cudaStream_t)stream, dof_state, base_lin_vel,
            base_ang_vel, (const unsigned char*)reset_buf, (const long long*)reset_ids, n_reset_dev, terminal_amp, norm_stats,
            eps, clip, amp_obs, x_out, ring_states, ring_next, (long long)ring_rows, (long long*)cursor, (long long)n_envs);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= AMP update minibatch
// HybridPPO.update's two discriminator batches (hybrid_ppo.py:160-281): amp_storage.feed_forward_generator's ring rows
// (replay_buffer.py:70-74), amp_data.feed_forward_generator's preload pairs (ML:315-343) and the normalised 60-wide
// inputs, for rows drawn from Philox stream 8 instead of host np.random.choice.  CTA = 64 rows: lane t of the first 64
// draws (or reads) row r0+t's two indices into shared memory, then the CTA walks the tile's 64 x 30 columns coalesced
// and writes the four raw states and both normalised inputs.  draw_counter = {draws, CTA ticket}: every CTA reads the
// key after griddepcontrol.wait; the last CTA to take a ticket advances it and re-arms the ticket (graph-safe).
constexpr int UPD_ROWS = 64, UPD_THREADS = 256;
__global__ void __launch_bounds__(UPD_THREADS) hl_amp_update_batch_kernel(HlAmpUpdateBatch a) {
  __shared__ float s_mean[HL_AMP_OBS], s_std[HL_AMP_OBS];
  __shared__ long long s_p[UPD_ROWS], s_x[UPD_ROWS];   // policy ring row, expert preload row; -1 = out of range
  __shared__ long long s_key, s_ns;
  hl_pdl_enter();
  const int tid = threadIdx.x;
  const long long r0 = (long long)blockIdx.x * UPD_ROWS;
  const int cnt = (int)(a.mb - r0 < UPD_ROWS ? a.mb - r0 : UPD_ROWS);
  const bool norm = a.norm_mean != nullptr;
  if (tid == 0) {
    s_key = a.draw_counter[0];
    const long long ns = a.ring_cursor ? a.ring_cursor[1] : a.num_samples;
    s_ns = ns < 1 ? 1 : ns;
  }
  // Normalizer.mean_std_f32(): fp32(mean), sqrt(fp32(var + eps)) with the add in float64
  if (norm && tid < HL_AMP_OBS) {
    s_mean[tid] = (float)a.norm_mean[tid];
    s_std[tid] = __fsqrt_rn((float)(a.norm_var[tid] + a.eps));
  }
  __syncthreads();
  if (tid < cnt) {
    const long long r = r0 + tid;
    long long p, x;
    if (a.idx_in) {
      p = a.idx_in[2 * r];
      x = a.idx_in[2 * r + 1];
    } else {
      // floor(u n / 2^64) of a 64-bit word: bias below n / 2^64
      const uint4 q = hl_noise_block(a.seed, (uint64_t)s_key, (uint64_t)(a.row_offset + r), 0u, 8u);
      p = (long long)__umul64hi(((unsigned long long)q.x << 32) | q.y, (unsigned long long)s_ns);
      x = (long long)__umul64hi(((unsigned long long)q.z << 32) | q.w, (unsigned long long)a.n_preloaded);
    }
    if (a.idx_out) {
      a.idx_out[2 * r] = p;
      a.idx_out[2 * r + 1] = x;
    }
    const bool ok = p >= 0 && p < a.ring_rows && x >= 0 && x < a.n_preloaded;   // parity indices out of range: skipped
    s_p[tid] = ok ? p : -1;
    s_x[tid] = ok ? x : -1;
  }
  __syncthreads();
  const float clip = a.clip;
  for (int i = tid; i < cnt * HL_AMP_OBS; i += UPD_THREADS) {
    const int lr = i / HL_AMP_OBS, k = i - lr * HL_AMP_OBS;
    const long long p = s_p[lr], x = s_x[lr];
    if (p < 0) continue;
    const long long r = r0 + lr;
    const int src = k < 12 ? 7 + k : 31 + (k - 12);          // expert columns [7:19] ++ [31:49]
    const float ps = __ldg(a.ring_states + p * HL_AMP_OBS + k), pn = __ldg(a.ring_next + p * HL_AMP_OBS + k);
    const float es = __ldg(a.preloaded_s + x * HL_AMP_FRAME + src), en = __ldg(a.preloaded_s_next + x * HL_AMP_FRAME + src);
    a.policy_s[r * HL_AMP_OBS + k] = ps;
    a.policy_sn[r * HL_AMP_OBS + k] = pn;
    a.expert_s[r * HL_AMP_OBS + k] = es;
    a.expert_sn[r * HL_AMP_OBS + k] = en;
    float v0 = ps, v1 = pn, v2 = es, v3 = en;
    if (norm) {
      const float m = s_mean[k], s = s_std[k];
      v0 = hl_clampf(__fdiv_rn(__fsub_rn(v0, m), s), -clip, clip);
      v1 = hl_clampf(__fdiv_rn(__fsub_rn(v1, m), s), -clip, clip);
      v2 = hl_clampf(__fdiv_rn(__fsub_rn(v2, m), s), -clip, clip);
      v3 = hl_clampf(__fdiv_rn(__fsub_rn(v3, m), s), -clip, clip);
    }
    a.x_policy[r * 60 + k] = v0;
    a.x_policy[r * 60 + HL_AMP_OBS + k] = v1;
    a.x_expert[r * 60 + k] = v2;
    a.x_expert[r * 60 + HL_AMP_OBS + k] = v3;
  }
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    unsigned long long* ticket = reinterpret_cast<unsigned long long*>(a.draw_counter + 1);
    if (atomicAdd(ticket, 1ull) == (unsigned long long)gridDim.x - 1ull) {   // every other CTA has read the key
      a.draw_counter[0] = s_key + 1;
      *ticket = 0ull;
    }
  }
}

extern "C" int hl_sizeof_amp_update_batch(void) { return (int)sizeof(HlAmpUpdateBatch); }

extern "C" int hl_amp_update_batch(const HlAmpUpdateBatch* b, void* stream) {
  HL_CHECK_ARG(b, "null argument struct");
  HL_CHECK_ARG(b->struct_bytes == (int32_t)sizeof(HlAmpUpdateBatch), "HlAmpUpdateBatch layout mismatch");
  HL_CHECK_ARG(b->ring_states && b->ring_next && b->ring_rows > 0, "null or empty replay ring");
  HL_CHECK_ARG(b->preloaded_s && b->preloaded_s_next && b->n_preloaded > 0, "null or empty preload tables");
  HL_CHECK_ARG((b->norm_mean == nullptr) == (b->norm_var == nullptr), "norm_mean and norm_var go together");
  HL_CHECK_ARG(b->draw_counter, "null draw counter");
  HL_CHECK_ARG(b->policy_s && b->policy_sn && b->expert_s && b->expert_sn && b->x_policy && b->x_expert, "null output");
  HL_CHECK_ARG(b->row_offset >= 0, "negative row_offset");
  if (b->mb <= 0) return HL_OK;
  const unsigned blocks = (unsigned)((b->mb + UPD_ROWS - 1) / UPD_ROWS);
  hl_launch(hl_amp_update_batch_kernel, dim3(blocks), dim3(UPD_THREADS), 0, (cudaStream_t)stream, *b);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// ============================================================================= a20: batch moments
// UT:90-94 on device, float64 accumulation (the reference copies the batch to the host and uses
// numpy): pass 1 = per-block column sums / sums of squares, pass 2 = one block folds them.
constexpr int MOM_BLOCKS = 148;
__global__ void __launch_bounds__(256) hl_moments_partial_kernel(const float* __restrict__ x, long long rows, int dim,
                                                                 double* __restrict__ part) {
  __shared__ double sh1[8][32], sh2[8][32];
  const int col = threadIdx.x & 31, ry = threadIdx.x >> 5;
  for (int c0 = 0; c0 < dim; c0 += 32) {
    const int cidx = c0 + col;
    double s1 = 0.0, s2 = 0.0;
    if (cidx < dim)
      for (long long r = (long long)blockIdx.x * 8 + ry; r < rows; r += (long long)gridDim.x * 8) {
        const double v = (double)x[r * dim + cidx];
        s1 += v;
        s2 += v * v;
      }
    sh1[ry][col] = s1;
    sh2[ry][col] = s2;
    __syncthreads();
    if (ry == 0 && cidx < dim) {
      for (int k = 1; k < 8; ++k) { s1 += sh1[k][col]; s2 += sh2[k][col]; }
      part[((long long)blockIdx.x * 2 + 0) * dim + cidx] = s1;
      part[((long long)blockIdx.x * 2 + 1) * dim + cidx] = s2;
    }
    __syncthreads();
  }
}
__global__ void hl_moments_final_kernel(const double* __restrict__ part, int nblk, long long rows, int dim,
                                        double* __restrict__ out) {
  const int cidx = blockIdx.x * blockDim.x + threadIdx.x;
  if (cidx >= dim) return;
  double s1 = 0.0, s2 = 0.0;
  for (int bk = 0; bk < nblk; ++bk) {
    s1 += part[((long long)bk * 2 + 0) * dim + cidx];
    s2 += part[((long long)bk * 2 + 1) * dim + cidx];
  }
  const double mean = s1 / (double)rows;
  double var = s2 / (double)rows - mean * mean;
  out[cidx] = mean;
  out[dim + cidx] = var > 0.0 ? var : 0.0;
}
extern "C" int64_t hl_moments_workspace_bytes(int32_t dim) { return (int64_t)MOM_BLOCKS * 2 * dim * sizeof(double); }
extern "C" int hl_column_moments(const float* x, int64_t rows, int32_t dim, double* mean_var_out, void* workspace,
                                 void* stream) {
  HL_CHECK_ARG(x && mean_var_out && workspace && rows > 0 && dim > 0, "bad argument");
  hl_moments_partial_kernel<<<MOM_BLOCKS, 256, 0, (cudaStream_t)stream>>>(x, rows, dim, (double*)workspace);
  HL_CHECK_LAUNCH();
  hl_moments_final_kernel<<<(dim + 63) / 64, 64, 0, (cudaStream_t)stream>>>((const double*)workspace, MOM_BLOCKS, rows, dim,
                                                                           mean_var_out);
  HL_CHECK_LAUNCH();
  return HL_OK;
}
