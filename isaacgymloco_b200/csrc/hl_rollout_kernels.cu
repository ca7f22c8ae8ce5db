// GAE / returns (sm_100a).  Reference: HIMRolloutStorage.compute_returns,
// rsl_rl/rsl_rl/storage/him_rollout_storage.py:113-127 (== amp_rollout_storage.py:141-155).
#include "hl_common.cuh"

// One thread per env walks its T transitions backwards; consecutive threads touch consecutive
// addresses of every (T,N,1) tensor, so all traffic is coalesced.  Each op is rounded on its own
// in the reference's order (SURVEY.md A.5), which makes `returns` bit-identical to eager torch:
//   nnt = 1 - done;  delta = (r + (nnt*gamma)*V_next) - V;  A = delta + ((nnt*gamma)*lam)*A;
//   ret = A + V
// Raw advantages (ret - V) are written and their moments accumulated in float64 for the
// normalisation pass (all-reduced first when envs are sharded over GPUs).
template <int UNROLL>
__global__ void __launch_bounds__(256) hl_gae_scan_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
                                                          const uint8_t* __restrict__ dones,
                                                          const float* __restrict__ last_values,
                                                          float* __restrict__ returns, float* __restrict__ adv,
                                                          double* __restrict__ moments, int t_len, long long n,
                                                          float gamma, float lam) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  double s1 = 0.0, s2 = 0.0;
  if (e < n) {
    float next_v = last_values[e];
    float a = 0.0f;
    int t = t_len - 1;
    for (; t - (UNROLL - 1) >= 0; t -= UNROLL) {
      float r[UNROLL], v[UNROLL], d[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {  // independent loads first: UNROLL requests in flight
        const long long i = (long long)(t - u) * n + e;
        r[u] = __ldg(rewards + i);
        v[u] = __ldg(values + i);
        d[u] = (float)__ldg(dones + i);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        const long long i = (long long)(t - u) * n + e;
        const float g = __fmul_rn(__fsub_rn(1.0f, d[u]), gamma);
        const float delta = __fsub_rn(__fadd_rn(r[u], __fmul_rn(g, next_v)), v[u]);
        a = __fadd_rn(delta, __fmul_rn(__fmul_rn(g, lam), a));
        const float ret = __fadd_rn(a, v[u]);
        returns[i] = ret;
        const float ad = __fsub_rn(ret, v[u]);
        adv[i] = ad;
        s1 += (double)ad;
        s2 += (double)ad * (double)ad;
        next_v = v[u];
      }
    }
    for (; t >= 0; --t) {
      const long long i = (long long)t * n + e;
      const float rr = __ldg(rewards + i), vv = __ldg(values + i), dd = (float)__ldg(dones + i);
      const float g = __fmul_rn(__fsub_rn(1.0f, dd), gamma);
      const float delta = __fsub_rn(__fadd_rn(rr, __fmul_rn(g, next_v)), vv);
      a = __fadd_rn(delta, __fmul_rn(__fmul_rn(g, lam), a));
      const float ret = __fadd_rn(a, vv);
      returns[i] = ret;
      const float ad = __fsub_rn(ret, vv);
      adv[i] = ad;
      s1 += (double)ad;
      s2 += (double)ad * (double)ad;
      next_v = vv;
    }
  }
  // block reduction of the two moments: shuffle inside warps, shared memory across warps
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  __shared__ double w1[8], w2[8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { w1[wid] = s1; w2[wid] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a1 = 0.0, a2 = 0.0;
    for (int w = 0; w < 8; ++w) { a1 += w1[w]; a2 += w2[w]; }
    atomicAdd(moments + 0, a1);
    atomicAdd(moments + 1, a2);
    if (blockIdx.x == 0) atomicAdd(moments + 2, (double)t_len * (double)n);
  }
}

extern "C" int hl_gae_scan(const float* rewards, const float* values, const uint8_t* dones, const float* last_values,
                           float* returns, float* advantages, double* moments, int32_t t_len, int64_t n, float gamma,
                           float lam, void* stream) {
  HL_CHECK_ARG(rewards && values && dones && last_values && returns && advantages && moments, "null pointer");
  HL_CHECK_ARG(t_len >= 0 && n >= 0, "negative size");
  if (n == 0 || t_len == 0) return HL_OK;
  const unsigned blocks = (unsigned)((n + 255) / 256);
  hl_gae_scan_kernel<8><<<blocks, 256, 0, (cudaStream_t)stream>>>(rewards, values, dones, last_values, returns, advantages,
                                                                moments, t_len, n, gamma, lam);
  HL_CHECK_LAUNCH();
  return HL_OK;
}

// advantages = (adv - mean) / (std + 1e-8), std unbiased (torch default) -- :126-127.  The clamp only removes a
// negative rounding residue: with one element the variance is 0/0 = NaN, as torch's std() of one element, and stays so.
__global__ void __launch_bounds__(256) hl_adv_normalize_kernel(float* __restrict__ adv, const double* __restrict__ moments,
                                                               long long n) {
  const double cnt = moments[2];
  const double mean = moments[0] / cnt;
  double var = (moments[1] - moments[0] * mean) / (cnt - 1.0);
  if (cnt > 1.0) var = var > 0.0 ? var : 0.0;
  const float meanf = (float)mean;
  const float denom = (float)sqrt(var) + 1e-8f;
  const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 + 3 < n && (((uintptr_t)adv & 15) == 0)) {
    float4 v = *reinterpret_cast<float4*>(adv + i4);
    v.x = (v.x - meanf) / denom;
    v.y = (v.y - meanf) / denom;
    v.z = (v.z - meanf) / denom;
    v.w = (v.w - meanf) / denom;
    *reinterpret_cast<float4*>(adv + i4) = v;
  } else {
    for (long long i = i4; i < n && i < i4 + 4; ++i) adv[i] = (adv[i] - meanf) / denom;
  }
}

extern "C" int hl_adv_normalize(float* advantages, const double* moments, int64_t n_elems, void* stream) {
  HL_CHECK_ARG(advantages && moments, "null pointer");
  if (n_elems <= 0) return HL_OK;
  const long long threads = (n_elems + 3) / 4;
  hl_adv_normalize_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(advantages, moments, n_elems);
  HL_CHECK_LAUNCH();
  return HL_OK;
}


// ============================================================================= record transition
// Fused runner patch + process_env_step + add_transitions (see include/himloco_b200.h).  Pure
// data movement: CTA = REC_TILE consecutive envs; every per-env tensor's rows of the tile are one
// contiguous slab (128-bit copies, all loads of a thread issued before its stores); the
// next-critic rows are copied per warp so a reset env can take its row from the terminal table
// (row index = rank of the env id in the ascending id list, found by binary search).
constexpr int REC_TILE = 32, REC_THREADS = 256;

__device__ __forceinline__ void rec_copy_slab(float* __restrict__ dst, const float* __restrict__ src, long long off, int count,
                                              int tid) {
  if (!dst || !src) return;
  dst += off;
  src += off;
  if ((((uintptr_t)dst | (uintptr_t)src) & 15) == 0) {
    const int n4 = count >> 2;
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    int i = tid;
    for (; i + 3 * REC_THREADS < n4; i += 4 * REC_THREADS) {  // 4 x 16 B in flight per thread
      const float4 a = __ldcs(s4 + i), b = __ldcs(s4 + i + REC_THREADS), c = __ldcs(s4 + i + 2 * REC_THREADS),
                   d = __ldcs(s4 + i + 3 * REC_THREADS);
      __stcs(d4 + i, a);
      __stcs(d4 + i + REC_THREADS, b);
      __stcs(d4 + i + 2 * REC_THREADS, c);
      __stcs(d4 + i + 3 * REC_THREADS, d);
    }
    for (; i < n4; i += REC_THREADS) __stcs(d4 + i, __ldcs(s4 + i));
    for (int k = (n4 << 2) + tid; k < count; k += REC_THREADS) dst[k] = src[k];
  } else {
    for (int k = tid; k < count; k += REC_THREADS) dst[k] = src[k];
  }
}

__global__ void __launch_bounds__(REC_THREADS) hl_record_transition_kernel(HlTransition t, long long n) {
  hl_pdl_enter();
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const long long e0 = (long long)blockIdx.x * REC_TILE;
  const int cnt = (int)((n - e0) < REC_TILE ? (n - e0) : REC_TILE);
  // per-env scalars first (their loads overlap the slab copies)
  if (tid < cnt) {
    const long long e = e0 + tid;
    if (t.rewards && t.rewards_out) {
      float r = t.rewards[e];
      if (t.time_outs) r = __fadd_rn(r, __fmul_rn(t.gamma, __fmul_rn(t.values[e], t.time_outs[e] ? 1.0f : 0.0f)));
      t.rewards_out[e] = r;
    }
    if (t.dones && t.dones_out) t.dones_out[e] = t.dones[e] ? 1 : 0;
    if (t.values && t.values_out) t.values_out[e] = t.values[e];
    if (t.log_prob && t.log_prob_out) t.log_prob_out[e] = t.log_prob[e];
  }
  rec_copy_slab(t.obs_out, t.obs, e0 * t.obs_dim, cnt * t.obs_dim, tid);
  rec_copy_slab(t.critic_out, t.critic_obs, e0 * t.priv_dim, cnt * t.priv_dim, tid);
  rec_copy_slab(t.actions_out, t.actions, e0 * t.act_dim, cnt * t.act_dim, tid);
  rec_copy_slab(t.mu_out, t.mu, e0 * t.act_dim, cnt * t.act_dim, tid);
  rec_copy_slab(t.sigma_out, t.sigma, e0 * t.act_dim, cnt * t.act_dim, tid);
  if (t.next_critic_obs && t.next_critic_out) {
    if (!t.term_ids) {
      rec_copy_slab(t.next_critic_out, t.next_critic_obs, e0 * t.priv_dim, cnt * t.priv_dim, tid);
    } else {
      const int n_term = *t.n_term_dev;
      const int PD = t.priv_dim;
      for (int r = wid; r < cnt; r += REC_THREADS / 32) {
        const long long e = e0 + r;
        // lower_bound(term_ids, e): warp-uniform binary search
        int lo = 0, hi = n_term;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (t.term_ids[mid] < e) lo = mid + 1;
          else hi = mid;
        }
        const bool hit = lo < n_term && t.term_ids[lo] == e;
        const float* src = hit ? t.term_rows + (long long)lo * PD : t.next_critic_obs + e * PD;
        float* dst = t.next_critic_out + e * PD;
        if (((PD & 1) == 0) && ((((uintptr_t)src | (uintptr_t)dst) & 7) == 0)) {
          const float2* s2 = reinterpret_cast<const float2*>(src);
          float2* d2 = reinterpret_cast<float2*>(dst);
          const int n2 = PD >> 1;
          float2 v[4];
          for (int i0 = 0; i0 < n2; i0 += 128) {
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = (i0 + u * 32 + lane < n2) ? __ldcs(s2 + i0 + u * 32 + lane) : make_float2(0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 4; ++u) if (i0 + u * 32 + lane < n2) __stcs(d2 + i0 + u * 32 + lane, v[u]);
          }
        } else {
          for (int i = lane; i < PD; i += 32) dst[i] = src[i];
        }
      }
    }
  }
}

extern "C" int hl_sizeof_transition(void) { return (int)sizeof(HlTransition); }
extern "C" int hl_record_transition(const HlTransition* t, int64_t n, void* stream) {
  HL_CHECK_ARG(t && t->struct_bytes == (int)sizeof(HlTransition), "HlTransition size mismatch (ABI)");
  HL_CHECK_ARG(t->obs_dim > 0 && t->priv_dim > 0 && t->act_dim > 0, "bad dims");
  HL_CHECK_ARG(!t->term_ids || (t->n_term_dev && t->term_rows), "term_ids needs n_term_dev and term_rows");
  HL_CHECK_ARG(!t->time_outs || t->values, "the time-out bootstrap needs values");
  if (n <= 0) return HL_OK;
  hl_launch(hl_record_transition_kernel, dim3((unsigned)((n + REC_TILE - 1) / REC_TILE)), dim3(REC_THREADS), 0, (cudaStream_t)stream, *t,
            (long long)n);
  HL_CHECK_LAUNCH();
  return HL_OK;
}


// ============================================================================= minibatch gather
// CTA = 32 minibatch rows, 8 warps x 4 rows.  A warp copies its rows field by field (64-bit
// accesses when the row width is even: 270/238/12-float rows are 8-B aligned), all loads of a
// row's field in flight before its stores; width-1 fields are copied by warp 0, one lane per row
// (coalesced stores).
constexpr int GA_ROWS = 32, GA_THREADS = 256;

__global__ void __launch_bounds__(GA_THREADS) hl_minibatch_gather_kernel(HlGatherFields f, const long long* __restrict__ indices,
                                                                        long long n_rows, long long n_src) {
  hl_pdl_enter();
  __shared__ long long s_idx[GA_ROWS];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const long long r0 = (long long)blockIdx.x * GA_ROWS;
  if (tid < GA_ROWS) {
    long long ix = -1;
    if (r0 + tid < n_rows) {
      ix = indices[r0 + tid];
      if (ix < 0 || ix >= n_src) ix = -1;
    }
    s_idx[tid] = ix;
  }
  __syncthreads();
  for (int k = 0; k < f.n_fields; ++k) {
    const int w = f.width[k];
    const float* __restrict__ src = f.src[k];
    float* __restrict__ dst = f.dst[k];
    if (w == 1) {
      if (wid == 0) {
        const long long ix = s_idx[lane];
        if (ix >= 0) dst[r0 + lane] = __ldg(src + ix);
      }
      continue;
    }
    const bool v2 = ((w & 1) == 0) && ((((uintptr_t)src | (uintptr_t)dst) & 7) == 0);
    for (int q = 0; q < GA_ROWS / 8; ++q) {
      const int r = wid * (GA_ROWS / 8) + q;
      const long long ix = s_idx[r];
      if (ix < 0) continue;
      const float* srow = src + ix * w;
      float* drow = dst + (r0 + r) * w;
      if (v2) {
        const float2* s2 = reinterpret_cast<const float2*>(srow);
        float2* d2 = reinterpret_cast<float2*>(drow);
        const int n2 = w >> 1;
        for (int i0 = 0; i0 < n2; i0 += 160) {
          float2 v[5];
#pragma unroll
          for (int u = 0; u < 5; ++u) v[u] = (i0 + u * 32 + lane < n2) ? __ldg(s2 + i0 + u * 32 + lane) : make_float2(0.f, 0.f);
#pragma unroll
          for (int u = 0; u < 5; ++u)
            if (i0 + u * 32 + lane < n2) __stcs(d2 + i0 + u * 32 + lane, v[u]);
        }
      } else {
        for (int i = lane; i < w; i += 32) drow[i] = __ldg(srow + i);
      }
    }
  }
}

extern "C" int hl_sizeof_gather_fields(void) { return (int)sizeof(HlGatherFields); }
extern "C" int hl_minibatch_gather(const HlGatherFields* f, const int64_t* indices, int64_t n_rows, int64_t n_src_rows,
                                   void* stream) {
  HL_CHECK_ARG(f && f->struct_bytes == (int)sizeof(HlGatherFields), "HlGatherFields size mismatch (ABI)");
  HL_CHECK_ARG(f->n_fields > 0 && f->n_fields <= HL_MAX_GATHER_FIELDS, "bad field count");
  HL_CHECK_ARG(indices, "null indices");
  for (int k = 0; k < f->n_fields; ++k) HL_CHECK_ARG(f->src[k] && f->dst[k] && f->width[k] > 0, "null field / bad width");
  if (n_rows <= 0) return HL_OK;
  hl_launch(hl_minibatch_gather_kernel, dim3((unsigned)((n_rows + GA_ROWS - 1) / GA_ROWS)), dim3(GA_THREADS), 0, (cudaStream_t)stream,
            *f, (const long long*)indices, (long long)n_rows, (long long)n_src_rows);
  HL_CHECK_LAUNCH();
  return HL_OK;
}


// ============================================================================= replay ring insert
__global__ void __launch_bounds__(256) hl_ring_insert_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                             float* __restrict__ ra, float* __restrict__ rb, long long n_rows,
                                                             int width, long long size, long long step) {
  hl_pdl_enter();
  const long long total = n_rows * width;
  const long long first = n_rows > size ? n_rows - size : 0;   // earlier rows would be overwritten
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / width;
    if (r < first) continue;
    const long long d = ((step + r) % size) * width + (i - r * width);
    ra[d] = a[i];
    rb[d] = b[i];
  }
}

extern "C" int hl_ring_insert(const float* states, const float* next_states, float* ring_states, float* ring_next,
                              int64_t n_rows, int32_t width, int64_t buffer_rows, int64_t step, void* stream) {
  HL_CHECK_ARG(states && next_states && ring_states && ring_next, "null pointer");
  HL_CHECK_ARG(width > 0 && buffer_rows > 0 && step >= 0 && step < buffer_rows, "bad ring geometry");
  if (n_rows <= 0) return HL_OK;
  const long long total = (long long)n_rows * width;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  hl_launch(hl_ring_insert_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, states, next_states, ring_states,
            ring_next, (long long)n_rows, (int)width, (long long)buffer_rows, (long long)step);
  HL_CHECK_LAUNCH();
  return HL_OK;
}


// ============================================================================= episode statistics
// The runner's rewbuffer / lenbuffer bookkeeping of one env-step (see include/himloco_b200.h), one thread per env.  A
// done env's entry is the j-th of the step (j = rank of its id in the ascending ids, binary search only where dones is
// set) and goes to ring slot (total + j) mod ring_size; only the last ring_size ranks of a step write, so no two writes
// of a step share a slot.  cursor = {total, CTA ticket}: every CTA reads total after griddepcontrol.wait; the CTA that
// takes the last ticket adds the step's count and re-arms the ticket, so the launch is graph-safe.
constexpr int EPS_THREADS = 256;
__global__ void __launch_bounds__(EPS_THREADS) hl_episode_stats_kernel(
    const float* __restrict__ rewards, const unsigned char* __restrict__ dones, const long long* __restrict__ ids,
    const int* __restrict__ n_ids, float* __restrict__ cur_r, float* __restrict__ cur_l, float* __restrict__ ring_r,
    float* __restrict__ ring_l, long long ring_size, long long* __restrict__ cursor, long long n) {
  __shared__ long long s_total;
  hl_pdl_enter();
  const int tid = threadIdx.x;
  if (tid == 0) s_total = cursor[0];
  __syncthreads();
  const long long e = (long long)blockIdx.x * EPS_THREADS + tid;
  if (e < n) {
    float r = __fadd_rn(cur_r[e], rewards[e]);       // cur_reward_sum += rewards
    float l = __fadd_rn(cur_l[e], 1.0f);             // cur_episode_length += 1
    if (dones[e]) {
      const int m = *n_ids;
      int lo = 0, hi = m;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (ids[mid] < e) lo = mid + 1; else hi = mid;
      }
      if (lo < m && ids[lo] == e && (long long)lo >= (long long)m - ring_size) {
        const long long slot = (s_total + lo) % ring_size;
        ring_r[slot] = r;
        ring_l[slot] = l;
      }
      r = 0.0f;
      l = 0.0f;
    }
    cur_r[e] = r;
    cur_l[e] = l;
  }
  if (tid == 0) {
    __threadfence();
    unsigned long long* ticket = reinterpret_cast<unsigned long long*>(cursor + 1);
    if (atomicAdd(ticket, 1ull) == (unsigned long long)gridDim.x - 1ull) {   // every other CTA has read total
      cursor[0] = s_total + *n_ids;
      *ticket = 0ull;
    }
  }
}

extern "C" int hl_episode_stats(const float* rewards, const uint8_t* dones, const int64_t* ids, const int32_t* n_ids_dev,
                                float* cur_reward_sum, float* cur_episode_length, float* ring_reward, float* ring_length,
                                int64_t ring_size, int64_t* cursor, int64_t n_envs, void* stream) {
  HL_CHECK_ARG(rewards && dones && ids && n_ids_dev, "null input");
  HL_CHECK_ARG(cur_reward_sum && cur_episode_length, "null running sums");
  HL_CHECK_ARG(ring_reward && ring_length && cursor, "null ring or cursor");
  HL_CHECK_ARG(ring_size >= 1, "ring_size must be at least 1");
  HL_CHECK_ARG(n_envs >= 1, "n_envs must be at least 1");
  const unsigned blocks = (unsigned)((n_envs + EPS_THREADS - 1) / EPS_THREADS);
  hl_launch(hl_episode_stats_kernel, dim3(blocks), dim3(EPS_THREADS), 0, (cudaStream_t)stream, rewards,
            (const unsigned char*)dones, (const long long*)ids, n_ids_dev, cur_reward_sum, cur_episode_length, ring_reward,
            ring_length, (long long)ring_size, (long long*)cursor, (long long)n_envs);
  HL_CHECK_LAUNCH();
  return HL_OK;
}
