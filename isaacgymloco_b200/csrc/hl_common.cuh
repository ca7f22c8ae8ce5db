// Shared device helpers for libhimloco_b200 (sm_100a).  See include/himloco_b200.h for the ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/himloco_b200.h"

// ----------------------------------------------------------------------------- errors
void hl_set_error(const char* fmt, ...);

#define HL_CHECK_ARG(cond, msg)          \
  do {                                   \
    if (!(cond)) {                       \
      hl_set_error("%s: %s", __func__, msg); \
      return HL_E_INVALID;               \
    }                                    \
  } while (0)

#define HL_CHECK_LAUNCH()                                                        \
  do {                                                                           \
    cudaError_t e__ = cudaGetLastError();                                        \
    if (e__ != cudaSuccess) {                                                    \
      hl_set_error("%s: CUDA error: %s", __func__, cudaGetErrorString(e__));     \
      return HL_E_CUDA;                                                          \
    }                                                                            \
  } while (0)

// ----------------------------------------------------------------------------- launches
// Programmatic dependent launch (griddepcontrol, sm_90+): the kernels of one env step form a chain
// of short dependent launches (4 x torque, fused, select/terminal, fix-up), so each kernel lets
// its successor be scheduled right away and then waits for its predecessor's memory: launch
// latency and the first wave's ramp-up overlap the predecessor's tail.  Every kernel launched
// through hl_launch() calls hl_pdl_enter() before its first global access and before any return.
// EARLY (griddepcontrol.launch_dependents at entry) lets the successor's CTAs become resident at
// once.  Measured and left off everywhere: parked successor CTAs take registers / warp slots from
// the running kernel (65,536 envs: 3.68 -> 3.78 ms per rollout with it on the short kernels, 4.26 ms
// with it on the fused kernel too; wait-only is 1 % better than no PDL at all).
template <bool EARLY = false>
__device__ __forceinline__ void hl_pdl_enter() {
#ifndef HL_PDL_NO_EARLY
  if (EARLY) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
bool hl_pdl_enabled();  // HL_PDL=0 turns the launch attribute off (A/B runs)

template <typename... KArgs, typename... Args>
static inline void hl_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t lc = {};
  lc.gridDim = grid;
  lc.blockDim = block;
  lc.dynamicSmemBytes = smem;
  lc.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  lc.attrs = at;
  lc.numAttrs = hl_pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&lc, kern, static_cast<KArgs>(args)...);   // errors surface in HL_CHECK_LAUNCH
}

// look-back state of a CTA / tile in the ordered reset-id compaction: epoch << 32 | flag << 30 | value
constexpr unsigned long long HL_LB_AGG = 1ull << 30, HL_LB_PREFIX = 2ull << 30, HL_LB_VALUE = (1ull << 30) - 1ull;

#ifndef HL_TILED_TMA
#define HL_TILED_TMA 0              // 1: compile the cp.async.bulk staging path into the tiled fused kernel (then HL_FUSED_TMA=1 selects it)
#endif
#ifndef HL_PK_WAIT_HINT
#define HL_PK_WAIT_HINT 0           // ns: mbarrier.try_wait suspend-time hint for long waits; 0 = probe + nanosleep
#endif
#ifndef HL_PK_WAIT_NS
#define HL_PK_WAIT_NS 500           // sleep between probes of a long wait (measured: 128 -> 500 ns: -3 us per launch)
#endif
// ----------------------------------------------------------------------------- mbarrier / TMA (sm_90+: cp.async.bulk)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// same for the S warps' long waits: try_wait with a suspend-time hint parks the warp in hardware for up
// to that many ns per probe instead of spinning through issue slots the H warps need
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) {
#if HL_PK_WAIT_HINT
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)), "r"(parity), "r"((unsigned)HL_PK_WAIT_HINT) : "memory");
#else
  for (;;) {
    uint32_t done;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (done) break;
    __nanosleep(HL_PK_WAIT_NS);
  }
#endif
}
// 1-D TMA bulk copy global -> shared; completion is signalled on `bar` as transaction bytes
__device__ __forceinline__ void tma_load(float* dst, const float* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ----------------------------------------------------------------------------- reward term ids
// sorted() order of the 51 unique `_reward_*` names (legged_robot.py:1444-1770); mirrored by
// isaacgymloco_b200/config.py::REWARD_TERMS.
enum HlTerm : int {
  T_action_rate = 0, T_ang_vel_xy, T_ang_vel_xy_up, T_base_height, T_base_height_up, T_calf_pose,
  T_calf_pose_up, T_collision, T_collision_up, T_dof_acc, T_dof_pos_dif, T_dof_pos_limits,
  T_dof_vel, T_dof_vel_limits, T_feet_air_time, T_feet_contact_forces, T_feet_mirror,
  T_feet_mirror_up, T_feet_slide, T_feet_slide_up, T_feet_stumble, T_feet_stumble_up,
  T_foot_clearance_base, T_foot_clearance_base_up, T_foot_clearance_terrain,
  T_foot_clearance_terrain_up, T_has_contact, T_hip_action_magnitude, T_hip_pos, T_hip_pos_up,
  T_joint_power, T_lin_vel_z, T_lin_vel_z_up, T_orientation, T_orientation_up, T_power,
  T_power_distribution, T_smoothness, T_stand_nice, T_stand_still, T_stuck, T_termination,
  T_thigh_pose, T_thigh_pose_up, T_torque_limits, T_torques, T_torques_dif,
  T_torques_distribution, T_tracking_ang_vel, T_tracking_lin_vel, T_upward, T_COUNT
};

// ----------------------------------------------------------------------------- Philox4x32-10
// Counter-based RNG for the throughput-mode observation noise (the reference draws it with
// torch.rand_like, LR:394,400,451,457, whose CUDA generator is the same Philox family; the
// streams are statistically, not bitwise, equivalent -- parity tests pass pre-drawn tensors).
__device__ __forceinline__ uint4 hl_philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}
// Same function with the 10 round keys precomputed (they depend on the seed only).
struct HlPhiloxKeys {
  uint32_t kx[10], ky[10];
  __device__ __forceinline__ void init(uint64_t seed) {
    uint32_t x = (uint32_t)seed, y = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      kx[r] = x;
      ky[r] = y;
      x += 0x9E3779B9u;
      y += 0xBB67AE85u;
    }
  }
};
__device__ __forceinline__ uint4 hl_philox4x32_10(uint4 c, const HlPhiloxKeys& k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.kx[r], lo1, hi0 ^ c.w ^ k.ky[r], lo0);
  }
  return c;
}

__device__ __forceinline__ float hl_u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

// one Philox block = 4 uniforms for (env, block index, stream, step)
__device__ __forceinline__ uint4 hl_noise_block(uint64_t seed, uint64_t offset, uint64_t env,
                                                uint32_t block, uint32_t stream) {
  const uint4 ctr = make_uint4(block | (stream << 24), (uint32_t)env, (uint32_t)(env >> 32) ^ (uint32_t)(offset >> 32),
                               (uint32_t)offset);
  return hl_philox4x32_10(ctr, make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}

__device__ __forceinline__ uint4 hl_noise_block(const HlPhiloxKeys& keys, uint64_t offset, uint64_t env, uint32_t block,
                                                uint32_t stream) {
  const uint4 ctr = make_uint4(block | (stream << 24), (uint32_t)env, (uint32_t)(env >> 32) ^ (uint32_t)(offset >> 32),
                               (uint32_t)offset);
  return hl_philox4x32_10(ctr, keys);
}

// The step index that keys every Philox stream: philox_offset, plus *step_base when the step counter lives on the
// device (a replayed CUDA graph, which cannot take a new value by argument).  Read after griddepcontrol.wait: the op
// that advanced the counter may be the predecessor in the stream.
__device__ __forceinline__ unsigned long long hl_step_key(const HlEnvBuffers& b) {
  return b.step_base ? (unsigned long long)(*b.step_base) + b.philox_offset : b.philox_offset;
}
// The same, read once per CTA: thread 0 loads it into `*slot` (shared memory) and the barrier publishes it; every
// thread of the CTA must call.
__device__ __forceinline__ uint64_t hl_step_key_cta(const HlEnvBuffers& b, unsigned long long* slot) {
  if (threadIdx.x == 0) *slot = hl_step_key(b);
  __syncthreads();
  return *slot;
}

__device__ __forceinline__ unsigned hl_pick(const uint4& q, int cpt) { return cpt == 0 ? q.x : (cpt == 1 ? q.y : (cpt == 2 ? q.z : q.w)); }

// Canonical mapping of one env's observation noise onto Philox blocks (stream 0 = observation,
// 1 = terminal observation), shared by every kernel:
//   height point p = 32*it + lane    -> component it&3 of block (it>>2)*32 + lane
//   one-step obs element k = lane    -> component c0   of block cb*32 + lane
//   one-step obs element k = lane+32 -> component c0+1 of block cb*32 + lane
// where the last height pass leaves two spare components when ceil(P/32) mod 4 is 1 or 2 (aliengo:
// P = 187 -> 6 iterations -> cb = 1, c0 = 2); otherwise a further block is drawn.
__device__ __forceinline__ void hl_cur_noise_slot(int P, int& cb, int& c0) {
  const int nit = (P + 31) >> 5, rem = nit & 3;
  if (rem == 1 || rem == 2) { cb = (nit - 1) >> 2; c0 = 2; }
  else { cb = (nit + 3) >> 2; c0 = 0; }
}

__device__ __forceinline__ float hl_clampf(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }

// torch `%` on floats (Python sign): fmod then fix-up.
__device__ __forceinline__ float hl_pymod(float a, float b) {
  float r = fmodf(a, b);
  if (r != 0.0f && ((r < 0.0f) != (b < 0.0f))) r += b;
  return r;
}
