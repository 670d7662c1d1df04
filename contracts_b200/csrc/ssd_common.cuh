// ssd_common.cuh — shared definitions for the sm_100a simulator kernels.
//
// Draw addressing (must match oracle/philox.py, which is what the reference is injected with):
//   u32 = philox4x32_10(ctr = (idx >> 2, site | call << 8, t, episode), key = (seed, env_id))[idx & 3]
// Site ids follow SURVEY.md §8a table R (reference file:line in oracle/philox.py).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#define SSD_MAXN 8            // agents per env ('1'..'9' colour ids exist, shipped configs use <= 8)
#define SSD_VIEW 7            // CLEANUP_VIEW_SIZE / HARVEST_VIEW_SIZE (cleanup_new.py:51, harvest_new.py:36)
#define SSD_OBSW 15
#define SSD_OBS_PIX (SSD_OBSW * SSD_OBSW)          // 225 pixels / agent
#define SSD_OBS_BYTES (SSD_OBS_PIX * 3)            // 675 B / agent

// env_kind / contract_kind constants come from the public header
#include "../../include/ssd_b200.h"

// orientation ints: Agent.py:18-23
enum { ORI_UP = 0, ORI_RIGHT = 1, ORI_DOWN = 2, ORI_LEFT = 3 };

// A tile byte is (palette index << 2) | occupancy bit 7: the byte is directly the byte offset of the
// cell's colour in the 16-entry palette (no shift in the observation gather).  Palette indices:
// cell codes 0..5, 6 + i = agent i painted for the observation, 15 = outside the map.
enum { C_EMPTY = 0 << 2, C_WALL = 1 << 2, C_APPLE = 2 << 2, C_WASTE = 3 << 2, C_RIVER = 4 << 2, C_STREAM = 5 << 2,
       C_OUTSIDE = 15 << 2 };
#define CODE_MASK 0x7Cu
#define CODE_MASK4 0x7C7C7C7Cu
#define TILE_FILL4 0x3C3C3C3Cu        // C_OUTSIDE in every byte
#define PAINT_CODE(i) ((6 + (i)) << 2)
#define OCC_BIT 0x80u

enum { SITE_MOVE_ORDER = 1, SITE_BEAM_ORDER = 2, SITE_SPAWN_DRAWS = 3, SITE_WASTE_ORDER = 4, SITE_SPAWN_ROT = 5,
       SITE_SPAWN_POINT = 6, SITE_CONTRACT = 7, SITE_NEGOTIATE = 8, SITE_SELFDRIVE_RESET = 9,
       SITE_FEAT_ORDER = 10, SITE_FEAT_ROT = 11, SITE_FEAT_SPAWN = 12, SITE_ACTIONS = 13, SITE_SOLVER = 14 };

// record flags
#define RF_STALE_EMPTY 1u     // cleanup: current_apple_points is [] until the first step (cleanup_new.py:181 runs before the reset-time spawn)
#define RF_ERR_SHIFT 8

// ssd_set_episode_log: the ring buffer a reset appends the episode it replaces to (records == nullptr: off).  Part of
// GridParams / FeatParams / CarParams, a runtime pointer like GridParams::stats.  A record (ssd_episode_record) is EPREC_VECS
// 16-byte vectors: 0 = {env_id, episode, t, ended}, 1 = {theta, 0}, 2 + j = {metrics[2 j], metrics[2 j + 1]}.
#define EPREC_VECS 30
struct EpisodeLog {
    uint4* records;                  // [capacity][EPREC_VECS]
    unsigned long long* count;       // records appended so far; record k goes to slot k % capacity
    unsigned long long capacity;
};
__device__ __forceinline__ uint4 eprec_head(uint32_t env_id, uint32_t episode, int t, bool ended)
{
    return make_uint4(env_id, episode, (uint32_t)t, ended ? 1u : 0u);
}
__device__ __forceinline__ uint4 eprec_pair(double lo, double hi)
{
    return make_uint4((uint32_t)__double2loint(lo), (uint32_t)__double2hiint(lo), (uint32_t)__double2loint(hi), (uint32_t)__double2hiint(hi));
}

struct Philox4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int i = 0; i < 10; i++) {
#ifdef __CUDA_ARCH__
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
#else
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
#endif
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    Philox4 r = { c0, c1, c2, c3 };
    return r;
}

// one Philox block of a (site, call) at (t, episode) for env key (seed, env_id)
__device__ __forceinline__ Philox4 draw_block(uint32_t seed, uint32_t env_id, uint32_t episode, uint32_t t,
                                              uint32_t site, uint32_t call, uint32_t block)
{
    return philox4x32_10(block, site | (call << 8), t, episode, seed, env_id);
}
__device__ __forceinline__ uint32_t pick(const Philox4& p, uint32_t w)
{
    return w == 0 ? p.x : (w == 1 ? p.y : (w == 2 ? p.z : p.w));
}
__device__ __forceinline__ uint32_t draw_u32(uint32_t seed, uint32_t env_id, uint32_t episode, uint32_t t,
                                             uint32_t site, uint32_t call, uint32_t idx)
{
    return pick(draw_block(seed, env_id, episode, t, site, call, idx >> 2), idx & 3);
}

// Agreement stage of SeparateContractNegotiateStage.step (two_stage_train.py:266-281) for one env: the acceptance
// probabilities of 2 sampled agents of 1..n-1 (all of them when n <= 3) are multiplied and one uniform draw decides.
// accept: the env's row double [n] (each agent's action[-1]).  Draws are addressed by the env's CURRENT episode at t = 0.
__device__ __forceinline__ bool negotiate_agreement(uint32_t seed, uint32_t env_id, uint32_t episode, int n, const double* accept)
{
    double prod = 1.0;
    if (n > 3) {
        // random.sample(range(1, n), 2): first two of the stateless shuffle of [1..n-1] (keys = draws 0..n-2 of call 0:
        // one Philox block, two when n - 1 > 4)
        const Philox4 b0 = draw_block(seed, env_id, episode, 0, SITE_NEGOTIATE, 0, 0);
        Philox4 b1 = b0;
        if (n - 1 > 4) b1 = draw_block(seed, env_id, episode, 0, SITE_NEGOTIATE, 0, 1);
        uint32_t k1 = 0, k2 = 0; int i1 = -1, i2 = -1;
        for (int j = 0; j < n - 1; j++) {
            const uint32_t k = pick(j < 4 ? b0 : b1, (uint32_t)j & 3u);
            if (i1 < 0 || k < k1) { k2 = k1; i2 = i1; k1 = k; i1 = j; }
            else if (i2 < 0 || k < k2) { k2 = k; i2 = j; }
        }
        prod = __dmul_rn(prod, accept[1 + i1]);
        prod = __dmul_rn(prod, accept[1 + i2]);
    } else {
        for (int i = 1; i < n; i++) prod = __dmul_rn(prod, accept[i]);
    }
    const double r = __dmul_rn((double)draw_u32(seed, env_id, episode, 0, SITE_NEGOTIATE, 1, 0), 1.0 / 4294967296.0);
    return r < prod;
}

// element types of the policy's input tensors (SSD_POLICY_*: ssd_policy_inputs, ssd_set_policy_output,
// ssd_set_flat_policy_output); an observation form 1 + SSD_POLICY_* writes T = PolicyElem<form>::T
template <int FORM> struct PolicyElem;
template <> struct PolicyElem<1 + SSD_POLICY_F32> { typedef float T; };
template <> struct PolicyElem<1 + SSD_POLICY_F16> { typedef __half T; };
template <> struct PolicyElem<1 + SSD_POLICY_BF16> { typedef __nv_bfloat16 T; };

template <typename T> __device__ __forceinline__ T policy_cast(float v);
template <> __device__ __forceinline__ float policy_cast<float>(float v) { return v; }
template <> __device__ __forceinline__ __half policy_cast<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 policy_cast<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// Observation form of the feature-env and selfdrive kernels: OBS_F64 = the float64 rows [E][n][F | D]; 1 + SSD_POLICY_* =
// the policy's flat rows T [E n][W] (ssd_set_flat_policy_output): features ++ [theta, 0] with a contract (W = F + 2), else
// the features alone (W = F), each value T(float32(x)).
#define OBS_F64 0

// the rows of a policy output that carry theta: (theta, 0) `reps` times from column `col` of each of an env's n rows,
// T [E n][width], T by dtype = SSD_POLICY_*; rows == nullptr: none.  A grid world's contract rows are {contract, dtype,
// 10, 0, 5}, flat rows under a contract {rows, dtype, W, W - 2, 1}.
struct ThetaRows { void* rows; int dtype, width, col, reps; };
template <typename T>
__device__ __forceinline__ void theta_rows_fill(T* rows, const ThetaRows& r, int n, double theta)
{
    const T v = policy_cast<T>(__double2float_rn(theta)), z = policy_cast<T>(0.0f);
    for (int a = 0; a < n; a++)
        for (int k = 0; k < r.reps; k++) {
            rows[(size_t)a * r.width + r.col + 2 * k] = v;
            rows[(size_t)a * r.width + r.col + 2 * k + 1] = z;
        }
}
// what the calls that change theta outside a step do to the policy output (thread-per-env kernels)
__device__ __forceinline__ void theta_rows_env(const ThetaRows& r, int n, int env, double theta)
{
    if (!r.rows) return;
    const size_t o = (size_t)env * n * r.width;
    if (r.dtype == SSD_POLICY_F32) theta_rows_fill(reinterpret_cast<float*>(r.rows) + o, r, n, theta);
    else if (r.dtype == SSD_POLICY_F16) theta_rows_fill(reinterpret_cast<__half*>(r.rows) + o, r, n, theta);
    else theta_rows_fill(reinterpret_cast<__nv_bfloat16*>(r.rows) + o, r, n, theta);
}

// SSD_STEP_AUTO (ssd_random_actions & co.): counter[0] = step index, counter[1] = CTAs finished.  Every CTA reads
// counter[0] before it arrives at counter[1]; the last one to arrive bumps the index for the next launch, so a captured
// CUDA graph draws fresh actions at every replay without a separate one-thread kernel.
__device__ __forceinline__ void counter_finish(uint32_t* counter, uint32_t step_index)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(counter + 1, 1u) == gridDim.x - 1) { counter[1] = 0u; counter[0] = step_index + 1u; }
    }
}
