// ssd_solver.cuh — the NegotiationSolver prologue of a vectorised sampler (ssd_solver_rows / ssd_solver_resolve).
//
// In the reference every env is its own NegotiationSolver (environments/two_stage_train.py:619-776): every reset samples
// 1 + S candidate contracts, queries the frozen policy's value function for each and installs the winner.  In a batch
// whose envs are each at their own point of an episode only the envs that were just reset need that, so the solver works
// on a queue of them:
//   pending   an env is at the start of an episode (initialised, t == 0) whose contract the solver has not chosen yet
//             (resolved[env] != its episode counter).  Nothing else marks it: every reset path already writes t and the
//             episode counter, so no step or reset kernel is involved.
//   window    the first C pending envs in env order: solver_count_kernel counts the pending envs of each block of
//             SQ_BLOCK envs, solver_scatter_kernel ranks them (the counts of the blocks before it + a block scan) and
//             stores the window.  Two launches, no host synchronisation, capturable in a CUDA graph.
//   rows      solver_rows_kernel writes the candidates (solver_candidate, the draw of solver_sample_kernel) and the
//             value-query rows [C][1 + S][n][W] of the window, zeros beyond it.
//   resolve   solver_resolve_kernel applies compute_best_param (solver_choose_env, the body of solver_choose_kernel) to each
//             window entry whose env is still at t == 0 of the same episode, writes theta and the policy output's rows
//             that carry it, and records the episode as resolved.
#pragma once
#include "ssd_views.cuh"

#define SQ_BLOCK 1024                 // envs (= threads) per block of the count / scatter kernels
#define SQ_NONE 0xFFFFFFFFu           // resolved[env]: no episode resolved yet

// where the pending test reads an env's t and initialised bit (every env kind; episode / theta are in SolverParams)
struct SolverQueue {
    SolverParams s;
    const uint8_t* t; long long t_stride;                 // int32
    const uint8_t* init; long long init_stride;           // uint32, bit 31
    uint32_t* resolved;                                   // [E] episode whose contract was chosen, or SQ_NONE
    uint32_t* block_count;                                // [ceil(E / SQ_BLOCK)] pending envs per block
    int C, S;                                             // window capacity, samples per env
    int32_t* env; uint32_t* episode; uint32_t* count;     // the window: [C], [C], {in window, pending in total}
    double* params;                                       // [C][1 + S]
};

__device__ __forceinline__ uint32_t sq_episode(const SolverQueue& q, int env)
{
    return *reinterpret_cast<const uint32_t*>(q.s.episode + (size_t)env * q.s.episode_stride) & q.s.episode_mask;
}
__device__ __forceinline__ bool sq_at_start(const SolverQueue& q, int env)
{
    return (*reinterpret_cast<const uint32_t*>(q.init + (size_t)env * q.init_stride) & 0x80000000u)
        && *reinterpret_cast<const int32_t*>(q.t + (size_t)env * q.t_stride) == 0;
}
__device__ __forceinline__ bool sq_pending(const SolverQueue& q, int env)
{
    return sq_at_start(q, env) && q.resolved[env] != sq_episode(q, env);
}

__global__ void __launch_bounds__(SQ_BLOCK) solver_count_kernel(const SolverQueue q)
{
    const int env = blockIdx.x * SQ_BLOCK + threadIdx.x;
    const int c = __syncthreads_count(env < q.s.E && sq_pending(q, env));
    if (threadIdx.x == 0) q.block_count[blockIdx.x] = (uint32_t)c;
}

__global__ void __launch_bounds__(SQ_BLOCK) solver_scatter_kernel(const SolverQueue q)
{
    __shared__ uint32_t warp_sum[SQ_BLOCK / 32];
    __shared__ uint32_t base_s, total_s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // pending envs of the blocks before this one (and, for block 0, of all blocks)
    const int nb = (q.s.E + SQ_BLOCK - 1) / SQ_BLOCK, upto = blockIdx.x == 0 ? nb : (int)blockIdx.x;
    uint32_t part = 0u;
    for (int b = threadIdx.x; b < upto; b += SQ_BLOCK) part += q.block_count[b];
    part = __reduce_add_sync(0xFFFFFFFFu, part);
    if (lane == 0) warp_sum[warp] = part;
    __syncthreads();
    if (warp == 0) {
        const uint32_t s = __reduce_add_sync(0xFFFFFFFFu, warp_sum[lane]);
        if (lane == 0) { if (blockIdx.x == 0) { total_s = s; base_s = 0u; } else base_s = s; }
    }
    __syncthreads();
    const uint32_t base = base_s;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        q.count[0] = total_s < (uint32_t)q.C ? total_s : (uint32_t)q.C;
        q.count[1] = total_s;
    }
    if (base >= (uint32_t)q.C) return;                     // (uniform) the window is full before this block
    // rank within the block: ballot prefix within the warp, exclusive scan over the warps
    const int env = blockIdx.x * SQ_BLOCK + threadIdx.x;
    const bool pend = env < q.s.E && sq_pending(q, env);
    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, pend);
    __syncthreads();                                       // warp_sum is reused
    if (lane == 0) warp_sum[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
        const uint32_t v = warp_sum[lane];
        uint32_t incl = v;
        for (int d = 1; d < 32; d <<= 1) { const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += u; }
        warp_sum[lane] = incl - v;
    }
    __syncthreads();
    const uint32_t rank = base + warp_sum[warp] + __popc(bal & ((1u << lane) - 1u));
    if (pend && rank < (uint32_t)q.C) {
        q.env[rank] = env;
        q.episode[rank] = sq_episode(q, env);
    }
}

// Row layout of the value queries, by the handle's observation form:
//   SQ_ROWS_CONTRACT  the contract part alone (image forms): (param, 0) `reps` times, T = double (uint8 windows, W = 2) or
//                     the policy dtype (policy image, W = 10, what the contract rows of ssd_set_policy_output hold)
//   SQ_ROWS_FLAT      obs ++ [param, 0], W = F + 2: the F feature columns copied from src (row e n + a, src_width
//                     elements apart), T = double (_obs_with's float64 rows) or the policy dtype (bit copies of the
//                     policy rows' feature columns, then T(float32(param)), 0 like their theta column)
#define SQ_ROWS_CONTRACT 0
#define SQ_ROWS_FLAT 1
template <typename T> __device__ __forceinline__ T sq_value(double v) { return policy_cast<T>(__double2float_rn(v)); }
template <> __device__ __forceinline__ double sq_value<double>(double v) { return v; }

// one thread per (window slot, candidate, agent) row
template <typename T, int LAYOUT>
__global__ void solver_rows_kernel(const SolverQueue q, T* __restrict__ rows, int W, int reps, const T* __restrict__ src, int F,
                                   int src_width)
{
    const int n = q.s.n, S1 = q.S + 1;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)q.C * S1 * n) return;
    const int c = (int)(idx / ((long long)S1 * n));
    const int r = (int)(idx - (long long)c * S1 * n), k = r / n, a = r - k * n;
    const int cnt = (int)q.count[0];
    T* row = rows + (size_t)idx * W;
    const T zero = sq_value<T>(0.0);
    if (c >= cnt) {                                        // beyond the window: zeros, no env
        for (int j = 0; j < W; j++) row[j] = zero;
        if (a == 0) q.params[(size_t)c * S1 + k] = 0.0;
        if (a == 0 && k == 0) { q.env[c] = -1; q.episode[c] = 0u; }
        return;
    }
    const int env = q.env[c];
    const double param = solver_candidate(q.s, env, q.episode[c], k);
    if (a == 0) q.params[(size_t)c * S1 + k] = param;
    const T v = sq_value<T>(param);
    if constexpr (LAYOUT == SQ_ROWS_CONTRACT) {
        for (int j = 0; j < reps; j++) { row[2 * j] = v; row[2 * j + 1] = zero; }
    } else {
        const T* s = src + ((size_t)env * n + a) * src_width;
        for (int j = 0; j < F; j++) row[j] = s[j];
        row[F] = v; row[F + 1] = zero;
    }
}

// host side: the rows kernel of the handle's form, one thread per row
template <typename T>
static void launch_solver_rows(const SolverQueue& q, int layout, void* rows, int W, int reps, const void* src, int F, int src_width,
                               cudaStream_t s)
{
    const long long total = (long long)q.C * (q.S + 1) * q.s.n;
    const unsigned blocks = (unsigned)((total + 255) / 256);
    if (layout == SQ_ROWS_FLAT)
        solver_rows_kernel<T, SQ_ROWS_FLAT><<<blocks, 256, 0, s>>>(q, (T*)rows, W, reps, (const T*)src, F, src_width);
    else
        solver_rows_kernel<T, SQ_ROWS_CONTRACT><<<blocks, 256, 0, s>>>(q, (T*)rows, W, reps, (const T*)src, F, src_width);
}

// one thread per window slot
__global__ void solver_resolve_kernel(const SolverQueue q, int rule, const double* __restrict__ vals, double* __restrict__ best_param,
                                      int* __restrict__ best_idx, uint32_t* __restrict__ stale)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= q.C) return;
    if (c >= (int)q.count[0]) {
        if (best_param) best_param[c] = 0.0;
        if (best_idx) best_idx[c] = -1;
        return;
    }
    const int env = q.env[c];
    if (!sq_at_start(q, env) || sq_episode(q, env) != q.episode[c]) {   // stepped or reset again since the rows call
        if (best_param) best_param[c] = *reinterpret_cast<const double*>(q.s.theta + (size_t)env * q.s.theta_stride);
        if (best_idx) best_idx[c] = -1;
        if (stale) atomicAdd(stale, 1u);
        return;
    }
    solver_choose_env(q.s, q.S, rule, q.params, vals, best_param, best_idx, env, c);
    q.resolved[env] = q.episode[c];
}

// ssd_checkpoint_load: a loaded env's theta came back with it, so its episode counts as resolved (an env that was never
// reset has no episode to resolve).  Rows that failed validation left their env as it was, and its record too.
__global__ void solver_mark_loaded_kernel(const SolverQueue q, const int32_t* env_idx, int count, const uint8_t* row_ok)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= count || !row_ok[r]) return;
    const int env = env_idx ? env_idx[r] : r;
    if (env < 0 || env >= q.s.E) return;
    const bool init = *reinterpret_cast<const uint32_t*>(q.init + (size_t)env * q.init_stride) & 0x80000000u;
    q.resolved[env] = init ? sq_episode(q, env) : SQ_NONE;
}
