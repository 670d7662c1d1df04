// ssd_views.cuh — the JointEnv output layouts (environments/two_stage_train.py:476-617), written from device state:
//
//   global_view_kernel   `global_obs`: MapEnv.global_view() (map_env.py:394-395) = the whole world_map_color with the
//                        agents painted (map_env.py:257-261), uint8 [E][H][W][3]; JointEnv.reset / global_step return
//                        it / 255 (cleanup_new.py:299-300, harvest_new.py:178-179)
//   concat_obs_kernel    `concatenated_obs`: np.concatenate of the agents' windows along the channel axis
//                        (two_stage_train.py:527-533,604-609): uint8 [E][n][15][15][3] -> [E][15][15][3 n]
//
// Both are pure byte streams bound by HBM (global view: map_bytes read + 3 H W written per env; concat: 675 n
// read + written per env).  A CTA owns VIEW_GROUP = 4 consecutive envs, so its output range is a whole number of
// 32-bit words whatever the per-env byte count is, stages the inputs in shared memory with 16-byte loads and
// writes aligned words.
#pragma once
#include "ssd_grid.cuh"

#define VIEW_THREADS 128
#define VIEW_GROUP 4

// full_map: 0 = global_view (agents from the first step on, no beams); 1 = MapEnv.full_map_to_colors (map_env.py:389-392,
// the render() frame): agents always, then the beams of the last step on top (get_map_with_agents :354-375) when the
// handle records them (GridParams::beam; 'F' (255, 255, 0), 'C' (100, 255, 255), DEFAULT_COLOURS map_env.py:40-41)
__global__ void __launch_bounds__(VIEW_THREADS) global_view_kernel(const GridParams p, uint8_t* __restrict__ out, const int full_map)
{
    extern __shared__ __align__(16) uint8_t vsm[];            // VIEW_GROUP compact maps
    __shared__ uint32_t s_pal[16];
    const int env0 = blockIdx.x * VIEW_GROUP;
    const int G = min(VIEW_GROUP, p.E - env0);
    const int nvec = p.map_bytes >> 4;
    if (threadIdx.x < 16) s_pal[threadIdx.x] = p.pal[threadIdx.x];
    for (int i = threadIdx.x; i < G * nvec; i += VIEW_THREADS) {            // the static map ...
        const int g = i / nvec, v = i - g * nvec;
        reinterpret_cast<uint4*>(vsm)[i] = __ldg(reinterpret_cast<const uint4*>(p.base_map) + v);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < G * (p.n_apple + p.n_waste); i += VIEW_THREADS) {   // ... + the dynamic cells from the masks
        const int g = i / (p.n_apple + p.n_waste), j = i - g * (p.n_apple + p.n_waste);
        const uint8_t* hdr = p.state + (size_t)(env0 + g) * p.rec_stride;
        if (j < p.n_apple) {
            if ((reinterpret_cast<const uint32_t*>(hdr + RO_AMASK)[j >> 5] >> (j & 31)) & 1u) vsm[g * p.map_bytes + p.apple_c[j]] = (uint8_t)C_APPLE;
        } else {
            const int k = j - p.n_apple;
            if ((reinterpret_cast<const uint32_t*>(hdr + RO_WMASK)[k >> 5] >> (k & 31)) & 1u) vsm[g * p.map_bytes + p.waste_c[k]] = (uint8_t)C_WASTE;
        }
    }
    __syncthreads();
    if (threadIdx.x < G) {                                    // paint in agent order: the highest index wins a shared cell
        const uint8_t* hdr = p.state + (size_t)(env0 + threadIdx.x) * p.rec_stride;
        const uint32_t* ag = reinterpret_cast<const uint32_t*>(hdr + RO_AGENTS);
        // MapEnv.reset (map_env.py:306-342) never paints the agents into world_map_color: they appear from the first step on
        const int na = (full_map || *reinterpret_cast<const int*>(hdr + RO_T) > 0) ? p.n : 0;
        for (int a = 0; a < na; a++) {
            const uint32_t v = ag[a];
            vsm[threadIdx.x * p.map_bytes + (int)(v & 255u) * p.Wp + (int)((v >> 8) & 255u)] = (uint8_t)PAINT_CODE(a);
        }
    }
    __syncthreads();
    if (full_map && p.beam) {                                 // beams overlay agents: palette slot 14 = 'F', agent 5's colour = 'C'
        for (int i = threadIdx.x; i < G * p.map_bytes; i += VIEW_THREADS) {
            const uint8_t bc = p.beam[(size_t)env0 * p.map_bytes + i];
            if (bc) vsm[i] = bc == 'F' ? (uint8_t)(14 << 2) : (uint8_t)PAINT_CODE(5);
        }
        if (threadIdx.x == 0) s_pal[14] = 255u | (255u << 8);
        __syncthreads();
    }
    const int cells = p.H * p.W, per_env = cells * 3, total = G * per_env;
    uint8_t* stage = vsm + VIEW_GROUP * p.map_bytes;          // the group's output bytes
    const int dq = VIEW_THREADS / p.W, dm = VIEW_THREADS - dq * p.W;       // (row, col) step of a thread's next cell
    const int r0 = (int)threadIdx.x / p.W, c0 = (int)threadIdx.x - r0 * p.W;
    for (int g = 0; g < G; g++) {
        const uint8_t* m = vsm + g * p.map_bytes;
        uint8_t* o = stage + g * per_env + 3 * threadIdx.x;
        int r = r0, c = c0;
        for (int cell = threadIdx.x; cell < cells; cell += VIEW_THREADS, o += 3 * VIEW_THREADS) {
            const uint32_t col = s_pal[(m[r * p.Wp + c] & CODE_MASK) >> 2];
            o[0] = (uint8_t)col; o[1] = (uint8_t)(col >> 8); o[2] = (uint8_t)(col >> 16);
            c += dm; r += dq;
            if (c >= p.W) { c -= p.W; r++; }
        }
    }
    __syncthreads();
    uint8_t* dst = out + (size_t)env0 * per_env;              // env0 % 4 == 0: word aligned
    for (int w = threadIdx.x; 4 * w + 3 < total; w += VIEW_THREADS) reinterpret_cast<uint32_t*>(dst)[w] = reinterpret_cast<const uint32_t*>(stage)[w];
    for (int k = (total & ~3) + threadIdx.x; k < total; k += VIEW_THREADS) dst[k] = stage[k];
}

// MapEnv.reset: self.beam_pos = [] (map_env.py:316) for the envs being reset; one warp per env
__global__ void beam_clear_kernel(const GridParams p, const uint8_t* __restrict__ mask)
{
    const int env = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (env >= p.E || (mask && !mask[env])) return;
    uint4* b = reinterpret_cast<uint4*>(p.beam + (size_t)env * p.map_bytes);
    for (int i = lane; i < (p.map_bytes >> 4); i += 32) b[i] = make_uint4(0u, 0u, 0u, 0u);
}

__global__ void __launch_bounds__(VIEW_THREADS) concat_obs_kernel(const GridParams p, const uint8_t* __restrict__ obs,
                                                                  long long obs_stride, uint8_t* __restrict__ out)
{
    extern __shared__ __align__(16) uint8_t vsm[];            // VIEW_GROUP x n windows
    const int n = p.n, per_env = n * SSD_OBS_BYTES;
    const int env0 = blockIdx.x * VIEW_GROUP;
    const int G = min(VIEW_GROUP, p.E - env0);
    const int total = G * per_env;
    __shared__ uint64_t bar;
    // dense batch tensor and a 16-byte multiple per group (n % 4 == 0): the group moves with one bulk (TMA) copy each way
    const bool bulk = obs_stride == per_env && G == VIEW_GROUP && (total & 15) == 0 &&
                      ((reinterpret_cast<uintptr_t>(obs) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
    if (bulk) {
        if (threadIdx.x == 0) mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) bulk_load(vsm, obs + (size_t)env0 * per_env, (uint32_t)total, &bar);
        mbar_wait(&bar, 0);
    } else if (obs_stride == per_env) {                       // dense: the group is one aligned word run
        const uint32_t* src = reinterpret_cast<const uint32_t*>(obs + (size_t)env0 * per_env);
        for (int w = threadIdx.x; 4 * w + 3 < total; w += VIEW_THREADS) reinterpret_cast<uint32_t*>(vsm)[w] = src[w];
        for (int b = (total & ~3) + threadIdx.x; b < total; b += VIEW_THREADS) vsm[b] = obs[(size_t)env0 * per_env + b];
    } else {
        for (int b = threadIdx.x; b < total; b += VIEW_THREADS) {
            const int g = b / per_env;
            vsm[b] = obs[(size_t)(env0 + g) * obs_stride + (b - g * per_env)];
        }
    }
    __syncthreads();
    uint8_t* stage = vsm + VIEW_GROUP * per_env;              // the group's output bytes
    const int n3 = 3 * n;
    for (int i = threadIdx.x; i < G * SSD_OBS_PIX; i += VIEW_THREADS) {
        const int g = i / SSD_OBS_PIX, pix = i - g * SSD_OBS_PIX;
        const uint8_t* src = vsm + g * per_env + pix * 3;
        uint8_t* o = stage + g * per_env + pix * n3;
        for (int a = 0; a < n; a++) {                         // out[pix][3 a + ch] = in[a][pix][ch]
            o[3 * a] = src[a * SSD_OBS_BYTES]; o[3 * a + 1] = src[a * SSD_OBS_BYTES + 1]; o[3 * a + 2] = src[a * SSD_OBS_BYTES + 2];
        }
    }
    uint8_t* dst = out + (size_t)env0 * per_env;
    if (bulk) {
        fence_async_smem();                                   // the staged bytes become visible to the async proxy
        __syncthreads();
        if (threadIdx.x == 0) { bulk_store(dst, stage, (uint32_t)total); bulk_wait_read<0>(); }
        return;
    }
    __syncthreads();
    for (int w = threadIdx.x; 4 * w + 3 < total; w += VIEW_THREADS) reinterpret_cast<uint32_t*>(dst)[w] = reinterpret_cast<const uint32_t*>(stage)[w];
    for (int k = (total & ~3) + threadIdx.x; k < total; k += VIEW_THREADS) dst[k] = stage[k];
}

// ---------------------------------------------------------------------------------------------
// NegotiationSolver (environments/two_stage_train.py:619-776), batched over envs.  The value-function
// queries (compute_vals :693-703, an RLlib policy forward) stay with the caller; the device side is
//   solver_sample_kernel   negotiate :705-746: candidate 0 is the null contract `contract_space.low`, candidates
//                          1..S are `contract_param_space.sample()` — gym 0.21 Box.sample: float32(uniform(low, high))
//                          evaluated in float64 — drawn from the env's Philox stream (site SOLVER, one draw each);
//   solver_choose_kernel   compute_best_param :748-776 on the caller's values [E][1 + S][n]: rule `max` = first
//                          argmax of the per-candidate welfare sum(vals) (agent order, left to right); rule
//                          `majority` = the same over {null} + candidates that at least half of the agents strictly
//                          prefer to the null contract, a candidate's parameter being looked up through
//                          `all_vals.index(k1)` (the FIRST candidate with identical values).  The winner becomes the
//                          env's contract parameter (reset :675-676).
// Works for every env kind: episode / theta are addressed through (pointer, byte stride, mask).
struct SolverParams {
    int E, n;
    uint32_t seed, first_env_id;
    double low, high;
    const uint8_t* episode; long long episode_stride; uint32_t episode_mask;
    uint8_t* theta; long long theta_stride;
    ThetaRows rows;                          // the policy output's rows that carry theta (rows NULL: none)
};
#define SOLVER_RULE_MAX 0
#define SOLVER_RULE_MAJORITY 1

// candidate k of `env` in its episode `episode` (solver_sample_kernel, solver_rows_kernel)
__device__ __forceinline__ double solver_candidate(const SolverParams& p, int env, uint32_t episode, int k)
{
    double v = p.low;
    if (k > 0) {
        const uint32_t u = draw_u32(p.seed, p.first_env_id + (uint32_t)env, episode, 0u, SITE_SOLVER, 0u, (uint32_t)(k - 1));
        const double x = __dadd_rn(p.low, __dmul_rn(__dsub_rn(p.high, p.low), (double)u * 2.3283064365386963e-10));
        v = (double)(float)x;                                       // .astype(np.float32)
    }
    return v;
}

__global__ void solver_sample_kernel(const SolverParams p, int S, double* __restrict__ params)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;          // one thread per (env, candidate)
    if (idx >= p.E * (S + 1)) return;
    const int env = idx / (S + 1), k = idx - env * (S + 1);
    uint32_t episode = 0u;
    if (k > 0) episode = *reinterpret_cast<const uint32_t*>(p.episode + (size_t)env * p.episode_stride) & p.episode_mask;
    params[idx] = solver_candidate(p, env, episode, k);
}

// compute_best_param for env `env`, whose values / candidates are row `slot` of vals [.][1 + S][n] / params [.][1 + S]: the
// winner becomes the env's theta (and the policy output's rows that carry it follow) and best_param[slot] / best_idx[slot]
// (nullable) receive it and its candidate index (solver_choose_kernel: slot = env; solver_resolve_kernel: the window slot)
__device__ __forceinline__ void solver_choose_env(const SolverParams& p, int S, int rule, const double* __restrict__ params,
                                                  const double* __restrict__ vals, double* __restrict__ best_param,
                                                  int* __restrict__ best_idx, int env, int slot)
{
    const int n = p.n;
    const double* V = vals + (size_t)slot * (S + 1) * n;
    const double* P = params + (size_t)slot * (S + 1);
    int best = 0;                       // the null contract is always a candidate
    double best_w = 0.0;
    for (int a = 0; a < n; a++) best_w = __dadd_rn(best_w, V[a]);
    for (int k = 1; k <= S; k++) {
        const double* vk = V + (size_t)k * n;
        if (rule == SOLVER_RULE_MAJORITY) {
            int accepted = 0;
            for (int a = 0; a < n; a++) accepted += vk[a] > V[a];
            if (accepted < n - accepted) continue;
        }
        double w = 0.0;
        for (int a = 0; a < n; a++) w = __dadd_rn(w, vk[a]);
        if (w > best_w) { best_w = w; best = k; }     // np.argmax: the first maximum
    }
    int src = best;
    if (rule == SOLVER_RULE_MAJORITY && best > 0) {   // all_params[all_vals.index(k1)]
        for (int j = 0; j < best; j++) {
            bool same = true;
            for (int a = 0; a < n; a++) same = same && (V[(size_t)j * n + a] == V[(size_t)best * n + a]);
            if (same) { src = j; break; }
        }
    }
    const double theta = P[src];
    if (best_param) best_param[slot] = theta;
    if (best_idx) best_idx[slot] = src;
    *reinterpret_cast<double*>(p.theta + (size_t)env * p.theta_stride) = theta;
    theta_rows_env(p.rows, n, env, theta);
}

__global__ void solver_choose_kernel(const SolverParams p, int S, int rule, const double* __restrict__ params,
                                     const double* __restrict__ vals, double* __restrict__ best_param, int* __restrict__ best_idx)
{
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.E) return;
    solver_choose_env(p, S, rule, params, vals, best_param, best_idx, env, env);
}

// ---------------------------------------------------------------------------------------------
// Policy-side consumer: what VisionNetwork.forward (environments/Networks/vision_net.py:150-181) does to the observation
// before its first convolution, fused into one pass over the uint8 batch tensor:
//   image    `orig_obs["image"].float().permute(0, 3, 1, 2)` with image = curr_obs / 255 (cleanup_new.py:258, a float64
//            quotient that RLlib hands over as float32): uint8 [E][n][15][15][3] -> T [E n][3][15][15],
//            value = T(float32(float64(x) / 255.0)) through a 256-entry table;
//   contract `orig_obs["contract"].float().repeat(1, 5)` (vision_net.py:160-161): (theta, 0) five times, T [E n][10].
// T = float32, float16 or bfloat16 (SSD_POLICY_F32 / F16 / BF16).  HBM-bound: 675 B read, 675 sizeof(T) written per agent.
// One CTA per env; the windows are staged in shared memory, the outputs leave as coalesced element runs.
// (PolicyElem and policy_cast are in ssd_common.cuh: the observe / reset kernels write the same tensor with a policy output set.)
template <typename T>
__global__ void __launch_bounds__(VIEW_THREADS) policy_inputs_kernel(const GridParams p, const uint8_t* __restrict__ obs, long long obs_stride,
                                                                     T* __restrict__ image, T* __restrict__ contract)
{
    extern __shared__ __align__(16) uint8_t vsm[];            // n windows
    __shared__ float lut[256];
    const int env = blockIdx.x, n = p.n, per_env = n * SSD_OBS_BYTES;
    for (int i = threadIdx.x; i < 256; i += VIEW_THREADS) lut[i] = __double2float_rn(__ddiv_rn((double)i, 255.0));
    const uint8_t* src = obs + (size_t)env * obs_stride;
    if (((reinterpret_cast<uintptr_t>(src) | (uintptr_t)per_env) & 3) == 0)
        for (int w = threadIdx.x; w < per_env / 4; w += VIEW_THREADS) reinterpret_cast<uint32_t*>(vsm)[w] = reinterpret_cast<const uint32_t*>(src)[w];
    else
        for (int b = threadIdx.x; b < per_env; b += VIEW_THREADS) vsm[b] = src[b];
    __syncthreads();
    T* dst = image + (size_t)env * per_env;
    // four consecutive outputs per thread (one 8- or 16-byte store); (agent, channel, pixel) of the first by division,
    // of the next three by stepping
    struct __align__(4 * sizeof(T)) Quad { T v[4]; };
    const bool quads = (per_env & 3) == 0 && (reinterpret_cast<uintptr_t>(image) & (4 * sizeof(T) - 1)) == 0;
    const int step = quads ? 4 : 1;
    for (int o = step * threadIdx.x; o < per_env; o += step * VIEW_THREADS) {          // o = a * 675 + c * 225 + pixel
        int a = o / SSD_OBS_BYTES, r = o - a * SSD_OBS_BYTES;
        int c = r / SSD_OBS_PIX, pix = r - c * SSD_OBS_PIX;
        Quad q;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (k < step) {
                q.v[k] = policy_cast<T>(lut[vsm[a * SSD_OBS_BYTES + pix * 3 + c]]);
                if (++pix == SSD_OBS_PIX) { pix = 0; if (++c == 3) { c = 0; a++; } }
            }
        }
        if (quads) *reinterpret_cast<Quad*>(dst + o) = q;
        else dst[o] = q.v[0];
    }
    if (contract && threadIdx.x < n * 10) {
        const double theta = *reinterpret_cast<const double*>(p.state + (size_t)env * p.rec_stride + RO_THETA);
        contract[(size_t)env * n * 10 + threadIdx.x] = policy_cast<T>((threadIdx.x & 1) ? 0.0f : __double2float_rn(theta));
    }
}
