// ssd_features.cuh — sm_100a kernels for the hand-designed-feature envs CleanupFeatures / HarvestFeatures
// ('Cleanup' / 'Harvest' tags) with the subgame contract wrapper fused in.
//
// Reference behaviour restated here (paths relative to the reference root):
//   environments/cleanup_features.py  step :156-254, reset :256-284, initialize_players :103-109,
//       spawn_apples_and_waste :111-125, compute_closest_* :127-154, compute_probabilities :286-303
//   environments/harvest_features.py  step :173-287, reset :289-336, spawn_apples :139-151,
//       count_apples_in_radius :128-137
//   contract/contract_list.py :22-27, :45-54 ; environments/two_stage_train.py :62-121, :159-187
//
// Mapping (round 2): EIGHT LANES PER ENV (an "octet"; lane = agent), four envs per warp.  Round 1 ran one thread per env:
// 128 registers, 16 warps per SM, 15 of 32 lanes active on average and every thread a ~30 k-instruction dependency chain
// (0.36 ms per step at 131072 envs = 12 % of HBM).  Here
//   * the env's state is the reference's own data structure: current_apple_points / current_waste_points as byte lists of
//     point indices IN LIST (= birth) ORDER — np.argmin ties in compute_closest_* fall to the lowest list position — plus
//     presence bitmasks for the membership tests; a 128-byte hot record (agents, counters, contract parameter, masks) and
//     the two lists are one coalesced load / store per octet;
//   * movement claims are resolved with one ballot per mover, same-cell apple conflicts with one match.any;
//   * a cleaning beam is a table row (cell, orientation) -> bitmask of the waste points its three rays reach (walls are
//     static), so firing is an AND with the waste mask and an exclusive OR-scan over the agents for the attribution;
//   * spawn draws: lane l computes Philox blocks l, l + 8, ... of the step's stream (apple draws and the first waste draws
//     in one pass) and compares its four draws in place; only the successes (a few per step) are mapped from draw rank back
//     to points; HarvestFeatures' regrowth, which reads the list it appends to, is iterated to its fixed point by all lanes;
//   * runtime-bounded loops stay rolled (#pragma unroll 1): unrolled four times by default the kernel was 51 KB of SASS and
//     missed the instruction cache with 32 warps in different phases (no-instruction stalls 3.1 -> 0.3 per issue, +13 %);
//   * closest apple / waste: lane = list slot; the L1 distances of an entry to four agents come from two VABSDIFF4 + one
//     add; a key is 16 bits (distance << 8 | list position) and two agents share a register, so one PRMT builds a pair of
//     keys and one VIMNMX.U16x2 takes both minima; a three-step transpose-reduce leaves agent a's winner in lane a;
//   * removals (eaten apples, cleaned waste) compact the list in place with a ballot-free octet prefix sum;
//   * every lane stores its own agent's feature row (16-byte stores; an octet's rows are one contiguous run).
#pragma once
#include "ssd_common.cuh"

#define FEAT_WARPS 8
#define FEAT_THREADS (FEAT_WARPS * 32)
#define FEAT_ENVS_PER_CTA (FEAT_WARPS * 4)
#define FEAT_MASK_WORDS 8               // up to 256 apple and 256 waste points: mask word w is owned by lane w of the octet
#define FEAT_MAXF 26                    // 10 + 2 * 8
#define FULLMASK 0xffffffffu

// hot record: uint32 [E][32]
enum { FR_AGENT = 0,                    // [8] row | col << 8 | ori << 16
       FR_NA = 8, FR_NW = 9,            // list lengths
       FR_T = 10, FR_EPISODE = 11,      // episode | initialised << 31
       FR_THETA = 12,                   // float64
       FR_AM = 16, FR_WM = 24,          // presence masks
       FR_WORDS = 32 };

struct FeatParams {
    int E, n, kind, H, W, F, horizon, contract;
    int n_apple, n_waste, n_spawn, potential;
    int nwa, nww;               // mask words in use
    int LA, LW, LS;             // list capacities in bytes (multiples of 16), LS = LA + LW
    int sm_static, oct_bytes;   // shared memory: static tables, bytes per octet
    uint32_t seed, first_env_id;
    double theta_low, theta_high, null_prob;
    uint32_t thr_harvest[4], thr_waste;
    // static tables (global memory, read-only)
    const uint8_t* wall;        // [H*W]
    const int16_t* apple_idx;   // [H*W] index into the apple point list or -1
    const int16_t* waste_idx;   // [H*W]
    const uint16_t* apple_rc;   // [n_apple] row << 8 | col
    const uint16_t* waste_rc;   // [n_waste]
    const uint16_t* spawn_rc;   // [n_spawn]
    const uint32_t* waste_start_mask; // [8] points that start as waste ('H')
    const uint32_t* thr_apple;  // [potential + 1] apple spawn threshold by #waste (cleanup)
    const uint8_t* waste_on;    // [potential + 1]
    const uint32_t* beam_tab;   // [H*W][4][nww] waste points reached by a cleaning beam fired from (cell, orientation)
    const uint32_t* near5;      // [H*W][nwa] apple points with j*j + k*k <= 5 around the cell (count_apples_in_radius)
    const uint32_t* nbr_mask;   // [n_apple][nwa] apple points in the 3x3 neighbourhood of a point (harvest regrowth)
    // state
    uint32_t* rec;              // [E][FR_WORDS]
    uint8_t* lists;             // [E][LS]: apple list (LA bytes) then waste list
    double* metrics;            // [8][E] dirt, raw, transfers, apples, low_density
    uint32_t* sum_raw;          // [n][E]
    unsigned long long* tsum_raw; // [n][E]
    double* sum_tr;             // [n][E]
    double* tsum_tr;            // [n][E]
    EpisodeLog elog;            // optional: ssd_set_episode_log ring buffer (appended to by the resets of feat_kernel)
};

struct FeatIO {
    const uint8_t* actions;     // [E][n]
    void* obs;                  // double [E][n][F] (OBS_F64), or the policy's rows T [E n][W] (1 + SSD_POLICY_*: feat_policy_row)
    double* rew; double* base_rew; double* transfers;   // [E][n]
    uint8_t* info;              // [E][n][4]: cleanup (cleaned_squares,0,0,0); harvest (eaten_apples, eaten_close_apples,0,0)
    uint8_t* done;              // [E]
    int auto_reset;             // next-step auto-reset (see feat_kernel)
    // compact result block of ssd_feat_step_host_async (all null otherwise): int8 rewards, dones, and records
    // { int32 env; int32 0; double rew[n] } for the envs whose rewards are not all integers in [-127, 127]
    int8_t* c_rew8; uint8_t* c_done; uint32_t* c_count; uint8_t* c_rec;
};

// ---- octet primitives (all 32 lanes execute them; an octet is lanes obase .. obase + 7) --------------------------------
__device__ __forceinline__ int oct_scan_incl(int v, int a)
{
#pragma unroll
    for (int d = 1; d < 8; d <<= 1) { const int t = __shfl_up_sync(FULLMASK, v, d, 8); if (a >= d) v += t; }
    return v;
}
__device__ __forceinline__ int oct_sum(int v)
{
    v += __shfl_xor_sync(FULLMASK, v, 1); v += __shfl_xor_sync(FULLMASK, v, 2); v += __shfl_xor_sync(FULLMASK, v, 4);
    return v;
}
__device__ __forceinline__ uint32_t oct_or(uint32_t v)
{
    v |= __shfl_xor_sync(FULLMASK, v, 1); v |= __shfl_xor_sync(FULLMASK, v, 2); v |= __shfl_xor_sync(FULLMASK, v, 4);
    return v;
}
__device__ __forceinline__ double shfl_f64(double v, int src)
{
    const int lo = __shfl_sync(FULLMASK, __double2loint(v), src, 8), hi = __shfl_sync(FULLMASK, __double2hiint(v), src, 8);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ uint32_t feat_valid_word(int npts, int w)
{
    const int left = npts - 32 * w;
    return left >= 32 ? 0xFFFFFFFFu : (left <= 0 ? 0u : ((1u << left) - 1u));
}
__device__ __forceinline__ int feat_cell(const FeatParams& p, uint32_t pos)
{
    const int r = min((int)(pos & 255u), p.H - 1), c = min((int)((pos >> 8) & 255u), p.W - 1);
    return r * p.W + c;
}
// position of the j-th (0-based) set bit of x (x has more than j set bits)
__device__ __forceinline__ int select_bit(uint32_t x, int j)
{
    int pos = 0, c;
    c = __popc(x & 0xFFFFu); if (j >= c) { j -= c; pos += 16; x >>= 16; }
    c = __popc(x & 0xFFu);   if (j >= c) { j -= c; pos += 8;  x >>= 8; }
    c = __popc(x & 0xFu);    if (j >= c) { j -= c; pos += 4;  x >>= 4; }
    c = __popc(x & 0x3u);    if (j >= c) { j -= c; pos += 2;  x >>= 2; }
    if (j >= (int)(x & 1u)) pos += 1;
    return pos;
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem)
{
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// list.remove() of every entry whose point left the presence mask m[0..7], in place (order kept).  Lane a takes words a,
// a + 8, ... of the list (4 entries each); a round's reads finish before its writes, and writes never pass the round's
// own read positions.  Octets with need == false keep their list.  Returns the new length (octet-uniform).  (Not inlined: see oct_closest.)
__device__ __noinline__ int oct_compact(uint8_t* list, int L, bool need, const uint32_t* m, int a)
{
    const int Leff = need ? L : 0;
    const int Lmax = __reduce_max_sync(FULLMASK, Leff);
    int out = 0;
#pragma unroll 1
    for (int w0 = 0; w0 * 4 < Lmax; w0 += 8) {
        const int wi = w0 + a;
        uint32_t e4 = 0u, keep = 0u;
        if (wi * 4 < Leff) {
            e4 = *reinterpret_cast<const uint32_t*>(list + 4 * wi);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint32_t idx = (e4 >> (8 * j)) & 255u;
                if (4 * wi + j < Leff && ((m[idx >> 5] >> (idx & 31u)) & 1u)) keep |= 1u << j;
            }
        }
        const int kc = __popc(keep);
        const int incl = oct_scan_incl(kc, a);
        const int tot = __shfl_sync(FULLMASK, incl, 7, 8);
        __syncwarp();
        int o = out + incl - kc;
#pragma unroll
        for (int j = 0; j < 4; j++) if ((keep >> j) & 1u) list[o++] = (uint8_t)((e4 >> (8 * j)) & 255u);
        out += tot;
        __syncwarp();
    }
    return need ? out : L;
}

// compute_closest_*: for agent a (left in lane a) the entry of the list with the smallest (L1 distance, list position);
// returns its row << 8 | col, or 0 — the reference's [0, 0] sentinel — for an empty list.  ar / ac: the agents' rows /
// columns packed one per byte (agents 0-3, 4-7); absent agents sit at (127, 127) so that no byte sum carries.
// A key is 16 bits (distance << 8 | list position), two agents share a register: one PRMT builds a pair of keys and one
// VIMNMX.U16x2 takes both minima.  (Not inlined: the cleanup kernel calls it for both lists and its hot path should stay
// inside the instruction cache.)
__device__ __noinline__ uint32_t oct_closest(const uint8_t* list, int L, const uint16_t* rc, uint32_t ar0, uint32_t ar1,
                                             uint32_t ac0, uint32_t ac1, bool n_gt4, int a)
{
    const int Lmax = __reduce_max_sync(FULLMASK, L);
    uint32_t b01 = 0xFFFFFFFFu, b23 = 0xFFFFFFFFu, b45 = 0xFFFFFFFFu, b67 = 0xFFFFFFFFu;
#pragma unroll 1
    for (int w0 = 0; w0 * 4 < Lmax; w0 += 8) {
        const int wi = w0 + a;
        if (wi * 4 >= L) continue;                               // (no collectives inside the loop)
        const uint32_t e4 = *reinterpret_cast<const uint32_t*>(list + 4 * wi);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t pos = (uint32_t)(4 * wi + j);
            const uint32_t prc = rc[(e4 >> (8 * j)) & 255u];
            const uint32_t pr4 = __byte_perm(prc, 0u, 0x1111), pc4 = __byte_perm(prc, 0u, 0x0000);   // row / col in every byte
            const bool live = (int)pos < L;
            uint32_t d0 = __vabsdiffu4(pr4, ar0) + __vabsdiffu4(pc4, ac0);
            if (!live) d0 = 0xFFFFFFFFu;
            b01 = __vminu2(b01, __byte_perm(d0, pos, 0x1404));   // (d_0 << 8 | pos) | (d_1 << 8 | pos) << 16
            b23 = __vminu2(b23, __byte_perm(d0, pos, 0x3424));
            if (n_gt4) {
                uint32_t d1 = __vabsdiffu4(pr4, ar1) + __vabsdiffu4(pc4, ac1);
                if (!live) d1 = 0xFFFFFFFFu;
                b45 = __vminu2(b45, __byte_perm(d1, pos, 0x1404));
                b67 = __vminu2(b67, __byte_perm(d1, pos, 0x3424));
            }
        }
    }
    // transpose-reduce: lane a ends with the minimum over the octet of agent a's key
    const bool h4 = (a & 4) != 0, h2 = (a & 2) != 0;
    uint32_t k0 = __vminu2(h4 ? b45 : b01, __shfl_xor_sync(FULLMASK, h4 ? b01 : b45, 4));
    uint32_t k1 = __vminu2(h4 ? b67 : b23, __shfl_xor_sync(FULLMASK, h4 ? b23 : b67, 4));
    uint32_t k = __vminu2(h2 ? k1 : k0, __shfl_xor_sync(FULLMASK, h2 ? k0 : k1, 2));
    k = __vminu2(k, __shfl_xor_sync(FULLMASK, k, 1));
    const uint32_t key = (a & 1) ? k >> 16 : k & 0xFFFFu;
    if ((key >> 8) >= 0xFFu) return 0u;                           // no live entry
    return rc[list[key & 255u]];
}

// Element q of env's ssd_feat_get_metrics row (40 doubles; 0 beyond): dirt, raw, transfers, apples, low_density, err_flags,
// 0, 0, sum_raw[8], tsum_raw[8], sum_tr[8], tsum_tr[8] from the [k][E] accumulators.  What ssd_feat_get_metrics writes and
// what a reset hands to the episode log.  (Scalar arguments: a FeatParams reference into the non-inlined caller below
// would copy the kernel parameters to the stack.)
__device__ __forceinline__ double feat_metric(const double* metrics, const uint32_t* sum_raw, const unsigned long long* tsum_raw,
                                              const double* sum_tr, const double* tsum_tr, int E, int n, int env, int q)
{
    if (q < 8) return q < 6 ? metrics[(size_t)q * E + env] : 0.0;    // [5]: err_flags (unused: no wrapping stamps any more)
    const int a = q & 7;
    if (a >= n) return 0.0;
    const size_t so = (size_t)a * E + env;
    switch (q >> 3) {
    case 1: return (double)sum_raw[so];
    case 2: return (double)tsum_raw[so];
    case 3: return sum_tr[so];
    case 4: return tsum_tr[so];
    default: return 0.0;
    }
}

// Episode log of the resets of one feat_kernel round (all 32 lanes; `mine`: this octet resets an initialised env): one
// atomic for the warp's up to four records, then the octet writes its env's record, lane a the vectors a, a + 8, ...  Reads
// the accumulators before the reset zeroes them.  Out of line: the step's hot path stays small in the instruction cache
// (DESIGN §4.5a).
__device__ __noinline__ void feat_log_episode(EpisodeLog log, const double* metrics, const uint32_t* sum_raw,
                                              const unsigned long long* tsum_raw, const double* sum_tr, const double* tsum_tr,
                                              int E, int n, int horizon, int env, uint32_t env_id, bool mine, uint32_t episode,
                                              int t, double theta, int lane)
{
    const int a = lane & 7, obase = lane & 24;
    const uint32_t lm = __ballot_sync(FULLMASK, mine && a == 0);
    if (!lm) return;
    const int leader = __ffs(lm) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(log.count, (unsigned long long)__popc(lm));
    base = __shfl_sync(FULLMASK, base, leader);
    if (!mine) return;
    const unsigned long long slot = (base + (unsigned long long)__popc(lm & ((1u << obase) - 1u))) % log.capacity;
    uint4* rec = log.records + slot * EPREC_VECS;
#pragma unroll 1
    for (int v = a; v < EPREC_VECS; v += 8) {
        uint4 w;
        if (v == 0) w = eprec_head(env_id, episode, t, t == horizon);
        else if (v == 1) w = eprec_pair(theta, 0.0);
        else w = eprec_pair(feat_metric(metrics, sum_raw, tsum_raw, sum_tr, tsum_tr, E, n, env, 2 * v - 4),
                            feat_metric(metrics, sum_raw, tsum_raw, sum_tr, tsum_tr, E, n, env, 2 * v - 3));
        rec[v] = w;
    }
}

#ifndef FEAT_MIN_BLOCKS
#define FEAT_MIN_BLOCKS 4
#endif
#ifndef FEAT_WASTE_DRAWS
#define FEAT_WASTE_DRAWS 8               // waste draws evaluated together with the apple draws (more only when all of them fail)
#endif

// two policy elements at a 4-byte (T = 16-bit) or 8-byte (T = float) aligned address
__device__ __forceinline__ void policy_store2(float* o, double x, double y)
{
    *reinterpret_cast<float2*>(o) = make_float2(__double2float_rn(x), __double2float_rn(y));
}
__device__ __forceinline__ void policy_store2(__half* o, double x, double y)
{
    *reinterpret_cast<__half2*>(o) = __halves2half2(__float2half_rn(__double2float_rn(x)), __float2half_rn(__double2float_rn(y)));
}
__device__ __forceinline__ void policy_store2(__nv_bfloat16* o, double x, double y)
{
    *reinterpret_cast<__nv_bfloat162*>(o) = __halves2bfloat162(__float2bfloat16_rn(__double2float_rn(x)), __float2bfloat16_rn(__double2float_rn(y)));
}

// The policy form's row of one agent: its F features ++ [theta, 0] with a contract, each T(float32(x)).  Row r starts at
// byte r W sizeof(T), so it can start on any multiple of 2 bytes: when W is even (then F is even too) every row starts on
// a pair and goes out in two-element stores, otherwise (cleanup with an odd agent count) element by element.
template <typename T>
__device__ __forceinline__ void feat_policy_row(T* o, const double (&v)[FEAT_MAXF], int F, bool contract, double theta)
{
    if ((F & 1) == 0) {
#pragma unroll
        for (int k = 0; k < FEAT_MAXF; k += 2) if (k < F) policy_store2(o + k, v[k], v[k + 1]);
        if (contract) policy_store2(o + F, theta, 0.0);
    } else {
#pragma unroll
        for (int k = 0; k < FEAT_MAXF; k++) if (k < F) o[k] = policy_cast<T>(__double2float_rn(v[k]));
        if (contract) { o[F] = policy_cast<T>(__double2float_rn(theta)); o[F + 1] = policy_cast<T>(0.0f); }
    }
}

// One launch = one step (or, RESET_ONLY, one masked reset) of every env.
// Next-step auto-reset (ssd_feat_io.auto_reset): an env that reached its horizon in the previous step starts its next
// episode in this one — reset observation, zero rewards, done cleared, the actions of this step ignored.
// FORM: OBS_F64 (float64 rows [E][n][F]) or 1 + SSD_POLICY_* (the policy's rows, feat_policy_row).
template <bool CLEANUP, bool RESET_ONLY, int FORM>
__global__ void __launch_bounds__(FEAT_THREADS, FEAT_MIN_BLOCKS) feat_kernel(const FeatParams p, const FeatIO io, const uint8_t* __restrict__ mask)
{
    extern __shared__ __align__(16) uint8_t fsm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, a = lane & 7, obase = lane & 24;
    const int n = p.n;
    // row << 8 | col of every point, 256 entries per table: the closest search also looks up the (ignored) bytes behind a
    // list's end in its last word, which may hold anything
    uint16_t* s_arc = reinterpret_cast<uint16_t*>(fsm);
    uint16_t* s_wrc = s_arc + 32 * FEAT_MASK_WORDS;
    for (int i = threadIdx.x; i < 32 * FEAT_MASK_WORDS; i += FEAT_THREADS) {
        s_arc[i] = i < p.n_apple ? __ldg(p.apple_rc + i) : (uint16_t)0;
        s_wrc[i] = i < p.n_waste ? __ldg(p.waste_rc + i) : (uint16_t)0;
    }
    __syncthreads();
    // persistent CTAs: a warp takes four envs per round
    const int ngroups = (p.E + FEAT_ENVS_PER_CTA - 1) / FEAT_ENVS_PER_CTA;
#pragma unroll 1
    for (int grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
    const int env_raw = (grp * FEAT_WARPS + warp) * 4 + (lane >> 3);
    bool active = env_raw < p.E;
    const int env = active ? env_raw : p.E - 1;
    if (RESET_ONLY && mask) active = active && mask[env] != 0;
    if (RESET_ONLY && !__any_sync(FULLMASK, active)) continue;

    uint8_t* ob = fsm + p.sm_static + (size_t)(warp * 4 + (lane >> 3)) * p.oct_bytes;
    uint32_t* s_rec = reinterpret_cast<uint32_t*>(ob);
    uint32_t* s_scr = s_rec + 32;                    // [0..7] eligibility, [8..15] / [16..23] success bits by draw rank
    uint8_t* s_al = ob + 256;
    uint8_t* s_wl = s_al + p.LA;
    uint32_t* grec = p.rec + (size_t)env * FR_WORDS;
    uint8_t* glist = p.lists + (size_t)env * p.LS;

    // ---- state in: the hot record (16 bytes per lane), then the live parts of the two lists (asynchronous copies)
    {
        uint4 h4 = make_uint4(0u, 0u, 0u, 0u);
        if (active) h4 = *reinterpret_cast<const uint4*>(grec + 4 * a);
        *reinterpret_cast<uint4*>(s_rec + 4 * a) = h4;
    }
    __syncwarp();
    const uint32_t c3 = s_rec[FR_EPISODE];
    const bool doreset = RESET_ONLY ? active : (active && io.auto_reset && (int)s_rec[FR_T] == p.horizon);
    const bool stepping = !RESET_ONLY && active && !doreset;
    int nA = stepping ? (int)s_rec[FR_NA] : 0, nW = stepping ? (int)s_rec[FR_NW] : 0;
    if (!RESET_ONLY) {
        // (LA, LW <= 256: at most two 16-byte chunks per lane and list)
        if (a * 16 < nA) cp_async16(s_al + 16 * a, glist + 16 * a);
        if ((a + 8) * 16 < nA) cp_async16(s_al + 16 * (a + 8), glist + 16 * (a + 8));
        if (a * 16 < nW) cp_async16(s_wl + 16 * a, glist + p.LA + 16 * a);
        if ((a + 8) * 16 < nW) cp_async16(s_wl + 16 * (a + 8), glist + p.LA + 16 * (a + 8));
    }
    uint32_t episode = c3 & 0x7fffffffu;
    const uint32_t env_id = p.first_env_id + (uint32_t)env;
    double theta = __hiloint2double((int)s_rec[FR_THETA + 1], (int)s_rec[FR_THETA]);
    uint32_t pos = a < n ? s_rec[FR_AGENT + a] : 0u;
    bool a_chg = false, w_chg = false;               // lists to write back

    // ---- reset (cleanup_features.py:256-284 / harvest_features.py:289-336 + two_stage_train.py:159-187)
    if (__any_sync(FULLMASK, doreset)) {
        if (p.elog.records)                          // hand the finished episodes over before their accumulators are zeroed
            feat_log_episode(p.elog, p.metrics, p.sum_raw, p.tsum_raw, p.sum_tr, p.tsum_tr, p.E, n, p.horizon, env, env_id,
                             doreset && (c3 & 0x80000000u), c3 & 0x7fffffffu, (int)s_rec[FR_T], theta, lane);
        uint32_t sm = (CLEANUP && doreset) ? __ldg(p.waste_start_mask + a) : 0u;
        const int sc = __popc(sm);
        const int sincl = oct_scan_incl(sc, a);
        const int stot = __shfl_sync(FULLMASK, sincl, 7, 8);
        if (doreset) {
            episode = (c3 & 0x80000000u) ? (c3 & 0x7fffffffu) + 1u : 0u;
            // initialize_arrays
            if (CLEANUP) {
                s_rec[FR_AM + a] = 0u; s_rec[FR_WM + a] = sm;
                int o = sincl - sc;
#pragma unroll 1
                while (sm) { const int b = __ffs(sm) - 1; sm &= sm - 1; s_wl[o++] = (uint8_t)(a * 32 + b); }
                nA = 0; nW = stot;
            } else {
                s_rec[FR_AM + a] = feat_valid_word(p.n_apple, a); s_rec[FR_WM + a] = 0u;
                for (int i = a; i < p.n_apple; i += 8) s_al[i] = (uint8_t)i;
                nA = p.n_apple; nW = 0;
            }
            a_chg = w_chg = true;
            // initialize_players: agent a takes the spawn point with the (a+1)-th smallest (key, index).  Every lane walks
            // all keys (one Philox block per four points) keeping the n smallest in a sorted register list.
            {
                uint32_t bk[SSD_MAXN]; int bj[SSD_MAXN];
#pragma unroll
                for (int q = 0; q < SSD_MAXN; q++) { bk[q] = 0xffffffffu; bj[q] = 0x7fffffff; }
                Philox4 blk = { 0, 0, 0, 0 };
#pragma unroll 1
                for (int j = 0; j < p.n_spawn; j++) {
                    if ((j & 3) == 0) blk = draw_block(p.seed, env_id, episode, 0u, SITE_FEAT_ORDER, 0u, (uint32_t)(j >> 2));
                    uint32_t kk = pick(blk, (uint32_t)j & 3u); int jj = j;
#pragma unroll
                    for (int q = 0; q < SSD_MAXN; q++) {             // insertion: (kk, jj) sinks to its place, the rest shift down
                        const bool less = kk < bk[q] || (kk == bk[q] && jj < bj[q]);
                        const uint32_t tk = bk[q]; const int tj = bj[q];
                        if (less) { bk[q] = kk; bj[q] = jj; kk = tk; jj = tj; }
                    }
                }
                int mine = bj[0];
#pragma unroll
                for (int q = 1; q < SSD_MAXN; q++) if (a == q) mine = bj[q];
                if (a < n) {
                    const uint32_t rc = __ldg(p.spawn_rc + mine);
                    const uint32_t o = draw_u32(p.seed, env_id, episode, 0u, SITE_FEAT_ROT, (uint32_t)a, 0u) >> 30;
                    pos = (rc >> 8) | ((rc & 255u) << 8) | (o << 16);
                }
            }
            theta = 0.0;
            if (p.contract != SSD_CONTRACT_NONE) {
                const double u0 = __dmul_rn((double)draw_u32(p.seed, env_id, episode, 0u, SITE_CONTRACT, 0u, 0u), 1.0 / 4294967296.0);
                const double u1 = __dmul_rn((double)draw_u32(p.seed, env_id, episode, 0u, SITE_CONTRACT, 0u, 1u), 1.0 / 4294967296.0);
                theta = (u0 > p.null_prob) ? __dadd_rn(p.theta_low, __dmul_rn(__dsub_rn(p.theta_high, p.theta_low), u1)) : p.theta_low;
            }
            if (a < n) {
                const size_t so = (size_t)a * p.E + env;
                p.sum_raw[so] = 0u; p.tsum_raw[so] = 0ull; p.sum_tr[so] = 0.0; p.tsum_tr[so] = 0.0;
            }
            p.metrics[(size_t)a * p.E + env] = 0.0;
        }
        __syncwarp();
    }

    int reward = 0, eaten = 0, eaten_close = 0, cleaned = 0, dirt = 0;
    if (!RESET_ONLY) {
        // ---- moves (cleanup_features.py:162-183): stays claim first, then the movers in agent order
        int act = 255;
        if (stepping && a < n) act = io.actions[(size_t)env * n + a];
        const bool agent_ok = stepping && a < n;
        const bool mover = agent_ok && act < 4;
        bool has = agent_ok && (CLEANUP ? act == 4 : act > 3);
        uint32_t claim = pos & 0xFFFFu, tgt = claim;
        bool wallblk = false;
        if (mover) {
            const int r = (int)(pos & 255u), c = (int)((pos >> 8) & 255u);
            const int tr = r + (act == 2 ? -1 : (act == 3 ? 1 : 0)), tc = c + (act == 0 ? -1 : (act == 1 ? 1 : 0));
            tgt = (uint32_t)tr | ((uint32_t)tc << 8);
            wallblk = (tr < 0 || tr >= p.H || tc < 0 || tc >= p.W) ? false : __ldg(p.wall + tr * p.W + tc) != 0;
        }
        const uint32_t mv_all = __ballot_sync(FULLMASK, mover);
        {
            // A mover is blocked by a wall or by a square claimed before it.  If the squares the agents WOULD claim — their
            // own for stays and for movers facing a wall, the target for the other movers — are all distinct, nobody can be
            // blocked by a claim; only otherwise the movers are taken one at a time.
            const uint32_t want = (mover && !wallblk) ? tgt : (pos & 0xFFFFu);
            const uint32_t key = (has || mover) ? (((uint32_t)obase << 16) | (want & 0xFFFFu)) : (0x80000000u | (uint32_t)lane);
            const bool clash = __popc(__match_any_sync(FULLMASK, key)) > 1;
            if (__any_sync(FULLMASK, clash)) {
                const uint32_t mv_any = (mv_all | (mv_all >> 8) | (mv_all >> 16) | (mv_all >> 24)) & 0xFFu;
#pragma unroll 1
                for (int m = 0; m < n; m++) {
                    if (!((mv_any >> m) & 1u)) continue;
                    const uint32_t tgt_m = __shfl_sync(FULLMASK, tgt, m, 8);
                    const uint32_t hit = (__ballot_sync(FULLMASK, has && claim == tgt_m) >> obase) & 0xFFu;
                    if (a == m && mover) { claim = (wallblk || hit) ? (pos & 0xFFFFu) : tgt; has = true; }
                }
            } else if (mover) { claim = want; has = true; }
        }
        if (has) pos = (pos & 0xFFFF0000u) | claim;

        // ---- consume in move_squares insertion order: stays (agent order), then movers (agent order)
        cp_async_wait_all();
        __syncwarp();
        const int cell = feat_cell(p, pos);
        int ai = -1;
        if (has) ai = __ldg(p.apple_idx + cell);
        bool cand = ai >= 0 && ((s_rec[FR_AM + (ai >> 5)] >> (ai & 31)) & 1u);
        {   // two agents can share a cell: the first in insertion order eats
            const uint32_t key = cand ? (((uint32_t)obase << 16) | (uint32_t)ai) : (0x80000000u | (uint32_t)lane);
            const uint32_t grp = __match_any_sync(FULLMASK, key);
            const uint32_t stays = grp & ~mv_all;
            const int winner = stays ? __ffs(stays) - 1 : __ffs(grp) - 1;
            cand = cand && winner == lane;
        }
        if (CLEANUP) {
            if (cand) { reward = 1; atomicAnd(&s_rec[FR_AM + (ai >> 5)], ~(1u << (ai & 31))); }
        } else {
            // harvest_features.py:204-215: an eater also counts the apples within the radius of its square at the moment it
            // eats (its own apple included, earlier eaters' apples gone), so the eaters go one at a time
            uint32_t pend = __ballot_sync(FULLMASK, cand);
#pragma unroll 1
            while (pend) {
                const uint32_t pe = (pend >> obase) & 0xFFu, st = pe & ~(mv_all >> obase);
                const int nxt = pe ? (st ? __ffs(st) - 1 : __ffs(pe) - 1) : -1;
                const int cell_n = __shfl_sync(FULLMASK, cell, nxt < 0 ? 0 : nxt, 8);
                int cnt = 0;
                if (nxt >= 0 && a < p.nwa) cnt = __popc(s_rec[FR_AM + a] & __ldg(p.near5 + (size_t)cell_n * p.nwa + a));
                cnt = oct_sum(cnt);
                __syncwarp();
                if (a == nxt) {
                    reward = 1; eaten = 1; eaten_close = cnt < 4 ? 1 : 0; cand = false;
                    s_rec[FR_AM + (ai >> 5)] &= ~(1u << (ai & 31));
                }
                __syncwarp();
                pend = __ballot_sync(FULLMASK, cand);
            }
        }
        const uint32_t ate = __ballot_sync(FULLMASK, reward != 0);
        if (ate) {
            __syncwarp();
            const bool need = ((ate >> obase) & 0xFFu) != 0u;
            nA = oct_compact(s_al, nA, need, s_rec + FR_AM, a);
            a_chg = a_chg || need;
        }
        // ---- rotations
        if (agent_ok) {
            uint32_t o = (pos >> 16) & 3u;
            if (act == 5) o = (o + 1u) & 3u;
            if (act == 6) o = (o + 3u) & 3u;
            pos = (pos & 0xFFFFu) | (o << 16);
        }
        // ---- cleaning beams (cleanup_features.py:196-219): 3 rays x 6 cells incl. the agent's own, stopped by walls only.
        // Agents fire in index order, so a waste cell goes to the first firing agent whose beam reaches it.
        if (CLEANUP) {
            const bool fire = agent_ok && act == 7;
            if (__any_sync(FULLMASK, fire)) {
                const uint32_t* row = p.beam_tab + ((size_t)feat_cell(p, pos) * 4 + ((pos >> 16) & 3u)) * p.nww;
#pragma unroll 1
                for (int w = 0; w < p.nww; w++) {
                    const uint32_t wmw = s_rec[FR_WM + w];
                    const uint32_t v = fire ? (__ldg(row + w) & wmw) : 0u;
                    uint32_t incl = v;
#pragma unroll
                    for (int d = 1; d < 8; d <<= 1) { const uint32_t t = __shfl_up_sync(FULLMASK, incl, d, 8); if (a >= d) incl |= t; }
                    uint32_t excl = __shfl_up_sync(FULLMASK, incl, 1, 8);
                    if (a == 0) excl = 0u;
                    cleaned += __popc(v & ~excl);
                    const uint32_t all = __shfl_sync(FULLMASK, incl, 7, 8);
                    dirt += __popc(all);
                    __syncwarp();
                    if (a == 0 && all) s_rec[FR_WM + w] = wmw & ~all;
                }
                __syncwarp();
                if (__any_sync(FULLMASK, dirt != 0)) {
                    nW = oct_compact(s_wl, nW, dirt != 0, s_rec + FR_WM, a);
                    w_chg = w_chg || dirt != 0;
                }
            }
        }
    }

    // ---- spawn_apples_and_waste (cleanup_features.py:111-125) / spawn_apples (harvest_features.py:139-151).
    // The k-th random.random() of the step is draw k of the step's Philox stream (block k >> 2, word k & 3); an apple point
    // that is neither in the list nor under an agent consumes one draw, in point order.
    const uint32_t tdraw = doreset ? 0u : s_rec[FR_T] + 1u;
    s_scr[a] = ~s_rec[FR_AM + a] & feat_valid_word(p.n_apple, a);
    s_scr[8 + a] = 0u;
    if (!CLEANUP) s_scr[16 + a] = 0u;
    __syncwarp();
    if (active && a < n) {
        const int aj = __ldg(p.apple_idx + feat_cell(p, pos));
        if (aj >= 0) atomicAnd(&s_scr[aj >> 5], ~(1u << (aj & 31)));
    }
    __syncwarp();
    const uint32_t elig = active ? s_scr[a] : 0u;
    const int ecnt = __popc(elig);
    // (cleanup: the waste candidates are counted in the same scan, in the upper half of the word)
    const uint32_t thrA = (CLEANUP && active) ? __ldg(p.thr_apple + nW) : 0u;       // compute_probabilities by the waste count
    const bool won = CLEANUP && active && __ldg(p.waste_on + nW) != 0;
    // at most one waste point: the first success over the points that are not waste, in point order; its draws
    // follow the apple draws in the step's stream (candidate rank j <-> draw nelig + j)
    const uint32_t cwm = won ? (~s_rec[FR_WM + a] & feat_valid_word(p.n_waste, a)) : 0u;
    const int ccnt = __popc(cwm);
    const int pincl = oct_scan_incl(ecnt | (ccnt << 16), a);
    const int ptot = __shfl_sync(FULLMASK, pincl, 7, 8);
    const int eexcl = (pincl & 0xFFFF) - ecnt, nelig = ptot & 0xFFFF;
    if constexpr (CLEANUP) {
        const int cexcl = (pincl >> 16) - ccnt, ncand = ptot >> 16;
        const int k0 = nelig;
        // ONE pass over the Philox blocks: the apple blocks (when the apple probability is not 0 — otherwise r < 0 never
        // holds and the draws are consumed unseen) and, with them, the blocks of the first FEAT_WASTE_DRAWS waste draws
        const int nblk_a = thrA ? (nelig + 3) >> 2 : 0;
        const bool wsearch = won && ncand > 0;
        const int bw0 = k0 >> 2;                                           // block of the first waste draw
        const int bw1 = wsearch ? ((k0 + min(ncand, FEAT_WASTE_DRAWS) + 3) >> 2) : 0;   // end of the first waste blocks
        const int bstart = thrA ? 0 : bw0, bend = max(nblk_a, bw1);
        const int maxcnt = __reduce_max_sync(FULLMASK, max(bend - bstart, 0));
        uint32_t wbits = 0u;                                               // waste successes by candidate rank (< 32)
#pragma unroll 1
        for (int b0 = 0; b0 < maxcnt; b0 += 8) {
            const int b = bstart + b0 + a;
            if (b < bend) {
                const Philox4 q = philox4x32_10((uint32_t)b, SITE_FEAT_SPAWN, tdraw, episode, p.seed, env_id);
                if (b < nblk_a) {
                    uint32_t bits = (q.x < thrA ? 1u : 0u) | (q.y < thrA ? 2u : 0u) | (q.z < thrA ? 4u : 0u) | (q.w < thrA ? 8u : 0u);
                    const int left = nelig - 4 * b;
                    if (left < 4) bits &= (1u << left) - 1u;
                    if (bits) atomicOr(&s_scr[8 + (b >> 3)], bits << ((b & 7) * 4));
                }
                if (wsearch && b >= bw0) {
                    const uint32_t bits = (q.x < p.thr_waste ? 1u : 0u) | (q.y < p.thr_waste ? 2u : 0u) | (q.z < p.thr_waste ? 4u : 0u) | (q.w < p.thr_waste ? 8u : 0u);
                    const int r0 = 4 * b - k0;                             // candidate rank of the block's first draw (>= -3)
                    wbits |= r0 >= 0 ? (r0 < 32 ? bits << r0 : 0u) : bits >> (-r0);
                }
            }
        }
        __syncwarp();
        {   // apple successes by draw rank -> points of this lane's mask word, appended in point order
            uint32_t sb = 0u;
            if (ecnt) {
                const int w = eexcl >> 5;
                const uint32_t lo = s_scr[8 + w], hi = w + 1 < 8 ? s_scr[8 + w + 1] : 0u;
                sb = __funnelshift_r(lo, hi, (uint32_t)(eexcl & 31));
                if (ecnt < 32) sb &= (1u << ecnt) - 1u;
            }
            if (__any_sync(FULLMASK, sb != 0u)) {
                const int scnt = __popc(sb);
                const int sincl = oct_scan_incl(scnt, a);
                const int stot = __shfl_sync(FULLMASK, sincl, 7, 8);
                int lp = nA + sincl - scnt;
#pragma unroll 1
                while (sb) {
                    const int j = __ffs(sb) - 1; sb &= sb - 1;
                    const int bit = select_bit(elig, j);
                    s_rec[FR_AM + a] |= 1u << bit;
                    s_al[lp++] = (uint8_t)(a * 32 + bit);
                }
                nA += stot;
                a_chg = a_chg || stot != 0;
            }
        }
        wbits = oct_or(wbits);
        int covered = wsearch ? min(4 * bw1 - k0, 32) : 0;                 // candidate ranks looked at so far
        if (covered > ncand) covered = ncand;
        if (covered < 32) wbits &= (1u << max(covered, 0)) - 1u;
        int jstar = wbits ? __ffs(wbits) - 1 : -1;
        bool searching = wsearch && jstar < 0 && covered < ncand;          // (1 / 2^FEAT_WASTE_DRAWS of the steps at p = 0.5)
#pragma unroll 1
        while (__any_sync(FULLMASK, searching)) {
            // eight more blocks: draws k0 + covered - ((k0 + covered) & 3) ...
            const int d0 = k0 + covered, bb = (d0 >> 2) + a;
            uint32_t bits = 0u;
            if (searching) {
                const Philox4 q = philox4x32_10((uint32_t)bb, SITE_FEAT_SPAWN, tdraw, episode, p.seed, env_id);
                bits = ((q.x < p.thr_waste ? 1u : 0u) | (q.y < p.thr_waste ? 2u : 0u) | (q.z < p.thr_waste ? 4u : 0u) | (q.w < p.thr_waste ? 8u : 0u)) << (4 * a);
            }
            bits = oct_or(bits);
            if (searching) {
                const int skip = d0 & 3;                                   // draws of the first block that were looked at already
                const int rbase = covered - skip;                          // candidate rank of bit 0
                uint32_t ok = bits & (0xFFFFFFFFu << skip);
                const int lim = ncand - rbase;
                if (lim < 32) ok &= (1u << lim) - 1u;
                if (ok) { jstar = rbase + __ffs(ok) - 1; searching = false; }
                else { covered = rbase + 32; if (covered >= ncand) searching = false; }
            }
        }
        if (jstar >= cexcl && jstar < cexcl + ccnt) {
            const int bit = select_bit(cwm, jstar - cexcl);
            s_rec[FR_WM + a] |= 1u << bit;
            s_wl[nW] = (uint8_t)(a * 32 + bit);
        }
        if (jstar >= 0) { nW++; w_chg = true; }
    } else {
        // regrowth probability by the number of apples in the 3x3 neighbourhood, READ FROM THE LIST BEING APPENDED TO: a
        // draw is ranked against the three thresholds (SPAWN_PROB is increasing: level 3 = below all of them) and the few
        // ranked draws are then resolved in point order against the live mask by the lane that owns the point's word.
        const int nblk = (nelig + 3) >> 2;
        const int maxblk = __reduce_max_sync(FULLMASK, nblk);
#pragma unroll 1
        for (int b0 = 0; b0 < maxblk; b0 += 8) {
            const int b = b0 + a;
            if (b < nblk) {
                const Philox4 q = philox4x32_10((uint32_t)b, SITE_FEAT_SPAWN, tdraw, episode, p.seed, env_id);
                if (min(min(q.x, q.y), min(q.z, q.w)) < p.thr_harvest[3]) {        // (one block in five)
                    const uint32_t d[4] = { q.x, q.y, q.z, q.w };
                    uint32_t lo = 0u, hi = 0u;
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const uint32_t lvl = (d[j] < p.thr_harvest[1] ? 1u : 0u) + (d[j] < p.thr_harvest[2] ? 1u : 0u) + (d[j] < p.thr_harvest[3] ? 1u : 0u);
                        lo |= (lvl & 1u) << j; hi |= (lvl >> 1) << j;
                    }
                    const int left = nelig - 4 * b;
                    if (left < 4) { lo &= (1u << left) - 1u; hi &= (1u << left) - 1u; }
                    if (lo) atomicOr(&s_scr[8 + (b >> 3)], lo << ((b & 7) * 4));
                    if (hi) atomicOr(&s_scr[16 + (b >> 3)], hi << ((b & 7) * 4));
                }
            }
        }
        __syncwarp();
        // The ranked draws (a few per step) are resolved by the lane that owns the point's mask word, all lanes at once.
        // A point sees the apples of the list plus this step's spawns BELOW it (the reference appends while it iterates in
        // point order), so the lanes iterate to the fixed point: every round only adds points the sequential loop adds too
        // (the thresholds grow with the count), and the lowest missing point of the sequential result passes in the next one.
        uint32_t lo_r = 0u, hi_r = 0u;                  // level bits of this lane's eligible points (bit j <-> j-th eligible point)
        if (ecnt) {
            const int w = eexcl >> 5;
            const uint32_t sh = (uint32_t)(eexcl & 31);
            lo_r = __funnelshift_r(s_scr[8 + w], w + 1 < 8 ? s_scr[8 + w + 1] : 0u, sh);
            hi_r = __funnelshift_r(s_scr[16 + w], w + 1 < 8 ? s_scr[16 + w + 1] : 0u, sh);
            if (ecnt < 32) { const uint32_t mk = (1u << ecnt) - 1u; lo_r &= mk; hi_r &= mk; }
        }
        uint32_t pending = lo_r | hi_r, mynew = 0u;
        s_scr[a] = 0u;                                  // points spawned in this step, by mask word (elig lives in a register)
        __syncwarp();
        bool go = __any_sync(FULLMASK, pending != 0u);
#pragma unroll 1
        while (go) {
            bool changed = false;
            uint32_t tmp = pending;
#pragma unroll 1
            while (tmp) {
                const int j = __ffs(tmp) - 1; tmp &= tmp - 1;
                const int bit = select_bit(elig, j), i = a * 32 + bit;
                const int lvl = (int)((lo_r >> j) & 1u) + 2 * (int)((hi_r >> j) & 1u);
                const uint32_t* nb = p.nbr_mask + (size_t)i * p.nwa;
                int num = 0;
#pragma unroll 1
                for (int q = 0; q < p.nwa; q++) {
                    const uint32_t below = q < a ? 0xFFFFFFFFu : (q == a ? (1u << bit) - 1u : 0u);
                    num += __popc(__ldg(nb + q) & (s_rec[FR_AM + q] | (s_scr[q] & below)));
                }
                if (min(num, 3) >= 4 - lvl) { pending &= ~(1u << j); mynew |= 1u << bit; changed = true; }
            }
            __syncwarp();
            if (changed) s_scr[a] = mynew;
            __syncwarp();
            go = __any_sync(FULLMASK, changed);
        }
        {   // the new apples join the list in point order
            const int scnt = __popc(mynew);
            const int sincl = oct_scan_incl(scnt, a);
            const int stot = __shfl_sync(FULLMASK, sincl, 7, 8);
            int lp = nA + sincl - scnt;
            uint32_t m = mynew;
#pragma unroll 1
            while (m) { const int bit = __ffs(m) - 1; m &= m - 1; s_al[lp++] = (uint8_t)(a * 32 + bit); }
            s_rec[FR_AM + a] |= mynew;
            nA += stot;
            a_chg = a_chg || stot != 0;
        }
    }
    __syncwarp();

    // ---- observations: closest apple / waste (cleanup), apples within the radius (harvest)
    uint32_t ar[2] = { 0x7F7F7F7Fu, 0x7F7F7F7Fu }, ac[2] = { 0x7F7F7F7Fu, 0x7F7F7F7Fu };
    {
        const uint32_t sh = 8u * (uint32_t)(a & 3);
        const bool lo4 = a < 4, on = a < n;
        const uint32_t rr = on ? (pos & 255u) : 0x7Fu, cc = on ? ((pos >> 8) & 255u) : 0x7Fu;
        ar[0] = oct_or(lo4 ? rr << sh : 0u); ar[1] = oct_or(lo4 ? 0u : rr << sh);
        ac[0] = oct_or(lo4 ? cc << sh : 0u); ac[1] = oct_or(lo4 ? 0u : cc << sh);
    }
    const uint32_t ca = oct_closest(s_al, nA, s_arc, ar[0], ar[1], ac[0], ac[1], n > 4, a);
    uint32_t cw = 0u; int close5 = 0;
    if (CLEANUP) cw = oct_closest(s_wl, nW, s_wrc, ar[0], ar[1], ac[0], ac[1], n > 4, a);
    else {
        const uint32_t* row = p.near5 + (size_t)feat_cell(p, pos) * p.nwa;
        for (int q = 0; q < p.nwa; q++) close5 += __popc(s_rec[FR_AM + q] & __ldg(row + q));
    }
    const uint32_t other = __shfl_sync(FULLMASK, pos, a == 0 ? (n > 1 ? 1 : 0) : 0, 8);       // compute_closest_pos quirk
    uint32_t cl_lo = 0u, cl_hi = 0u;                                       // cleaned_squares of every agent, one per byte
    if (CLEANUP) {
        cl_lo = oct_or(a < 4 ? (uint32_t)cleaned << (8 * a) : 0u);
        cl_hi = oct_or(a < 4 ? 0u : (uint32_t)cleaned << (8 * (a - 4)));
    }
    if (io.obs && active && a < n) {
        double v[FEAT_MAXF];
        v[0] = (double)(pos & 255u); v[1] = (double)((pos >> 8) & 255u); v[2] = (double)((pos >> 16) & 3u);
        v[3] = (double)(other & 255u); v[4] = (double)((other >> 8) & 255u); v[5] = (double)((other >> 16) & 3u);
        v[6] = (double)(ca >> 8); v[7] = (double)(ca & 255u);
        if (CLEANUP) {
            v[8] = (double)(cw >> 8); v[9] = (double)(cw & 255u); v[10] = (double)nA; v[11] = (double)nW;
#pragma unroll
            for (int i = 0; i < SSD_MAXN; i++) v[12 + i] = (double)(((i < 4 ? cl_lo : cl_hi) >> (8 * (i & 3))) & 255u);
#pragma unroll
            for (int i = 20; i < FEAT_MAXF; i++) v[i] = 0.0;
        } else {
            v[8] = (double)close5; v[9] = (double)nA;
#pragma unroll
            for (int i = 10; i < FEAT_MAXF; i++) v[i] = 0.0;
        }
        const int F = p.F;
        if constexpr (FORM == OBS_F64) {
            double* o = static_cast<double*>(io.obs) + ((size_t)env * n + a) * F;
            if ((F & 1) == 0) {                                            // rows are 16-byte aligned iff F is even
#pragma unroll
                for (int k = 0; k < FEAT_MAXF; k += 2) if (k < F) reinterpret_cast<double2*>(o)[k >> 1] = make_double2(v[k], v[k + 1]);
            } else {
#pragma unroll
                for (int k = 0; k < FEAT_MAXF; k++) if (k < F) o[k] = v[k];
            }
        } else {
            const bool con = p.contract != SSD_CONTRACT_NONE;
            typedef typename PolicyElem<FORM>::T T;
            feat_policy_row(static_cast<T*>(io.obs) + ((size_t)env * n + a) * (F + (con ? 2 : 0)), v, F, con, theta);
        }
    }

    // ---- rewards, contract transfers (contract_list.py:22-27,45-54), redistribution (two_stage_train.py:71-92)
    const int t_new = doreset ? 0 : (int)s_rec[FR_T] + 1;
    if (!RESET_ONLY) {
        double rew = (double)reward, tr = 0.0, total = 0.0;
        if (stepping && a < n) {
            if (p.contract == SSD_CONTRACT_CLEANUP) tr = __dmul_rn(-theta, (double)cleaned);
            else if (p.contract == SSD_CONTRACT_HARVEST_LOCAL) tr = (close5 < 4 && eaten_close > 0) ? theta : 0.0;
        }
        // (all transfers +-0: the loop below would leave every reward as it is — x - +-0 = x, x + +-0 / (n - 1) = x for x >= +0)
        if (p.contract != SSD_CONTRACT_NONE && __any_sync(FULLMASK, tr != 0.0)) {
            const double share = __ddiv_rn(tr, (double)(n - 1));
#pragma unroll 1
            for (int i = 0; i < n; i++) {
                const double tri = shfl_f64(tr, i), shi = shfl_f64(share, i);
                total = __dadd_rn(total, tri);
                rew = i == a ? __dsub_rn(rew, tri) : __dadd_rn(rew, shi);
            }
        }
        const int raw = oct_sum(reward), n_eaten = oct_sum(eaten), n_close = oct_sum(eaten_close);
        if (active && a < n) {
            const size_t o = (size_t)env * n + a, so = (size_t)a * p.E + env;
            if (io.rew) io.rew[o] = rew;
            if (io.base_rew) io.base_rew[o] = (double)reward;
            if (io.transfers) io.transfers[o] = tr;
            if (io.info) reinterpret_cast<uint32_t*>(io.info)[o] = CLEANUP ? (uint32_t)cleaned : ((uint32_t)eaten | ((uint32_t)eaten_close << 8));
            // episode accumulators as fire-and-forget reductions (one add per address and step: a float64 RED rounds
            // exactly like `x = x + y`)
            if (reward) {
                red_add(p.sum_raw + so, (uint32_t)reward);
                red_add(reinterpret_cast<long long*>(p.tsum_raw + so), (long long)((unsigned long long)(t_new - 1) * (unsigned long long)reward));
            }
            if (rew != 0.0) {
                red_add(p.sum_tr + so, rew);
                red_add(p.tsum_tr + so, __dmul_rn((double)(t_new - 1), rew));
            }
        }
        if (stepping && a == 0) {
            if (dirt) red_add(p.metrics + (size_t)0 * p.E + env, (double)dirt);
            if (raw) red_add(p.metrics + (size_t)1 * p.E + env, (double)raw);
            if (total != 0.0) red_add(p.metrics + (size_t)2 * p.E + env, total);
            if (n_eaten) red_add(p.metrics + (size_t)3 * p.E + env, (double)n_eaten);
            if (n_close) red_add(p.metrics + (size_t)4 * p.E + env, (double)n_close);
        }
        if (active && a == 0 && io.done) io.done[env] = (stepping && t_new == p.horizon) ? 1 : 0;
        if (io.c_rew8) {                                                   // the pipelined host path's lossless result block
            int vi = 0;
            const bool mine = active && a < n, fits = reward_fits_i8(rew, vi);
            if (mine) io.c_rew8[(size_t)env * n + a] = fits ? (int8_t)vi : (int8_t)0;
            if (active && a == 0) io.c_done[env] = (stepping && t_new == p.horizon) ? 1 : 0;
            const uint32_t badm = __ballot_sync(FULLMASK, mine && !fits);
            if (badm) {                                                    // one record per env with such a reward, one atomic per warp
                const bool need = ((badm >> obase) & 0xFFu) != 0u;
                const uint32_t needm = __ballot_sync(FULLMASK, need && a == 0);
                const int leader = __ffs(needm) - 1;
                uint32_t base = 0u;
                if (lane == leader) base = atomicAdd(io.c_count, (uint32_t)__popc(needm));
                base = __shfl_sync(FULLMASK, base, leader);
                if (need) {
                    uint8_t* rec = io.c_rec + (size_t)(base + (uint32_t)__popc(needm & ((1u << obase) - 1u))) * (size_t)(8 + 8 * n);
                    if (a == 0) { reinterpret_cast<int32_t*>(rec)[0] = env; reinterpret_cast<int32_t*>(rec)[1] = 0; }
                    if (a < n) reinterpret_cast<double*>(rec + 8)[a] = rew;
                }
            }
        }
    }

    // ---- state out
    __syncwarp();
    if (active) {
        if (a < n) s_rec[FR_AGENT + a] = pos;
        if (a == 0) {
            s_rec[FR_NA] = (uint32_t)nA; s_rec[FR_NW] = (uint32_t)nW; s_rec[FR_T] = (uint32_t)t_new;
            s_rec[FR_EPISODE] = episode | 0x80000000u;
            s_rec[FR_THETA] = (uint32_t)__double2loint(theta); s_rec[FR_THETA + 1] = (uint32_t)__double2hiint(theta);
        }
    }
    __syncwarp();
    if (active) {
        *reinterpret_cast<uint4*>(grec + 4 * a) = *reinterpret_cast<const uint4*>(s_rec + 4 * a);
        if (a_chg) {
            if (a * 16 < nA) *reinterpret_cast<uint4*>(glist + 16 * a) = *reinterpret_cast<const uint4*>(s_al + 16 * a);
            if ((a + 8) * 16 < nA) *reinterpret_cast<uint4*>(glist + 16 * (a + 8)) = *reinterpret_cast<const uint4*>(s_al + 16 * (a + 8));
        }
        if (w_chg) {
            if (a * 16 < nW) *reinterpret_cast<uint4*>(glist + p.LA + 16 * a) = *reinterpret_cast<const uint4*>(s_wl + 16 * a);
            if ((a + 8) * 16 < nW) *reinterpret_cast<uint4*>(glist + p.LA + 16 * (a + 8)) = *reinterpret_cast<const uint4*>(s_wl + 16 * (a + 8));
        }
    }
    __syncwarp();                                    // the octet's shared state is rewritten by the next round
    }
}

// metrics [E][40]: dirt, raw, transfers, apples, low_density, 0, 0, 0, sum_raw[8], tsum_raw[8], sum_tr[8], tsum_tr[8]
__global__ void feat_get_metrics_kernel(const FeatParams p, double* out)
{
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.E) return;
    double* o = out + (size_t)env * 40;
    for (int q = 0; q < 40; q++) o[q] = feat_metric(p.metrics, p.sum_raw, p.tsum_raw, p.sum_tr, p.tsum_tr, p.E, p.n, env, q);
}
// pos int32 [E][n][2], ori int32 [E][n], cells u8 [E][H][W] (1 apple, 2 waste), theta f64 [E], t int32 [E]
__global__ void feat_get_state_kernel(const FeatParams p, int32_t* pos, int32_t* ori, uint8_t* cells, double* theta, int32_t* t)
{
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.E) return;
    const uint32_t* rec = p.rec + (size_t)env * FR_WORDS;
    for (int a = 0; a < p.n; a++) {
        const uint32_t v = rec[FR_AGENT + a];
        if (pos) { pos[((size_t)env * p.n + a) * 2] = (int)(v & 255u); pos[((size_t)env * p.n + a) * 2 + 1] = (int)((v >> 8) & 255u); }
        if (ori) ori[(size_t)env * p.n + a] = (int)((v >> 16) & 3u);
    }
    if (cells) {
        uint8_t* c = cells + (size_t)env * p.H * p.W;
        for (int i = 0; i < p.H * p.W; i++) c[i] = 0;
        // the lists are the state of record (the masks mirror them)
        const uint8_t* al = p.lists + (size_t)env * p.LS; const uint8_t* wl = al + p.LA;
        for (int i = 0; i < (int)rec[FR_NA]; i++) { const uint32_t rc = p.apple_rc[al[i]]; c[(rc >> 8) * p.W + (rc & 255u)] = 1; }
        for (int i = 0; i < (int)rec[FR_NW]; i++) { const uint32_t rc = p.waste_rc[wl[i]]; c[(rc >> 8) * p.W + (rc & 255u)] = 2; }
    }
    if (theta) theta[env] = *reinterpret_cast<const double*>(rec + FR_THETA);
    if (t) t[env] = (int)rec[FR_T];
}
__global__ void feat_random_actions_kernel(const FeatParams p, uint32_t step_index, uint32_t* counter, int num_actions, uint8_t* actions)
{
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (counter) step_index = *reinterpret_cast<volatile uint32_t*>(counter);
    if (env < p.E) {
        const uint32_t env_id = p.first_env_id + (uint32_t)env;
        for (int b = 0; b * 4 < p.n; b++) {
            Philox4 q = philox4x32_10((uint32_t)b, SITE_ACTIONS, step_index, 0u, p.seed, env_id);
            uint32_t w[4] = { q.x, q.y, q.z, q.w };
            for (int j = 0; j < 4 && b * 4 + j < p.n; j++)
                actions[(size_t)env * p.n + b * 4 + j] = (uint8_t)(((uint64_t)w[j] * (uint32_t)num_actions) >> 32);
        }
    }
    if (counter) counter_finish(counter, step_index);
}
