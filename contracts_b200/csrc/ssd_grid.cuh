// ssd_grid.cuh — sm_100a kernels for the gridworld envs (cleanup_new / harvest_new): shared definitions, the spawn
// and observation building blocks, and the reset kernel.  The step kernels are in ssd_grid2.cuh.
//
// State (DESIGN.md §3).  Everything that changes in a map is an apple on an apple point or waste on a waste point, so
// an env's dynamic map state is two BITMASKS (bit j = point j of the canonical row-major point list holds an apple /
// waste), kept in the first 128-byte line of the env's record together with the agents, t, episode, theta, flags and
// #waste.  Walls, river, stream and the point lists are static per handle.  The step's decision logic works on that
// one line + static tables; the observe kernel keeps a padded uint8 tile T of the map (7 cells of C_OUTSIDE border =
// the view radius) AND its transpose T2 per warp in shared memory and only rewrites the dynamic cells for each env.
//
// Reference behaviour restated here (paths relative to the reference root):
//   environments/map_env.py   step :216-304, update_moves :483-676, update_custom_moves :678-693,
//                             update_map_fire :721-814, color_view :397-411, reset :306-342,
//                             spawn_point :816-827, spawn_rotation :829-832
//   environments/cleanup_new.py  step :211-267, custom_action :269-292, spawn_apples_and_waste :322-349,
//                             compute_probabilities :351-368, custom_reset :171-189
//   environments/harvest_new.py  step :181-239, spawn_apples :284-317, count_apples_in_radius :326-336
//   contract/contract_list.py :22-27, :45-54 ; environments/two_stage_train.py :62-121, :159-187
#pragma once
#include "ssd_common.cuh"

// Observation form written by the observe / reset kernels: OBS_U8 = the uint8 windows [E][n][15][15][3]; 1 + SSD_POLICY_* =
// the policy's image tensor T [E n][3][15][15] (ssd_set_policy_output), the values ssd_policy_inputs would make of the windows.
#define OBS_U8 0
template <int FORM> struct ObsForm : PolicyElem<FORM> {};
template <> struct ObsForm<OBS_U8> { typedef uint8_t T; };

#ifndef GRID_WARPS
#define GRID_WARPS 8
#endif
#define GRID_THREADS (GRID_WARPS * 32)
#define SCRATCH_DRAWS 256               // u32 draws per warp scratch
#define SCRATCH_KEYS 256                // u32 shuffle keys per warp scratch
#define MAX_POINT_ROUNDS 8              // point lists are handled 32 per round => <= 256 points, 8 mask words
#define FULL 0xffffffffu

// record layout.  Bytes 0..127 are the HOT line (one coalesced 128-byte access per env), the episode accumulators follow.
#define RO_AGENTS 0        // u32[8]: row | col << 8 | ori << 16
#define RO_T 32            // i32
#define RO_EPISODE 36      // u32
#define RO_THETA 40        // f64
#define RO_FLAGS 48        // u32
#define RO_HCOUNT 52       // u32 (#waste cells, cleanup)
#define RO_AMASK 64        // u32[8]: apple bitmask over the apple point list
#define RO_WMASK 96        // u32[8]: waste bitmask over the waste point list (cleanup)
#define RO_HOT 128
#define RO_APPLES 128      // u32 total_apples_eaten
#define RO_LOWDENS 132     // u32 low_density_apples_eaten
#define RO_DIRT 136        // u32 dirt_cleaned
#define RO_TRANSFERS 144   // f64 metrics['transfers']
#define RO_SUM_TR 152      // f64[8]
#define RO_TSUM_TR 216     // f64[8]
#define RO_TSUM_RAW 280    // i64[8]
#define RO_SUM_RAW 344     // i32[8]
#define RO_AGENT_A 376     // u32[8] waste_cleaned | apples_consumed
#define RO_AGENT_B 408     // u32[8] close_apples_consumed
#define RO_SIZE 440
// extension, present only when rewards are shaped (use_collective_reward / inequity_averse_reward,
// map_env.py:289-301): the env rewards are float64 then, so their episode sums are too
#define RO_XSUM 440        // f64[8] sum_t r
#define RO_XTSUM 504       // f64[8] sum_t t * r
#define RO_XRAW 568        // f64 metrics['raw_env_rewards']
#define RO_XSIZE 576
#define RM_COLLECTIVE 1
#define RM_INEQUITY 2

// static per-cell word of the logic kernel (cell_info[row * Wp + col])
#define CI_IDX 0xFFu       // index in the apple / waste point list
#define CI_WALL 0x2000u
#define CI_APPLE 0x4000u   // the cell is an apple point
#define CI_WASTE 0x8000u   // the cell is a waste point

struct GridParams {
    int E, n, H, W, Wp, S, TH;
    int map_bytes;           // H * Wp rounded up to 16: size of a compact map (beam overlay, views, get / set state)
    int rec_stride;          // bytes per env record (512, or 640 when rewards are shaped)
    int hdr_bytes;           // RO_SIZE, or RO_XSIZE when rewards are shaped
    int mw;                  // mask words per point list in use (4 or 8)
    int reward_mode;         // RM_* bits
    double alpha, beta;      // inequity aversion weights (map_env.py:71-72)
    // shared memory of the observe / reset kernels: CTA tables first, then per warp [T | T2 | stage (obs staging, aliased
    // by the spawn scratch) | misc]
    int sm_thr, sm_won, sm_apple_rc, sm_waste_rc, sm_warp0;
    int tile_r16, stage_r16, tile2_off, g2_stage, g2_misc, g2_warp_bytes, g2_smem_bytes;
    int S2;                  // transposed tile: row stride 8 + Hp + 8
    int obs_items;           // ceil(15 n / 4): 4-row (180 B) work items of the observation gather
    int kind, contract, horizon;
    int n_apple, n_waste, n_spawn, n_waste_start, F;
    uint32_t seed, first_env_id;
    double theta_low, theta_high, null_prob;
    uint32_t thr_harvest[4]; // SPAWN_PROB thresholds (harvest_new.py:34)
    uint32_t thr_waste;      // wasteSpawnProbability = 0.5
    uint32_t s_magic;        // ceil(2^32 / S): row = umulhi(offset, s_magic)
    const uint32_t* pal;     // [16] packed RGB per tile byte value (cell codes 0..5, agents 6..13, outside 15)
    const uint32_t* apple_pt;    // [256] offset in T | offset in T2 << 16 of each apple point (0 beyond the list)
    const uint32_t* waste_pt;    // [256]
    const uint16_t* spawn_pts;   // offsets in T
    const uint16_t* apple_rc;    // row << 8 | col of each apple point (feature_obs only)
    const uint16_t* waste_rc;
    const uint32_t* thr_apple;   // [n_waste + 1] apple spawn threshold by #waste
    const uint8_t* waste_on;     // [n_waste + 1]
    const uint8_t* tile0;        // [tile_r16 + tile2 bytes]: static T | T2 with every dynamic cell OFF (apple point empty, waste point river)
    const uint16_t* cell_info;   // [H * Wp] CI_* words (logic kernel)
    const uint4* beam_tab;       // [H * Wp][4 orientations][2]: a beam's static part — .x of the first word: wall mask of the 15 ray
                                 // cells (RAY_* bit layout, cells outside the map are walls); bytes 4..18: the cells' waste-point
                                 // indices (0xFF: not a waste point), order left ray 0-4, centre 0-4, right 0-4
    const uint8_t* base_map;     // [map_bytes] compact static codes, dynamic cells OFF (views, get / set state)
    const uint16_t* apple_c;     // compact offsets (row * Wp + col) of the points (views, get / set state)
    const uint16_t* waste_c;
    uint32_t reset_amask[MAX_POINT_ROUNDS];   // dynamic state of the reset map (harvest: every point holds an apple;
    uint32_t reset_wmask[MAX_POINT_ROUNDS];   // cleanup: the 'H' cells), before the reset-time spawn
    uint8_t* state;
    uint8_t* beam;               // optional [E][map_bytes]: beam_pos of the last step as a char overlay (render only)
    double* stats;               // optional [8]: ssd_set_episode_stats accumulator (added to by the reset kernel)
    EpisodeLog elog;             // optional: ssd_set_episode_log ring buffer (appended to by the reset kernel)
    uint32_t* obs_ctr;           // [2] observe kernel: next env of the dynamically scheduled tail, CTAs finished
    int obs_static_iters;        // observe kernel: iterations every warp takes from the static grid-stride schedule
};

// use_collective_reward / inequity_averse_reward (map_env.py:289-301): the shaped reward of agent a from the
// integer env rewards.  Differences and their partial sums are exact integers; alpha * sum, beta * sum, their
// sum, the division by (num_agents - 1) and the subtraction are float64, in that order.  (Scalar arguments and
// no local arrays: a GridParams reference into a non-inlined function would copy the kernel parameters to the stack.)
__device__ __forceinline__ double inequity_term(int ra, int sp, int sn, double alpha, double beta, int n)
{
    const double dis = __dmul_rn(alpha, (double)sp), adv = __dmul_rn(beta, (double)sn);
    return __dsub_rn((double)ra, __ddiv_rn(__dadd_rn(dis, adv), (double)(n - 1)));
}
// Element q of the env's ssd_get_metrics row (SSD_METRIC_STRIDE doubles, include/ssd_b200.h) from its record: what
// ssd_get_metrics writes and what the reset kernel hands to the episode log.
__device__ __forceinline__ double grid_metric(const GridParams& p, const uint8_t* hdr, int q)
{
    if (q >= 8) {
        const int a = q & 7;
        switch (q >> 3) {
        case 1: return (double)reinterpret_cast<const uint32_t*>(hdr + RO_AGENT_A)[a];
        case 2: return (double)reinterpret_cast<const uint32_t*>(hdr + RO_AGENT_B)[a];
        case 3: return p.reward_mode ? reinterpret_cast<const double*>(hdr + RO_XSUM)[a]        // shaped rewards: float64 sums
                                     : (double)reinterpret_cast<const int*>(hdr + RO_SUM_RAW)[a];
        case 4: return p.reward_mode ? reinterpret_cast<const double*>(hdr + RO_XTSUM)[a]
                                     : (double)reinterpret_cast<const long long*>(hdr + RO_TSUM_RAW)[a];
        case 5: return reinterpret_cast<const double*>(hdr + RO_SUM_TR)[a];
        default: return reinterpret_cast<const double*>(hdr + RO_TSUM_TR)[a];
        }
    }
    switch (q) {
    case 0: return (double)*reinterpret_cast<const uint32_t*>(hdr + RO_APPLES);
    case 1: return (double)*reinterpret_cast<const uint32_t*>(hdr + RO_LOWDENS);
    case 2: {
        if (p.reward_mode) return *reinterpret_cast<const double*>(hdr + RO_XRAW);
        double raw = 0;
#pragma unroll 1
        for (int a = 0; a < SSD_MAXN; a++) raw += (double)reinterpret_cast<const int*>(hdr + RO_SUM_RAW)[a];
        return raw;
    }
    case 3: return *reinterpret_cast<const double*>(hdr + RO_TRANSFERS);
    case 4: return (double)*reinterpret_cast<const uint32_t*>(hdr + RO_DIRT);
    case 5: return (double)((*reinterpret_cast<const uint32_t*>(hdr + RO_FLAGS) >> RF_ERR_SHIFT) & 0xFFFFu);
    default: return 0.0;
    }
}

// thread per env: the int16 rewards sit in the RS_* words rsp[j * rstride] (bits 16-31)
__device__ __noinline__ double shaped_reward(int mode, double alpha, double beta, int n, const uint32_t* rsp, int rstride, int a)
{
    int coll = 0;
    for (int j = 0; j < n; j++) coll += (int)rsp[j * rstride] >> 16;
    const bool collective = mode & RM_COLLECTIVE;
    const int ra = collective ? coll : ((int)rsp[a * rstride] >> 16);
    if (!(mode & RM_INEQUITY)) return (double)ra;
    int sp = 0, sn = 0;
    for (int j = 0; j < n; j++) {
        const int d = (collective ? coll : ((int)rsp[j * rstride] >> 16)) - ra;
        if (d > 0) sp += d; else sn += d;
    }
    return inequity_term(ra, sp, sn, alpha, beta, n);
}
// warp per env, lane = agent (every lane calls)
__device__ __noinline__ double shaped_reward_warp(int mode, double alpha, double beta, int n, int reward)
{
    int coll = 0;
    for (int j = 0; j < n; j++) coll += __shfl_sync(FULL, reward, j);
    const bool collective = mode & RM_COLLECTIVE;
    const int ra = collective ? coll : reward;
    int sp = 0, sn = 0;
    for (int j = 0; j < n; j++) {
        const int d = (collective ? coll : __shfl_sync(FULL, reward, j)) - ra;
        if (d > 0) sp += d; else sn += d;
    }
    return (mode & RM_INEQUITY) ? inequity_term(ra, sp, sn, alpha, beta, n) : (double)ra;
}

// per-warp misc area
#define MISC_VDESC 0        // int4[8]: per-agent view descriptor {offset of out[0][0], pixel step, row step, 0}
#define MISC_BYTES 128

struct StepIO {
    const uint8_t* actions;
    uint8_t* obs; long long obs_stride;
    double* rew; double* base_rew; double* transfers;
    uint8_t* info; double* feat; uint8_t* done;
    // compact result block of ssd_step_host_async (all null otherwise): int8 rewards, dones, and records
    // { int32 env; int32 0; double rew[n] } for the envs whose rewards are not all integers in [-127, 127]
    int8_t* c_rew8; uint8_t* c_done; uint32_t* c_count; uint8_t* c_rec;
    // auto_reset: envs that finish in this step (t == horizon) are reset by the step itself — their observation becomes
    // the reset observation — and, when neg_prop / neg_acc are given, negotiate their next contract (two_stage_train.py:266-281)
    int auto_reset;
    const double* neg_prop; const double* neg_acc; uint8_t* neg_dec;
};

// is `r` exactly an integer in [-127, 127]?  (bit pattern compared: -0.0 is not)
__device__ __forceinline__ bool reward_fits_i8(double r, int& v)
{
    v = __double2int_rn(r);
    return v >= -127 && v <= 127 && __double_as_longlong((double)v) == __double_as_longlong(r);
}
// slot of this thread's record in the compact block: one atomic per group of converged threads
__device__ __forceinline__ uint32_t compact_slot(uint32_t* count)
{
    const unsigned am = __activemask();
    const int lane = threadIdx.x & 31, leader = __ffs(am) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(count, (uint32_t)__popc(am));
    base = __shfl_sync(am, base, leader);
    return base + (uint32_t)__popc(am & ((1u << lane) - 1u));
}

struct EnvRng { uint32_t seed, env_id, episode, t; };

// per-CTA copies of the static tables in shared memory
struct SharedTables {
    const uint32_t* pal; const uint32_t* thr_apple; const uint8_t* waste_on;
    const uint16_t* apple_rc; const uint16_t* waste_rc;
};

__device__ __forceinline__ uint32_t lanemask_lt(int lane) { return (1u << lane) - 1u; }
__device__ __forceinline__ int dir_delta(int ori, int S)
{
    return ori == ORI_UP ? -S : (ori == ORI_RIGHT ? 1 : (ori == ORI_DOWN ? S : -1));
}

// ---------------------------------------------------------------------------------------------
// bulk-copy (TMA) + mbarrier primitives.  Bulk async-groups are per thread: lane 0 issues and waits.
__device__ __forceinline__ uint32_t smem_u32(const void* ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }
__device__ __forceinline__ void mbar_init(void* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(void* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared, completion signalled on `bar` (expect_tx armed by the same lane)
__device__ __forceinline__ void bulk_load(void* sdst, const void* gsrc, uint32_t bytes, void* bar)
{
    const uint32_t b = smem_u32(bar);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(b), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(sdst)), "l"(gsrc), "r"(bytes), "r"(b) : "memory");
}
// shared -> global, one bulk group per call
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int PENDING>
__device__ __forceinline__ void bulk_wait_read()
{
    asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(PENDING) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Programmatic dependent launch (PDL): a kernel launched with the programmatic-serialization attribute may become resident
// while its predecessor in the stream still runs; pdl_wait() blocks until the predecessor has completed and its writes are
// visible, so everything before it (table loads, tile set-up) overlaps the predecessor's tail.  pdl_launch_dependents() in
// the predecessor lets the dependent grid be scheduled as soon as every predecessor CTA has issued it (or exited).
// Both are no-ops for a kernel that was launched normally.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }

// One out-of-line copy of the 10 Philox rounds for the step kernel (the inlined form is ~80
// instructions per call site; the hot loop has to fit the instruction cache).
__device__ __noinline__ uint4 draw_block_ool(uint32_t seed, uint32_t env_id, uint32_t episode, uint32_t t,
                                             uint32_t site_call, uint32_t block)
{
    Philox4 q = philox4x32_10(block, site_call, t, episode, seed, env_id);
    return make_uint4(q.x, q.y, q.z, q.w);
}
__device__ __forceinline__ uint32_t draw_u32_ool(const EnvRng& g, uint32_t t, uint32_t site, uint32_t idx)
{
    uint4 q = draw_block_ool(g.seed, g.env_id, g.episode, t, site, idx >> 2);
    const uint32_t w = idx & 3u;
    return w == 0 ? q.x : (w == 1 ? q.y : (w == 2 ? q.z : q.w));
}

// Two Philox blocks of the same (env, episode, t) with interleaved rounds: two independent dependency chains instead of
// two calls back to back (the spawn is latency-bound).  Results go to shared memory; a null pointer skips the store.
__device__ __noinline__ void draw_blocks2_ool(uint32_t seed, uint32_t env_id, uint32_t episode, uint32_t t,
                                              uint32_t site_a, uint32_t block_a, uint4* dst_a,
                                              uint32_t site_b, uint32_t block_b, uint4* dst_b)
{
    uint32_t a0 = block_a, a1 = site_a, a2 = t, a3 = episode, b0 = block_b, b1 = site_b, b2 = t, b3 = episode;
    uint32_t k0 = seed, k1 = env_id;
#pragma unroll
    for (int i = 0; i < 10; i++) {
        const uint32_t ah0 = __umulhi(0xD2511F53u, a0), al0 = 0xD2511F53u * a0, ah1 = __umulhi(0xCD9E8D57u, a2), al1 = 0xCD9E8D57u * a2;
        const uint32_t bh0 = __umulhi(0xD2511F53u, b0), bl0 = 0xD2511F53u * b0, bh1 = __umulhi(0xCD9E8D57u, b2), bl1 = 0xCD9E8D57u * b2;
        const uint32_t na0 = ah1 ^ a1 ^ k0, na2 = ah0 ^ a3 ^ k1, nb0 = bh1 ^ b1 ^ k0, nb2 = bh0 ^ b3 ^ k1;
        a0 = na0; a1 = al1; a2 = na2; a3 = al0;
        b0 = nb0; b1 = bl1; b2 = nb2; b3 = bl0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    if (dst_a) *dst_a = make_uint4(a0, a1, a2, a3);
    if (dst_b) *dst_b = make_uint4(b0, b1, b2, b3);
}

// ---------------------------------------------------------------------------------------------
// The literal ordering of the reference (rare: some movers share a target or a real move targets an
// occupied cell).  Out of line: it is cold and would otherwise bloat the hot loop's instruction
// footprint.  Returns err << 16 | new tile offset.
__device__ __noinline__ uint32_t resolve_moves_slow(int lane, int n, uint32_t seed, uint32_t env_id, uint32_t episode,
                                                    uint32_t t, int ao, bool has_move, int tgt, unsigned movers,
                                                    bool contested)
{
    const bool act_lane = lane < n;
    uint32_t err = 0;
    // shuffled priority (map_env.py:545-547): key of list position m = rank among movers
    uint32_t key = 0xFFFFFFFFu;
    if (has_move) key = draw_u32(seed, env_id, episode, t, SITE_MOVE_ORDER, 0,
                                 (uint32_t)__popc(movers & lanemask_lt(lane)));
    int cur_mv = tgt;                               // agent_moves[agent]
    // contested cells in lexicographic (row, col) order == increasing tile offset (np.unique, :548)
    unsigned remaining = __ballot_sync(FULL, contested);
    while (remaining) {
        uint32_t v = ((remaining >> lane) & 1u) ? (uint32_t)tgt : 0xFFFFFFFFu;
        int cmin = (int)__reduce_min_sync(FULL, v);
        bool in_group = has_move && tgt == cmin;
        unsigned group = __ballot_sync(FULL, in_group);
        remaining &= ~group;
        unsigned occm = __ballot_sync(FULL, act_lane && ao == cmin);   // live positions (:574)
        bool cell_free = true;
        if (occm) {
            int occ = 31 - __clz(occm);             // agent_by_pos: the highest index wins duplicates
            bool occ_has = (movers >> occ) & 1u;
            int occ_mv = __shfl_sync(FULL, cur_mv, occ);
            unsigned swapm = __ballot_sync(FULL, in_group && ao == occ_mv);
            if (!occ_has || occ_mv == cmin) cell_free = false;      // conditions (1),(2) :585-595
            else if (swapm) cell_free = false;                      // condition (3) :599-605
        }
        if (cell_free) {
            uint32_t kmin = __reduce_min_sync(FULL, in_group ? key : 0xFFFFFFFFu);
            unsigned cand = __ballot_sync(FULL, in_group && key == kmin);
            if (lane == __ffs(cand) - 1) ao = cmin;                 // first contestant of the shuffled list (:610)
        }
        if (in_group) cur_mv = ao;                                   // :620-621
    }
    // remaining moves, multi-pass (:624-676)
    unsigned live = movers;
    while (live) {
        const int snap = ao;                        // agent_by_pos snapshot (:625)
        const unsigned copy = live;
        const int num = __popc(live);
        for (int i = 0; i < n; i++) {
            if (!((copy >> i) & 1u) || !((live >> i) & 1u)) continue;
            int mv_i = __shfl_sync(FULL, cur_mv, i);
            int pos_i = __shfl_sync(FULL, ao, i);
            unsigned occ_live = __ballot_sync(FULL, act_lane && ao == mv_i);
            if (occ_live) {
                unsigned snap_b = __ballot_sync(FULL, act_lane && snap == mv_i);
                if (!snap_b) { err |= 2; live &= ~(1u << i); continue; }      // KeyError in the reference
                int occ = 31 - __clz(snap_b);
                int pos_occ = __shfl_sync(FULL, ao, occ);
                int mv_occ_raw = __shfl_sync(FULL, cur_mv, occ);
                int mv_occ = ((live >> occ) & 1u) ? mv_occ_raw : pos_occ;      // agent_moves.get(occ, pos)
                if (occ == i) live &= ~(1u << i);
                else if (!((copy >> occ) & 1u) || pos_occ == mv_occ) live &= ~(1u << i);
                else if (mv_occ == pos_i && mv_i == pos_occ) live &= ~((1u << i) | (1u << occ));
            } else {
                if (lane == i) ao = mv_i;
                live &= ~(1u << i);
            }
        }
        if (__popc(live) == num) {                  // no progress: move everyone left (:673-676)
            if ((live >> lane) & 1u) ao = cur_mv;
            break;
        }
    }
    return (err << 16) | (uint32_t)ao;
}

// ---------------------------------------------------------------------------------------------
// Per-lane point registers: lane l owns points l, l + 32, ... of each list.  pt[q] = offset in T | offset in T2 << 16,
// both relative to the warp's tile base (T2 follows T).  Slots beyond a list point at spare sink bytes behind T / T2, so
// the dynamic-cell rewrite needs no bounds tests.
template <int MW>
struct PointRegs { uint32_t a[MW], w[MW]; };
template <int MW>
__device__ __forceinline__ PointRegs<MW> load_point_regs(const GridParams& p, int lane)
{
    PointRegs<MW> r;
#pragma unroll
    for (int q = 0; q < MW; q++) { r.a[q] = __ldg(p.apple_pt + lane + 32 * q); r.w[q] = __ldg(p.waste_pt + lane + 32 * q); }
    return r;
}
// bits of round q that belong to the list (point index < count)
__device__ __forceinline__ uint32_t round_valid(int count, int q)
{
    const int left = count - 32 * q;
    return left >= 32 ? 0xFFFFFFFFu : (left <= 0 ? 0u : ((1u << left) - 1u));
}
// write a dynamic cell into T and (when kept) T2
__device__ __forceinline__ void put_cell(uint8_t* tile, bool has2, uint32_t pt, uint32_t code)
{
    tile[pt & 0xFFFFu] = (uint8_t)code;
    if (has2) tile[pt >> 16] = (uint8_t)code;
}

// ---------------------------------------------------------------------------------------------
// cleanup spawn (cleanup_new.py:322-349).  Occupancy bits of the agents' cells must be set in T.  `t` = 0 at reset.
// am / wm: the env's apple / waste masks (warp-uniform, updated); hcount: #waste cells (updated).  Returns whether
// anything spawned.
__device__ __forceinline__ bool cleanup_spawn_active(const SharedTables& tb, int hcount)
{
    return tb.thr_apple[hcount] != 0 || tb.waste_on[hcount] != 0;
}
template <int MW>
__device__ __forceinline__ bool cleanup_spawn(const GridParams& p, const SharedTables& tb, int lane, uint8_t* tile, bool tile2,
                                              uint32_t* scratch, const EnvRng& g, uint32_t t, int& hcount,
                                              const PointRegs<MW>& pr, uint32_t (&am)[MW], uint32_t (&wm)[MW])
{
    const uint32_t thrA = tb.thr_apple[hcount];
    const bool waste_on = tb.waste_on[hcount] != 0;
    if (thrA == 0 && !waste_on) return false;
    uint32_t* draws = scratch;
    uint32_t* keys = scratch + SCRATCH_DRAWS;
    // apples: eligible = no agent there and not already 'A'; draw index = rank among eligible (:328-335)
    unsigned eligm[MW];
    int M = 0;
#pragma unroll
    for (int q = 0; q < MW; q++) {
        eligm[q] = 0;
        if (q * 32 < p.n_apple) {
            const bool occ = (tile[pr.a[q] & 0xFFFFu] & OCC_BIT) != 0;            // beyond the list: offset 0, a border cell
            eligm[q] = ~am[q] & round_valid(p.n_apple, q) & ~__ballot_sync(FULL, occ);
            M += __popc(eligm[q]);
        }
    }
    // waste candidates = non-'H' cells of waste_points (apple points and waste points are disjoint, so the apple
    // spawns below cannot change them)
    unsigned candm[MW];
    int C = 0;
#pragma unroll
    for (int q = 0; q < MW; q++) {
        candm[q] = waste_on ? (~wm[q] & round_valid(p.n_waste, q)) : 0u;
        C += __popc(candm[q]);
    }
    // one Philox pass for everything this spawn can need: the apple draws [0, M), the first waste draws [M, M + wfirst)
    // (the waste scan stops at its first success, p = 0.5) and the shuffle keys of the waste points
    const int wfirst = C > 0 ? min(min(C, 8), SCRATCH_DRAWS - M) : 0;
    const int nblk = (thrA || wfirst) ? (M + wfirst + 3) >> 2 : 0;
    const int nkblk = C > 0 ? (p.n_waste + 3) >> 2 : 0;
    for (int bl = lane; __any_sync(FULL, bl < nblk || bl < nkblk); bl += 32)
        draw_blocks2_ool(g.seed, g.env_id, g.episode, t,
                         SITE_SPAWN_DRAWS, (uint32_t)bl, bl < nblk ? reinterpret_cast<uint4*>(draws) + bl : nullptr,
                         SITE_WASTE_ORDER, (uint32_t)bl, bl < nkblk ? reinterpret_cast<uint4*>(keys) + bl : nullptr);
    __syncwarp();
    bool apples = false;
    if (thrA) {
        int base = 0;
#pragma unroll
        for (int q = 0; q < MW; q++) {
            if (q * 32 < p.n_apple) {
                bool sp = false;
                if ((eligm[q] >> lane) & 1u) sp = draws[base + __popc(eligm[q] & lanemask_lt(lane))] < thrA;
                if (sp) put_cell(tile, tile2, pr.a[q], C_APPLE);
                const unsigned spm = __ballot_sync(FULL, sp);
                am[q] |= spm;
                apples = apples || spm != 0u;
                base += __popc(eligm[q]);
            }
        }
    }
    if (!waste_on || C == 0) return apples;
    // waste: shuffle waste_points (stateless: key per canonical index), scan non-'H' cells in that
    // order, draw continues at rank M; first success spawns and breaks (:338-348)
    // number of failed draws before the first success
    int kstar = -1;
    {
        const unsigned succ = __ballot_sync(FULL, lane < wfirst && draws[M + lane] < p.thr_waste);
        if (succ) kstar = __ffs(succ) - 1;
    }
    for (int k0 = wfirst; k0 < C && kstar < 0; k0 += 32) {
        uint32_t dr = draw_u32_ool(g, t, SITE_SPAWN_DRAWS, (uint32_t)(M + k0 + lane));
        unsigned succ = __ballot_sync(FULL, (k0 + lane) < C && dr < p.thr_waste);
        if (succ) kstar = k0 + __ffs(succ) - 1;
    }
    if (kstar < 0) return apples;
    // the (kstar+1)-th smallest (key, index) among the candidates.  Each lane's <= MW candidate keys are read once; a
    // taken candidate's key becomes +inf.  Ties between equal keys go to the smaller index (a lane's own candidates are
    // scanned in index order, across lanes the second reduction decides).
    uint32_t ck[MW];
#pragma unroll
    for (int q = 0; q < MW; q++) ck[q] = ((candm[q] >> lane) & 1u) ? keys[lane + 32 * q] : 0xFFFFFFFFu;
    int chosen = -1;
    for (int it = 0; it <= kstar; it++) {
        uint32_t bk = 0xFFFFFFFFu; int bj = 0x7FFFFFFF;
#pragma unroll
        for (int q = 0; q < MW; q++)
            if (((candm[q] >> lane) & 1u) && ck[q] < bk) { bk = ck[q]; bj = lane + 32 * q; }
        uint32_t kmin = __reduce_min_sync(FULL, bk);
        int jmin = (int)__reduce_min_sync(FULL, (bk == kmin) ? (uint32_t)bj : 0x7FFFFFFFu);
        chosen = jmin;
        // remove it from the candidate set (uniform update of the owning lane's bit)
        int ql = jmin >> 5, ll = jmin & 31;
#pragma unroll
        for (int q = 0; q < MW; q++) if (q == ql) candm[q] &= ~(1u << ll);
    }
    {
        const int ql = chosen >> 5, ll = chosen & 31;
#pragma unroll
        for (int q = 0; q < MW; q++)
            if (q == ql) {
                if (lane == ll) put_cell(tile, tile2, pr.w[q], C_WASTE);
                wm[q] |= 1u << ll;
            }
    }
    hcount += 1;
    return true;
}

// harvest spawn (harvest_new.py:284-317): neighbour counts read the pre-spawn map.
// Every eligible point consumes one draw (by rank), but only a draw below the LARGEST spawn probability (0.05) can spawn
// whatever the neighbour count is.  So the 3x3 neighbour counts (8 tile reads) are evaluated only for those ~5 % of the
// eligible points, compacted into a list: one pass of the warp instead of one per 32 points.
template <int MW>
__device__ __forceinline__ bool harvest_spawn(const GridParams& p, int lane, uint8_t* tile, bool tile2, uint32_t* scratch,
                                              const EnvRng& g, uint32_t t, const PointRegs<MW>& pr, uint32_t (&am)[MW])
{
    const int S = p.S;
    unsigned eligm[MW];
    int M = 0;
#pragma unroll
    for (int q = 0; q < MW; q++) {
        eligm[q] = 0;
        if (q * 32 < p.n_apple) {
            const bool occ = (tile[pr.a[q] & 0xFFFFu] & OCC_BIT) != 0;
            eligm[q] = ~am[q] & round_valid(p.n_apple, q) & ~__ballot_sync(FULL, occ);
            M += __popc(eligm[q]);
        }
    }
    if (M == 0) return false;
    {   // draws [0, M): Philox blocks lane and lane + 32 as two interleaved chains (M > 128 needs more than 32 blocks)
        const int nblk = (M + 3) >> 2;
        uint4* d4 = reinterpret_cast<uint4*>(scratch);
        if (nblk <= 32) {
            if (lane < nblk) d4[lane] = draw_block_ool(g.seed, g.env_id, g.episode, t, SITE_SPAWN_DRAWS, (uint32_t)lane);
        } else {
            for (int bl = lane; __any_sync(FULL, bl < nblk); bl += 64)
                draw_blocks2_ool(g.seed, g.env_id, g.episode, t, SITE_SPAWN_DRAWS, (uint32_t)bl, bl < nblk ? d4 + bl : nullptr,
                                 SITE_SPAWN_DRAWS, (uint32_t)(bl + 32), bl + 32 < nblk ? d4 + bl + 32 : nullptr);
        }
        __syncwarp();                                                  // also orders the tile reads above
    }
    // candidates: (round << 5 | lane) | draw rank << 16, compacted behind the draws (M <= 256 draws + M <= 256 entries)
    uint32_t* list = scratch + SCRATCH_DRAWS;
    const uint32_t thr_max = p.thr_harvest[3];                         // SPAWN_PROB is increasing (harvest_new.py:34)
    int base = 0, ncand = 0;
#pragma unroll
    for (int q = 0; q < MW; q++) {
        if (q * 32 < p.n_apple) {
            const bool el = (eligm[q] >> lane) & 1u;
            const int r = base + __popc(eligm[q] & lanemask_lt(lane));
            const bool c = el && scratch[r] < thr_max;
            const unsigned cm = __ballot_sync(FULL, c);
            // the entry carries the point's offsets: the lane that evaluates it is not the lane that owns the point
            if (c) { const int k = ncand + __popc(cm & lanemask_lt(lane)); list[k] = pr.a[q]; list[256 + k] = (uint32_t)(lane + 32 * q) | ((uint32_t)r << 16); }
            ncand += __popc(cm);
            base += __popc(eligm[q]);
        }
    }
    if (ncand == 0) return false;
    __syncwarp();
    // neighbour counts of the candidates on the PRE-spawn map (j*j + k*k <= APPLE_RADIUS(=2): the 3x3 block; the own cell
    // is not 'A'), decisions first, writes after all of them
    for (int k = lane; k < ncand; k += 32) {
        const uint32_t pt = list[k], ent = list[256 + k];
        const int cell = (int)(pt & 0xFFFFu);
        int cnt = 0;
#pragma unroll
        for (int dr = -1; dr <= 1; dr++)
#pragma unroll
            for (int dc = -1; dc <= 1; dc++)
                if (dr | dc) cnt += ((tile[cell + dr * S + dc] & CODE_MASK) == C_APPLE);
        if (!(scratch[ent >> 16] < p.thr_harvest[cnt < 3 ? cnt : 3])) list[256 + k] = 0xFFFFFFFFu;
    }
    __syncwarp();
    bool spawned = false;
    for (int k0 = 0; k0 < ncand; k0 += 32) {
        const int k = k0 + lane;
        const uint32_t ent = k < ncand ? list[256 + k] : 0xFFFFFFFFu;
        if (ent != 0xFFFFFFFFu) { put_cell(tile, tile2, list[k], C_APPLE); spawned = true; }
        // mask bits of the spawned points (point index = ent & 0xFFFF), gathered by round
        const uint32_t j = ent & 0xFFFFu;
#pragma unroll
        for (int q = 0; q < MW; q++) {
            uint32_t bit = (ent != 0xFFFFFFFFu && (j >> 5) == (uint32_t)q) ? (1u << (j & 31u)) : 0u;
            am[q] |= __reduce_or_sync(FULL, bit);
        }
    }
    __syncwarp();
    return __any_sync(FULL, spawned);
}

// count_apples_in_radius(5, loc) (harvest_new.py:326-336): the 21 cells with j*j + k*k <= 5
__device__ __forceinline__ int count_apples_r5(const uint8_t* tile, int o, int S)
{
    int cnt = 0;
#pragma unroll
    for (int dr = -2; dr <= 2; dr++)
#pragma unroll
        for (int dc = -2; dc <= 2; dc++)
            if (dr * dr + dc * dc <= 5) cnt += ((tile[o + dr * S + dc] & CODE_MASK) == C_APPLE);
    return cnt;
}

// ---------------------------------------------------------------------------------------------
// infos['feature_obs'] (cleanup_new.py:235-251, harvest_new.py:208-222).  Lists are the row-major
// scans of the post-step map (compute_current_apples / _wastes) = the set bits of the masks in point order; np.argmin
// takes the first minimum, i.e. the smallest (L1 distance, list index).  Returns (dist << 16 | index) or 0xFFFFFFFF.
template <int MW>
__device__ __forceinline__ uint32_t closest_point(int lane, const uint32_t (&m)[MW], const uint16_t* rc, int ar, int ac)
{
    uint32_t best = 0xFFFFFFFFu;
#pragma unroll
    for (int q = 0; q < MW; q++) {
        if ((m[q] >> lane) & 1u) {
            const int j = lane + 32 * q;
            int r = rc[j] >> 8, c = rc[j] & 255;
            uint32_t key = ((uint32_t)(abs(r - ar) + abs(c - ac)) << 16) | (uint32_t)j;
            best = key < best ? key : best;
        }
    }
    return __reduce_min_sync(FULL, best);
}
// element k of a feature row: float64 as it is, a policy element type as T(float32(x))
template <typename T>
__device__ __forceinline__ void feat_put(T* f, int k, double x) { f[k] = policy_cast<T>(__double2float_rn(x)); }
template <>
__device__ __forceinline__ void feat_put<double>(double* f, int k, double x) { f[k] = x; }
// out: the env's n rows of `width` elements (0: p.F; columns p.F.. of a wider row are left to the caller)
template <int KIND, int MW, typename OUT = double>
__device__ __forceinline__ void write_features(const GridParams& p, const SharedTables& tb, int lane, uint32_t hw /* agent word of lane < n */,
                                               const uint32_t (&am)[MW], const uint32_t (&wm)[MW],
                                               int cleaned, int total_close, int hcount, OUT* out, int width = 0)
{
    const int n = p.n;
    const int my_r = (int)(hw & 255u), my_c = (int)((hw >> 8) & 255u), ori = (int)((hw >> 16) & 3u);
    int n_apples = 0;
#pragma unroll
    for (int q = 0; q < MW; q++) n_apples += __popc(am[q]);
    int ca_r = 0, ca_c = 0, cw_r = 0, cw_c = 0;        // sentinel [0, 0] when the list is empty
    for (int a = 0; a < n; a++) {
        int ar = __shfl_sync(FULL, my_r, a), ac = __shfl_sync(FULL, my_c, a);
        uint32_t ka = closest_point<MW>(lane, am, tb.apple_rc, ar, ac);
        uint32_t kw = 0xFFFFFFFFu;
        if (KIND == SSD_ENV_CLEANUP) kw = closest_point<MW>(lane, wm, tb.waste_rc, ar, ac);
        if (lane == a) {
            if (ka != 0xFFFFFFFFu) { ca_r = tb.apple_rc[ka & 0xFFFFu] >> 8; ca_c = tb.apple_rc[ka & 0xFFFFu] & 255; }
            if (kw != 0xFFFFFFFFu) { cw_r = tb.waste_rc[kw & 0xFFFFu] >> 8; cw_c = tb.waste_rc[kw & 0xFFFFu] & 255; }
        }
    }
    // compute_closest_pos (cleanup_new.py:405-412): distances are 0 for every other agent, so the
    // argmin is agent 0 (agent 1 for agent 0; itself when alone)
    const int cp = lane == 0 ? (n > 1 ? 1 : 0) : 0;
    const int cp_r = __shfl_sync(FULL, my_r, cp), cp_c = __shfl_sync(FULL, my_c, cp), cp_o = __shfl_sync(FULL, ori, cp);
    int cl[SSD_MAXN];
#pragma unroll
    for (int j = 0; j < SSD_MAXN; j++) cl[j] = __shfl_sync(FULL, cleaned, j);
    if (lane < n) {
        OUT* f = out + (size_t)lane * (width ? width : p.F);
        feat_put(f, 0, my_r); feat_put(f, 1, my_c); feat_put(f, 2, ori); feat_put(f, 3, cp_r); feat_put(f, 4, cp_c);
        feat_put(f, 5, cp_o); feat_put(f, 6, ca_r); feat_put(f, 7, ca_c);
        if (KIND == SSD_ENV_CLEANUP) {
            feat_put(f, 8, cw_r); feat_put(f, 9, cw_c); feat_put(f, 10, n_apples); feat_put(f, 11, hcount);
#pragma unroll
            for (int j = 0; j < SSD_MAXN; j++) if (j < n) feat_put(f, 12 + j, cl[j]);
        } else {
            feat_put(f, 8, total_close); feat_put(f, 9, n_apples);
            for (int j = 0; j < 2 * n; j++) feat_put(f, 10 + j, 0.0);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// observations (color_view, map_env.py:397-411): out[i][j] of agent a is a strided walk over the
// painted tile: V[i][j] (UP), V[j][14-i] (LEFT), V[14-i][14-j] (DOWN), V[14-j][i] (RIGHT), with
// V[a][b] = tile[origin + a*S + b].  So output row i starts at start0 + i*rs and advances by `step`
// per pixel; {start0, step, rs} per agent live in vdesc.  The env's observation stream is 15 n rows
// of 45 B; a work item is 4 consecutive rows = 60 pixels = 45 words (word aligned whatever the
// agents), one item per lane, staged with conflict-free word stores (lane stride 45 words) and
// shipped with one bulk async store (head / tail up to the 16-B boundaries by plain stores).
__device__ __forceinline__ void pack4(uint32_t* dst, uint32_t p0, uint32_t p1, uint32_t p2, uint32_t p3)
{
    dst[0] = __byte_perm(p0, p1, 0x4210);
    dst[1] = __byte_perm(p1, p2, 0x5421);
    dst[2] = __byte_perm(p2, p3, 0x6542);
}
// the staged observation stream of one env (L bytes at stage + shift, congruent to gdst modulo 16) -> HBM:
// one bulk async store for the 16-byte aligned middle, plain stores for the head / tail
__device__ __forceinline__ void obs_stream_store(int lane, uint8_t* stage, int shift, bool word_ok, int L, uint8_t* gdst)
{
    uint32_t* sw = reinterpret_cast<uint32_t*>(stage + shift);
    __syncwarp();
    if (word_ok) {
        const int a0 = (16 - shift) & 15;               // head bytes up to the first 16-B boundary
        const int mid = (L - a0) & ~15;
        const int tail0 = a0 + mid;
        // head / tail: whole words first, then bytes
        if (lane < (a0 >> 2)) reinterpret_cast<uint32_t*>(gdst)[lane] = sw[lane];
        {
            int tw = (L - tail0) >> 2;
            if (lane < tw) reinterpret_cast<uint32_t*>(gdst + tail0)[lane] = sw[(tail0 >> 2) + lane];
            int tb0 = tail0 + tw * 4;
            if (lane < L - tb0) gdst[tb0 + lane] = (stage + shift)[tb0 + lane];
        }
        if (mid > 0) {
            fence_async_smem();
            __syncwarp();
            if (lane == 0) bulk_store(gdst + a0, stage + shift + a0, (uint32_t)mid);
        }
    } else {
        for (int i = lane; i < L; i += 32) gdst[i] = stage[i];
    }
}


// view descriptor of an agent at tile offset ao for byte-step reads over T (gather_obs): {out[0][0], pixel step, row step, 0}
__device__ __forceinline__ int4 view_desc(int ao, int ori, int S)
{
    const int origin = ao - SSD_VIEW * S - SSD_VIEW;     // V[0][0] of this lane's agent
    const int last = SSD_OBSW - 1;
    int start0 = origin, step = 1, rs = S;               // UP
    if (ori == ORI_RIGHT) { start0 = origin + last * S; step = -S; rs = 1; }
    else if (ori == ORI_DOWN) { start0 = origin + last * S + last; step = -1; rs = -S; }
    else if (ori == ORI_LEFT) { start0 = origin + last; step = S; rs = -1; }
    return make_int4(start0, step, rs, 0);
}

// view descriptor for word reads over T and its transpose T2 (gather_obs2, see there): {lowest byte of out row 0's run, row
// step, backwards, 0}
__device__ __forceinline__ int4 view_desc2(const GridParams& p, int ao, int ori)
{
    const int S = p.S, S2 = p.S2;
    const uint32_t trow = __umulhi((uint32_t)ao, p.s_magic);            // ao / S
    const int row = (int)trow - SSD_VIEW, col = ao - (int)trow * S - 8;
    const int origin = ao - SSD_VIEW * S - SSD_VIEW;                     // V[0][0] in T
    const int origin2 = p.tile2_off + (col + SSD_VIEW) * S2 + 8 + row - SSD_VIEW * S2 - SSD_VIEW;   // V[0][0] in T2
    const int last = SSD_OBSW - 1;
    int lo0 = origin, rstep = S, back = 0;                                // UP
    if (ori == ORI_DOWN) { lo0 = origin + last * S; rstep = -S; back = 1; }
    else if (ori == ORI_LEFT) { lo0 = origin2 + last * S2; rstep = -S2; }
    else if (ori == ORI_RIGHT) { lo0 = origin2; rstep = S2; back = 1; }
    return make_int4(lo0, rstep, back, 0);
}
// the 15-byte run whose lowest byte is tile[lo], from 5 aligned words: pixel j is byte j & 3 of bw[j >> 2] (back: the run
// read backwards, pixel j = byte 14 - j)
__device__ __forceinline__ void run_bytes15(const uint8_t* tile, int lo, int back, uint32_t (&bw)[4])
{
    const uint32_t* wsrc = reinterpret_cast<const uint32_t*>(tile + (lo & ~3));
    const uint32_t w0 = wsrc[0], w1 = wsrc[1], w2 = wsrc[2], w3 = wsrc[3], w4 = wsrc[4];
    const uint32_t sh = (uint32_t)(lo & 3) * 8u;
    uint32_t b0 = __funnelshift_r(w0, w1, sh), b1 = __funnelshift_r(w1, w2, sh);
    uint32_t b2 = __funnelshift_r(w2, w3, sh), b3 = __funnelshift_r(w3, w4, sh);   // bytes lo .. lo + 15
    if (back) {
        const uint32_t r0 = __byte_perm(b2, b3, 0x3456), r1 = __byte_perm(b1, b2, 0x3456);
        const uint32_t r2 = __byte_perm(b0, b1, 0x3456), r3 = __byte_perm(b0, b0, 0x0012);
        b0 = r0; b1 = r1; b2 = r2; b3 = r3;
    }
    bw[0] = b0; bw[1] = b1; bw[2] = b2; bw[3] = b3;
}

// PENDING: bulk groups of this lane-0 that may stay in flight while `stage` is rewritten
template <int PENDING>
__device__ __forceinline__ void gather_obs(const GridParams& p, int lane, const uint8_t* tile, uint8_t* stage,
                                           const uint32_t* sm_pal, int4* vdesc, int ao, int ori, uint8_t* gdst)
{
    const int n = p.n, S = p.S;
    const int L = n * SSD_OBS_BYTES;
    const uint32_t gaddr = (uint32_t)(reinterpret_cast<uintptr_t>(gdst) & 15u);
    const bool word_ok = (gaddr & 3u) == 0;
    const int shift = word_ok ? (int)gaddr : 0;          // staged stream is congruent to gdst modulo 16
    uint32_t* sw = reinterpret_cast<uint32_t*>(stage + shift);
    if (lane < n) vdesc[lane] = view_desc(ao, ori, S);
    if (lane == 0) bulk_wait_read<PENDING>();                // the previous env's store has drained `stage`
    __syncwarp();
    if (lane < p.obs_items) {
        uint32_t col[60];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int r = 4 * lane + q;
            int a = (int)(((uint32_t)r * 0x8889u) >> 19);    // r / 15
            int i = r - 15 * a;
            if (a >= n) { a = n - 1; i = SSD_OBSW - 1; }     // rows past the stream end: harmless in-bounds reads
            const int4 d = vdesc[a];
            const uint8_t* src = tile + (d.x + i * d.z);
#pragma unroll
            for (int j = 0; j < SSD_OBSW; j++)      // a tile byte IS the byte offset of its palette entry
                col[15 * q + j] = *reinterpret_cast<const uint32_t*>(reinterpret_cast<const uint8_t*>(sm_pal) + src[j * d.y]);
        }
        uint32_t* dst = sw + 45 * lane;
#pragma unroll
        for (int g4 = 0; g4 < 15; g4++) pack4(dst + 3 * g4, col[4 * g4], col[4 * g4 + 1], col[4 * g4 + 2], col[4 * g4 + 3]);
    }
    obs_stream_store(lane, stage, shift, word_ok, L, gdst);
}

// ---------------------------------------------------------------------------------------------
// Policy forms of the observation (ssd_set_policy_output): the windows as VisionNetwork.forward feeds them to its first
// convolution, T [n][3][15][15] per env, value T(float32(float64(byte) / 255)) — what ssd_policy_inputs makes of the uint8
// windows, written directly.
//
// Per-CTA palette of a policy form: element b of it, for a tile byte b = palette index << 2, is channel 0 of that colour,
// b + 1 / b + 2 channels 1 / 2 (b + 3 unused), so one 16-byte (float) or 8-byte (half types) shared load gives a pixel.
// Static shared memory, addressed where it is read (a pointer kept in a register across the env loop would spill).
template <typename T>
__device__ __forceinline__ T* policy_palette()
{
    __shared__ __align__(16) T s_ppal[64];
    return s_ppal;
}
// (visible after the caller's next __syncthreads)
template <typename T>
__device__ __forceinline__ void load_policy_palette(const GridParams& p)
{
    T* pal = policy_palette<T>();
    for (int i = threadIdx.x; i < 64; i += blockDim.x) {
        const uint32_t c = (uint32_t)i & 3u, rgb = __ldg(p.pal + (i >> 2));
        const uint32_t v = c < 3u ? (rgb >> (8u * c)) & 255u : 0u;
        pal[i] = policy_cast<T>(__double2float_rn(__ddiv_rn((double)v, 255.0)));
    }
}
// pixel j of an image row: its three channel planes are 225 elements apart
__device__ __forceinline__ void put_pixel(float* o, const float* e, int j)
{
    const float4 v = *reinterpret_cast<const float4*>(e);
    o[j] = v.x; o[SSD_OBS_PIX + j] = v.y; o[2 * SSD_OBS_PIX + j] = v.z;
}
template <typename H>
__device__ __forceinline__ void put_pixel(H* o, const H* e, int j)
{
    const uint2 v = *reinterpret_cast<const uint2*>(e);
    uint16_t* o16 = reinterpret_cast<uint16_t*>(o);
    o16[j] = (uint16_t)v.x; o16[SSD_OBS_PIX + j] = (uint16_t)(v.x >> 16); o16[2 * SSD_OBS_PIX + j] = (uint16_t)v.y;
}
// a staged chunk (L bytes at stage + shift, shift = gdst mod 16; gdst and L even) -> HBM: one bulk async store for the
// 16-byte aligned middle, halfword stores for the head / tail (an env block of n 675 sizeof(T) bytes starts on any even
// address when n is odd)
__device__ __forceinline__ void policy_stream_store(int lane, uint8_t* stage, int shift, int L, uint8_t* gdst)
{
    const uint16_t* sh = reinterpret_cast<const uint16_t*>(stage + shift);
    __syncwarp();
    const int a0 = (16 - shift) & 15;                  // head bytes up to the first 16-B boundary (L >= 1350 > a0)
    const int mid = (L - a0) & ~15;
    const int tail0 = a0 + mid;
    if (lane < (a0 >> 1)) reinterpret_cast<uint16_t*>(gdst)[lane] = sh[lane];
    if (lane < ((L - tail0) >> 1)) reinterpret_cast<uint16_t*>(gdst + tail0)[lane] = sh[(tail0 >> 1) + lane];
    if (mid > 0) {
        fence_async_smem();
        __syncwarp();
        if (lane == 0) bulk_store(gdst + a0, stage + shift + a0, (uint32_t)mid);
    }
}
// One env's windows in policy form T at gdst.  The staging area holds `per` agents' planes (stage_r16 = g2_misc - g2_stage
// bytes: cleanup n = 8 gives 2 agents of float or 4 of a half type, 5400 B), so the env goes out in ceil(n / per) chunks,
// each staged and shipped like the uint8 stream.  A lane builds whole image rows: row (a, i) is a run of 15 tile bytes,
// read as gather_obs2 reads it (TWO: 5 aligned words of T or T2) or as gather_obs does (byte steps over T, the reset kernel).
template <int FORM, bool TWO>
__device__ __forceinline__ void gather_policy(const GridParams& p, int lane, const uint8_t* tile, uint8_t* stage,
                                              int4* vdesc, int ao, int ori, uint8_t* gdst)
{
    typedef typename ObsForm<FORM>::T T;
    const T* ppal = policy_palette<T>();
    const int n = p.n;
    if (lane < n) vdesc[lane] = TWO ? view_desc2(p, ao, ori) : view_desc(ao, ori, p.S);
    const int per = (p.g2_misc - p.g2_stage - 16) / (SSD_OBS_BYTES * (int)sizeof(T));
    for (int a0 = 0; a0 < n; a0 += per) {
        const int k = min(per, n - a0);
        uint8_t* g = gdst + (size_t)a0 * SSD_OBS_BYTES * sizeof(T);
        const int shift = (int)(reinterpret_cast<uintptr_t>(g) & 15u);
        T* st = reinterpret_cast<T*>(stage + shift);
        if (lane == 0) bulk_wait_read<0>();              // the previous chunk's (env's) store has drained `stage`
        __syncwarp();
        for (int r = lane; r < SSD_OBSW * k; r += 32) {
            const int ar = (int)(((uint32_t)r * 0x8889u) >> 19), i = r - SSD_OBSW * ar;     // r / 15, r % 15
            const int4 d = vdesc[a0 + ar];
            T* o = st + ar * SSD_OBS_BYTES + i * SSD_OBSW;
            if (TWO) {
                uint32_t bw[4];
                run_bytes15(tile, d.x + i * d.y, d.z, bw);
#pragma unroll
                for (int j = 0; j < SSD_OBSW; j++) put_pixel(o, ppal + __byte_perm(bw[j >> 2], 0u, 0x4440u + (uint32_t)(j & 3)), j);
            } else {
                const uint8_t* src = tile + (d.x + i * d.z);
#pragma unroll
                for (int j = 0; j < SSD_OBSW; j++) put_pixel(o, ppal + src[j * d.y], j);
            }
        }
        policy_stream_store(lane, stage, shift, k * SSD_OBS_BYTES * (int)sizeof(T), g);
    }
}
// the contract rows of one env: (theta, 0) x 5 per agent, T [n][10] (vision_net.py:160-161, as ssd_policy_inputs)
template <typename T>
__device__ __forceinline__ void policy_contract_rows(T* c, int n, double theta, int lane, int lanes)
{
    const T v = policy_cast<T>(__double2float_rn(theta)), z = policy_cast<T>(0.0f);
    for (int k = lane; k < n * 10; k += lanes) c[k] = (k & 1) ? z : v;
}

// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ SharedTables load_shared_tables(const GridParams& p, uint8_t* smem, bool feat)
{
    uint32_t* pal = reinterpret_cast<uint32_t*>(smem);          // [16]: 16 distinct banks, no replication needed
    uint32_t* thr = reinterpret_cast<uint32_t*>(smem + p.sm_thr);
    uint8_t* won = smem + p.sm_won;
    uint16_t* apple_rc = reinterpret_cast<uint16_t*>(smem + p.sm_apple_rc);
    uint16_t* waste_rc = reinterpret_cast<uint16_t*>(smem + p.sm_waste_rc);
    for (int i = threadIdx.x; i < 16; i += blockDim.x) pal[i] = __ldg(p.pal + i);
    for (int i = threadIdx.x; i <= p.n_waste; i += blockDim.x) { thr[i] = __ldg(p.thr_apple + i); won[i] = __ldg(p.waste_on + i); }
    if (feat) {
        for (int i = threadIdx.x; i < p.n_apple; i += blockDim.x) apple_rc[i] = __ldg(p.apple_rc + i);
        for (int i = threadIdx.x; i < p.n_waste; i += blockDim.x) waste_rc[i] = __ldg(p.waste_rc + i);
    }
    SharedTables t = { pal, thr, won, apple_rc, waste_rc };
    return t;
}
// this warp's [T | T2] <- the static tiles (every dynamic cell OFF)
__device__ __forceinline__ void init_warp_tiles(const GridParams& p, uint8_t* tile, int lane)
{
    const uint4* src = reinterpret_cast<const uint4*>(p.tile0);
    for (int i = lane; i < (p.g2_stage >> 4); i += 32) reinterpret_cast<uint4*>(tile)[i] = __ldg(src + i);
}
// rewrite every dynamic cell of T (and T2) from the env's masks.  rot3 = (lane - 3) & 31, rot2 = (lane - 2) & 31: rotating a
// mask word right by them puts this lane's bit where the cell code wants it (C_APPLE = 8 = bit 3; C_RIVER - C_WASTE = 4).
template <int MW, bool HAS2>
__device__ __forceinline__ void apply_masks(const GridParams& p, uint8_t* tile, const PointRegs<MW>& pr,
                                            const uint32_t (&am)[MW], const uint32_t (&wm)[MW], uint32_t rot3, uint32_t rot2)
{
    static_assert(C_APPLE == 8 && C_EMPTY == 0 && C_RIVER == 16 && C_WASTE == 12, "cell codes are folded into bit tricks here");
#pragma unroll
    for (int q = 0; q < MW; q++) {
        if (q * 32 < p.n_apple) put_cell(tile, HAS2, pr.a[q], __funnelshift_r(am[q], am[q], rot3) & 8u);
        if (q * 32 < p.n_waste) put_cell(tile, HAS2, pr.w[q], 16u - (__funnelshift_r(wm[q], wm[q], rot2) & 4u));
    }
}

// =============================================================================================
// RESET of one env by one warp: setup_agents + reset_map + custom_reset + reset-time spawn + contract sample + reset obs
// (+ the negotiation agreement when the policy's negotiation outputs are given).  `tile` is the warp's T with every agent
// mark removed; it is left that way.
// (Measured and dropped in round 2: doing this inside the observe kernel for the envs that finish in the step.  Inlined it
// costs the hot loop registers (12 -> 68 B of spills), out of line it forces spills around the call, and a warp that
// resets an env finishes ~10 us after the others of the one-wave persistent grid: observe kernel 0.204 -> 0.223 ms, more
// than the launch it saves.  ssd_step_io.auto_reset therefore launches the masked reset kernel behind the step.)
// FORM: the observation form written to obs_dst (OBS_U8, or a policy form and, when pcontract is given, the env's contract
// rows there).
template <int KIND, int MW, int FORM>
__device__ __forceinline__ void reset_env(const GridParams& p, const SharedTables& tb, int lane, uint8_t* tile, uint8_t* stage, int4* vdesc,
                                          const PointRegs<MW>& pr, int env, uint8_t* obs_dst, const double* neg_prop,
                                          const double* neg_acc, uint8_t* neg_dec, void* pcontract)
{
    const int n = p.n, S = p.S;
    const bool act_lane = lane < n;
    uint32_t* scratch = reinterpret_cast<uint32_t*>(stage);
    uint8_t* hdr = p.state + (size_t)env * p.rec_stride;
    uint32_t flags = *reinterpret_cast<const uint32_t*>(hdr + RO_FLAGS);
    uint32_t episode = *reinterpret_cast<const uint32_t*>(hdr + RO_EPISODE);
    if (p.stats && (flags & 0x80000000u)) {       // a finished episode is replaced: hand its accumulators over
        double tr = 0.0, raw = 0.0;
        if (act_lane) {
            tr = reinterpret_cast<const double*>(hdr + RO_SUM_TR)[lane];
            raw = p.reward_mode ? reinterpret_cast<const double*>(hdr + RO_XSUM)[lane]
                                : (double)reinterpret_cast<const int*>(hdr + RO_SUM_RAW)[lane];
        }
        for (int o = 16; o; o >>= 1) { tr += __shfl_xor_sync(FULL, tr, o); raw += __shfl_xor_sync(FULL, raw, o); }
        if (lane == 0) {
            atomicAdd(p.stats + 0, (double)*reinterpret_cast<const uint32_t*>(hdr + RO_APPLES));
            atomicAdd(p.stats + 1, p.reward_mode ? *reinterpret_cast<const double*>(hdr + RO_XRAW) : raw);
            atomicAdd(p.stats + 2, *reinterpret_cast<const double*>(hdr + RO_TRANSFERS));
            atomicAdd(p.stats + 3, (double)*reinterpret_cast<const uint32_t*>(hdr + RO_DIRT));
            atomicAdd(p.stats + 4, tr);
            atomicAdd(p.stats + 5, raw);
            atomicAdd(p.stats + 6, 1.0);
            // non-negative doubles order like their bit patterns
            atomicMax(reinterpret_cast<unsigned long long*>(p.stats + 7),
                      (unsigned long long)__double_as_longlong((double)((flags >> RF_ERR_SHIFT) & 0xFFFFu)));
        }
    }
    if (p.elog.records && (flags & 0x80000000u)) {   // the same episode as one record of the episode log: lane v writes vector v
        unsigned long long slot = 0;
        if (lane == 0) slot = atomicAdd(p.elog.count, 1ull) % p.elog.capacity;
        slot = __shfl_sync(FULL, slot, 0);
        uint4 w;
        if (lane == 0) {
            const int t = *reinterpret_cast<const int*>(hdr + RO_T);
            w = eprec_head(p.first_env_id + (uint32_t)env, episode, t, t == p.horizon);
        } else if (lane == 1) {
            w = eprec_pair(*reinterpret_cast<const double*>(hdr + RO_THETA), 0.0);
        } else {
            w = eprec_pair(grid_metric(p, hdr, 2 * lane - 4), grid_metric(p, hdr, 2 * lane - 3));
        }
        if (lane < EPREC_VECS) p.elog.records[slot * EPREC_VECS + lane] = w;
    }
    // the first reset of a record (flags bit 31 clear) is episode 0; later resets increment
    episode = (flags & 0x80000000u) ? episode + 1u : 0u;
    EnvRng g = { p.seed, p.first_env_id + (uint32_t)env, episode, 0u };

    // ---- setup_agents (cleanup_new.py:302-320 / harvest_new.py:132-141; map_env.py:816-832)
    // Lane l owns the canonical spawn-list entries 4 l .. 4 l + 3 (<= 128 entries), so ONE Philox block per agent gives
    // the lane's four shuffle keys (draw idx j lives in block j >> 2, word j & 3); lane i draws agent i's rotation.
    int ao = 0, ori = 0;
    uint32_t cells[4];
#pragma unroll
    for (int k = 0; k < 4; k++) cells[k] = 4 * lane + k < p.n_spawn ? (uint32_t)__ldg(p.spawn_pts + 4 * lane + k) : 0xFFFFFFFFu;
    uint32_t rot = 0;
    if (act_lane) rot = draw_u32(g.seed, g.env_id, g.episode, 0, SITE_SPAWN_ROT, (uint32_t)lane, 0u) >> 30;
    unsigned taken[4] = { 0, 0, 0, 0 };          // taken[k] bit l: entry 4 l + k is occupied (uniform)
    for (int i = 0; i < n; i++) {
        // shuffled list = canonical entries ordered by (key, idx); the LAST free entry wins (:822-825)
        const Philox4 kq = draw_block(g.seed, g.env_id, g.episode, 0, SITE_SPAWN_POINT, (uint32_t)i, (uint32_t)lane);
        const uint32_t kk4[4] = { kq.x, kq.y, kq.z, kq.w };
        uint32_t bk = 0; int bj = -1;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int j = 4 * lane + k;
            if (j < p.n_spawn && !((taken[k] >> lane) & 1u)) {
                const uint32_t kk = kk4[k];
                if (bj < 0 || kk > bk || (kk == bk && j > bj)) { bk = kk; bj = j; }
            }
        }
        uint32_t kmax = __reduce_max_sync(FULL, bj >= 0 ? bk : 0u);
        int jmax = (int)__reduce_max_sync(FULL, (bj >= 0 && bk == kmax) ? (uint32_t)(bj + 1) : 0u) - 1;
        const uint32_t mine = (jmax & 3) == 0 ? cells[0] : ((jmax & 3) == 1 ? cells[1] : ((jmax & 3) == 2 ? cells[2] : cells[3]));
        const int cell = (int)__shfl_sync(FULL, mine, jmax >> 2);
        // every canonical entry on that cell becomes occupied (cleanup lists each point twice)
#pragma unroll
        for (int k = 0; k < 4; k++) taken[k] |= __ballot_sync(FULL, cells[k] == (uint32_t)cell);
        const uint32_t rdraw = __shfl_sync(FULL, rot, i);
        // list(ORIENTATIONS.keys()) = LEFT, RIGHT, UP, DOWN (map_env.py:22, :829-832)
        int o = rdraw == 0 ? ORI_LEFT : (rdraw == 1 ? ORI_RIGHT : (rdraw == 2 ? ORI_UP : ORI_DOWN));
        if (lane == i) { ao = cell; ori = o; }
    }
    // ---- reset_map + custom_reset: the initial dynamic state, occupancy, reset-time spawn (map_env.py:319-320)
    uint32_t am[MW], wm[MW];
#pragma unroll
    for (int q = 0; q < MW; q++) { am[q] = p.reset_amask[q]; wm[q] = p.reset_wmask[q]; }
    apply_masks<MW, false>(p, tile, pr, am, wm, (uint32_t)(lane - 3) & 31u, (uint32_t)(lane - 2) & 31u);
    if (lane == 0) bulk_wait_read<0>();          // `stage` doubles as the spawn scratch
    __syncwarp();
    if (act_lane) tile[ao] |= OCC_BIT;           // co-located lanes write the same value
    __syncwarp();
    int hcount = p.n_waste_start;
    if (KIND == SSD_ENV_CLEANUP) cleanup_spawn<MW>(p, tb, lane, tile, false, scratch, g, 0u, hcount, pr, am, wm);
    else harvest_spawn<MW>(p, lane, tile, false, scratch, g, 0u, pr, am);
    __syncwarp();
    if (act_lane) tile[ao] &= CODE_MASK;              // MapEnv.reset never paints agents into the colour grid; the tile is clean again
    __syncwarp();
    if (obs_dst) {
        if constexpr (FORM == OBS_U8) gather_obs<0>(p, lane, tile, stage, tb.pal, vdesc, ao, ori, obs_dst);
        else gather_policy<FORM, false>(p, lane, tile, stage, vdesc, ao, ori, obs_dst);
    }

    // ---- SeparateContractSubgameStage.reset (two_stage_train.py:163-168)
    double theta = 0.0;
    if (p.contract != SSD_CONTRACT_NONE) {
        Philox4 q = draw_block(g.seed, g.env_id, g.episode, 0, SITE_CONTRACT, 0, 0);
        double u0 = __dmul_rn((double)q.x, 1.0 / 4294967296.0), u1 = __dmul_rn((double)q.y, 1.0 / 4294967296.0);
        theta = (u0 > p.null_prob) ? __dadd_rn(p.theta_low, __dmul_rn(__dsub_rn(p.theta_high, p.theta_low), u1))
                                   : p.theta_low;
    }
    // ---- negotiation prologue of the new episode (SeparateContractNegotiateStage.step, two_stage_train.py:257-281)
    if (neg_prop && lane == 0) {
        const bool dec = negotiate_agreement(g.seed, g.env_id, episode, n, neg_acc + (size_t)env * n);
        theta = dec ? neg_prop[env] : 0.0;
        if (neg_dec) neg_dec[env] = dec ? 1 : 0;
    }
    if constexpr (FORM != OBS_U8) {
        if (pcontract) {                                  // lane 0 holds the negotiated theta
            typedef typename ObsForm<FORM>::T T;
            policy_contract_rows(reinterpret_cast<T*>(pcontract) + (size_t)env * n * 10, n, __shfl_sync(FULL, theta, 0), lane, 32);
        }
    }
    // ---- record: zero everything, then the hot line
    for (int i = lane; i < p.hdr_bytes / 4; i += 32) reinterpret_cast<uint32_t*>(hdr)[i] = 0u;
    __syncwarp();
    if (act_lane) {
        uint32_t row = (uint32_t)(ao / S) - SSD_VIEW, col = (uint32_t)(ao % S) - 8u;
        reinterpret_cast<uint32_t*>(hdr + RO_AGENTS)[lane] = row | (col << 8) | ((uint32_t)ori << 16);
    }
#pragma unroll
    for (int q = 0; q < MW; q++)
        if (lane == q) {
            reinterpret_cast<uint32_t*>(hdr + RO_AMASK)[q] = am[q];
            reinterpret_cast<uint32_t*>(hdr + RO_WMASK)[q] = wm[q];
        }
    if (lane == 0) {
        *reinterpret_cast<uint32_t*>(hdr + RO_EPISODE) = episode;
        *reinterpret_cast<double*>(hdr + RO_THETA) = theta;
        *reinterpret_cast<uint32_t*>(hdr + RO_FLAGS) = 0x80000000u | (KIND == SSD_ENV_CLEANUP ? RF_STALE_EMPTY : 0u);
        *reinterpret_cast<int*>(hdr + RO_HCOUNT) = hcount;
    }
    __syncwarp();
}

// RESET kernel: one warp per env; the warp's envs are env0 + i * estride, their mask bytes are read 32 at a time (one round
// trip, one ballot), so a sparse mask — a vectorised sampler in steady state resets ~E / horizon envs per step — costs a
// few loads per warp.
// FORM (see OBS_U8): obs is a policy image tensor T for the policy forms, pcontract its contract rows (nullable; unused for OBS_U8).
template <int KIND, int FORM = OBS_U8>
__global__ void __launch_bounds__(GRID_THREADS) grid_reset_kernel(const GridParams p, const uint8_t* mask,
                                                                  uint8_t* obs, long long obs_stride, const StepIO io, void* pcontract)
{
    constexpr int MW = MAX_POINT_ROUNDS;
    extern __shared__ __align__(16) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int env0 = blockIdx.x * GRID_WARPS + warp, estride = gridDim.x * GRID_WARPS;
    pdl_wait();                                       // the mask (dones) and the records come from the step's kernels
    // nothing to do for this CTA (steady state: most of them)?  Leave before the table / tile set-up.
    {
        bool any = false;
        for (long long e = env0 + (long long)lane * estride; e < p.E; e += 32ll * estride) any = any || !mask || mask[e];
        if (!__syncthreads_or(any)) return;
    }
    const SharedTables tb = load_shared_tables(p, smem, false);
    if constexpr (FORM != OBS_U8) load_policy_palette<typename ObsForm<FORM>::T>(p);
    uint8_t* tile = smem + p.sm_warp0 + warp * p.g2_warp_bytes;
    uint8_t* stage = tile + p.g2_stage;
    int4* vdesc = reinterpret_cast<int4*>(tile + p.g2_misc + MISC_VDESC);
    const PointRegs<MW> pr = load_point_regs<MW>(p, lane);
    init_warp_tiles(p, tile, lane);
    __syncthreads();
    for (int i0 = 0; env0 + (long long)i0 * estride < p.E; i0 += 32) {
        const long long el = env0 + (long long)(i0 + lane) * estride;
        unsigned todo = __ballot_sync(FULL, el < p.E && (!mask || mask[el]));
        while (todo) {
            const int env = env0 + (i0 + __ffs(todo) - 1) * estride;
            todo &= todo - 1;
            reset_env<KIND, MW, FORM>(p, tb, lane, tile, stage, vdesc, pr, env, obs ? obs + (size_t)env * (size_t)obs_stride : nullptr,
                                      io.neg_prop, io.neg_acc, io.neg_dec, pcontract);
        }
    }
    if (lane == 0) bulk_wait_read<0>();
}
