// ssd_grid2.cuh — the gridworld step as two kernels: LOGIC (lane = env) + OBSERVE (warp = env).
//
// Why two mappings.  The reference's per-env decision logic (update_moves, consume, beams, reward
// redistribution) is serial and tiny (n <= 8 agents).  Run with a warp per env it keeps 8 of 32 lanes busy and costs
// ~600 warp-instructions per env; run with a lane per env it costs ~200, but a fused kernel that alternates both mappings
// inside one warp (measured in round 1: 884 instead of 1411 warp-instructions per env, yet 0.49-0.64 ms instead of
// 0.36 ms) is left with 6-13 warps per SM.  So the step is split:
//
//   grid_logic_kernel    one THREAD per env.  It reads the env's 128-byte hot line (agents, t, episode, theta, flags,
//                        #waste, apple / waste bitmasks) and NOTHING else of the env: walls and "which point of which list
//                        is this cell" come from a static per-cell table in shared memory, apples / waste from the masks.
//                        Action decode, rotations, moves, consume, beams, then — cleanup — contract transfers, rewards,
//                        outputs; the episode accumulators are updated with fire-and-forget REDs.
//                        Envs whose moves are contested (a few %) are resolved by the whole warp, lane =
//                        agent, with the literal reference ordering (resolve_moves_slow).
//   grid_obs_kernel      one WARP per env, 24 warps per SM.  Each warp keeps the padded map tile T AND its transpose T2 in
//                        shared memory for its whole life: per env it rewrites only the dynamic cells (apple / waste
//                        points, from the masks) and the agents' cells, runs the spawn (ballot ranks over mask words, one
//                        interleaved two-chain Philox pass), and gathers the n 15x15x3 windows into one bulk async store.
//                        The next env's hot line is prefetched (one coalesced 128-byte load) meanwhile.  HBM-bound part.
//   grid_reward_kernel   harvest only: the contract transfer needs total_close_apples of the post-spawn
//                        map, so transfers / rewards / header run after grid_obs_kernel (thread per env).
//
// Per-agent results travel between the kernels in a u32 [E][8] scratch array (RS_* fields).
// Reference behaviour restated here: see the citations in ssd_grid.cuh (same functions, same order).
#pragma once
#include "ssd_grid.cuh"

#ifndef LOGIC_THREADS
#define LOGIC_THREADS 128
#endif
#ifndef LOGIC_MIN_BLOCKS
#define LOGIC_MIN_BLOCKS 7    // 7 x 128 = 896 threads per SM: the E / 148 = 886 envs of the headline batch in one wave, 72 registers
#endif
#define LOGIC_WARPS (LOGIC_THREADS / 32)
#ifndef OBS_WARPS
#define OBS_WARPS 8           // observe kernel: 3 CTAs of 8 warps per SM (~8.4 KB shared memory per warp, <= 80 registers)
#endif
#ifndef OBS_MAXREG
#define OBS_MAXREG 80
#endif

// per-(agent, env) result word
#define RS_CLEANED_MASK 3u          // bits 0-1  cleaned_squares (0..3)
#define RS_EATEN 4u                 // bit 2     eaten_apples (stale list)
#define RS_EATEN_CLOSE 8u           // bit 3     eaten_close_apples
#define RS_CLOSE_SHIFT 4            // bits 4-8  total_close_apples (0..21)
#define RS_REWARD_SHIFT 16          // bits 16-31 reward accumulator (int16)

__device__ __forceinline__ int rc_off(uint32_t rc, int Wp) { return (int)(rc & 255u) * Wp + (int)((rc >> 8) & 255u); }
__device__ __forceinline__ uint32_t rc_lex(uint32_t rc) { return ((rc & 255u) << 8) | ((rc >> 8) & 255u); }
__device__ __forceinline__ int ori_dr(int d) { return d == ORI_UP ? -1 : (d == ORI_DOWN ? 1 : 0); }
__device__ __forceinline__ int ori_dc(int d) { return d == ORI_RIGHT ? 1 : (d == ORI_LEFT ? -1 : 0); }

// bit `idx` of a lane-strided mask array in shared memory (word w of this thread's env at mk[w * 32])
__device__ __forceinline__ uint32_t mask_bit(const uint32_t* mk, uint32_t idx) { return (mk[(idx >> 5) * 32] >> (idx & 31u)) & 1u; }
// does the cell with static word c hold an apple / waste?  (branch-free: the list bit ANDed with "is such a point")
__device__ __forceinline__ uint32_t cell_has(const uint32_t* mk, uint32_t c, int kind_shift) { return (c >> kind_shift) & mask_bit(mk, c & CI_IDX); }

// count_apples_in_radius(5, loc) (explicit bounds): harvest_new.py:326-336
__device__ __noinline__ int g2_count_r5(const uint16_t* ci, const uint32_t* amk, int row, int col, int H, int W, int Wp)
{
    int cnt = 0;
#pragma unroll
    for (int dr = -2; dr <= 2; dr++)
#pragma unroll
        for (int dc = -2; dc <= 2; dc++)
            if (dr * dr + dc * dc <= 5) {
                int r = row + dr, c = col + dc;
                if ((unsigned)r < (unsigned)H && (unsigned)c < (unsigned)W) cnt += (int)cell_has(amk, ci[r * Wp + c], 14);
            }
    return cnt;
}

// one shooter's beam (update_map_fire, map_env.py:721-814).
//
// In the shooter's frame (along = steps in the firing direction, across = steps to its right) the three rays are
//   centre  across  0, along 1..5      right  across +1, along 0..4      left  across -1, along 0..4
// (firing_points :766-779: the side rays start beside the shooter).  Which agents stand on a ray cell is found per
// AGENT, not per cell: with x = (drow + 64) | (dcol + 64) << 8 relative to the shooter, one PRMT (selector by
// orientation) over x and 0x8080 - x gives y = (along + 64) | (across + 64) << 8, and z = y - 0x3F40 is
// along (left ray), 0x100 + along (centre) or 0x200 + along (right) exactly for the agents on a ray: bit
// (z & 7) + 8 (z >> 8) of a 32-bit occupancy mask.  The 15 ray cells' static words come from the shared-memory cell table
// (cells outside the map count as walls), waste from the env's mask, so a ray is walked with three 5-bit masks: a ray
// stops at its first wall / agent / (CLEAN beam) waste cell (:785-805).  The rays are distinct lines, so applying
// H -> R immediately equals the reference's deferred `updates` list.  Returns the number of cleaned cells.
#define RAY_L 0            // mask bit of cell i of the left / centre / right ray: RAY_x + i (centre: along = i + 1)
#define RAY_C 9
#define RAY_R 16

// Agent.hit for the agents' cell `bit` of the occupancy mask: the highest index wins duplicates (agent_by_pos)
__device__ __noinline__ void g2_hit(const uint32_t* ags /* lane-strided */, int n, uint32_t* res, uint32_t cs, uint32_t sel, uint32_t bit)
{
    int victim = -1;
    for (int a = 0; a < n; a++) {
        const uint32_t v = ags[a * 32];
        const uint32_t x = (v & 0xFFFFu) + cs, z = __byte_perm(x, 0x8080u - x, sel) - 0x3F40u;
        if ((z & 0xFFFFFCF8u) == 0u && ((z & 7u) | ((z >> 5) & 0x18u)) == bit) victim = a;
    }
    if (victim >= 0) res[victim * 32] -= 50u << RS_REWARD_SHIFT;            // Agent.hit(b"F"): -50 (Agent.py:224-226)
}

__device__ __forceinline__ int g2_fire(const uint4* btab, int mwords, uint32_t* wmk, uint8_t* beam, uint32_t shooter, const uint32_t (&agc)[SSD_MAXN],
                                       const uint32_t* ags, int n, uint32_t* res, bool clean, int Wp)
{
    const int row = (int)(shooter & 255u), col = (int)((shooter >> 8) & 255u), ori = (int)((shooter >> 16) & 3u);
    // the static part of the beam (which ray cells are walls or outside the map, which are waste points) is a table row
    const uint4* trow = btab + ((size_t)(row * Wp + col) * 4 + ori) * 2;
    const uint4 t0 = __ldg(trow);
    const uint32_t wall = t0.x;
    uint32_t waste = 0;
    uint32_t widx[4] = { t0.y, t0.z, t0.w, 0u };
    if (clean) {
        widx[3] = __ldg(trow + 1).x;
        const uint32_t imask = (uint32_t)(mwords * 32 - 1);
#pragma unroll
        for (int k = 0; k < 15; k++) {
            const uint32_t idx = (widx[k >> 2] >> (8 * (k & 3))) & 255u;
            const int pos = (k < 5 ? RAY_L : (k < 10 ? RAY_C - 5 : RAY_R - 10)) + k;
            waste |= (idx != 255u ? mask_bit(wmk, idx & imask) : 0u) << pos;
        }
    }
    // agents on the rays
    const uint32_t sel = ori == ORI_UP ? 0x3214u : (ori == ORI_DOWN ? 0x3250u : (ori == ORI_RIGHT ? 0x3201u : 0x3245u));
    const uint32_t cs = 0x4040u - (shooter & 0xFFFFu);
    uint32_t occ = 0;
#pragma unroll
    for (int a = 0; a < SSD_MAXN; a++) {
        const uint32_t x = agc[a] + cs;                                       // absent agents (0xFFFF): bits above 15 set
        const uint32_t z = __byte_perm(x, 0x8080u - x, sel) - 0x3F40u;
        const uint32_t b = 1u << ((z & 7u) | ((z >> 5) & 0x18u));
        occ |= (z & 0xFFFFFCF8u) == 0u ? b : 0u;
    }
    occ &= (31u << RAY_L) | (31u << RAY_C) | (31u << RAY_R);
    const uint32_t stop = wall | waste | occ;
    int nup = 0;
#pragma unroll
    for (int b = 0; b < 3; b++) {
        const int sh = b == 0 ? RAY_L : (b == 1 ? RAY_C : RAY_R);
        const uint32_t s5 = (stop >> sh) & 31u;
        const uint32_t f = (s5 & (0u - s5)) << sh;                            // the ray's first stopping cell (0: none)
        if (beam) {                                                            // firing_points -> beam_pos (map_env.py:789,812)
            const int dr = ori_dr(ori), dc = ori_dc(ori);
            const int rr = ori_dr((ori + 1) & 3), rcl = ori_dc((ori + 1) & 3);  // right = clockwise of dir
            const int step = dr * Wp + dc, side = rr * Wp + rcl, base = row * Wp + col;
            const int cnt = f ? __ffs(f) - 1 - sh + ((f & ~wall) ? 1 : 0) : 5; // cells up to and including a non-wall stop
            for (int i = 0; i < cnt; i++)
                beam[base + (b == 0 ? -side : (b == 1 ? step : side)) + i * step] = clean ? (uint8_t)'C' : (uint8_t)'F';
        }
        if (f & ~wall) {
            if (f & waste) {                                                   // CLEAN: H -> R (cleanup_new.py:285-290)
                const int k = 5 * b + __ffs(f) - 1 - sh;                       // the cell's place in the table row
                const uint32_t wk = k < 8 ? (k < 4 ? widx[0] : widx[1]) : (k < 12 ? widx[2] : widx[3]);   // (no dynamic register index)
                const uint32_t c = (wk >> (8 * (k & 3))) & 255u;
                wmk[(c >> 5) * 32] &= ~(1u << (c & 31u));
                nup++;
            }
            if (!clean && (f & occ)) g2_hit(ags, n, res, cs, sel, (uint32_t)(__ffs(f) - 1));
        }
    }
    return nup;
}

// fire-and-forget global reductions (RED): the add happens at the L2, nothing comes back to the thread
__device__ __forceinline__ void red_add(uint32_t* p, uint32_t v)
{
    asm volatile("red.global.add.u32 [%0], %1;" :: "l"(__cvta_generic_to_global(p)), "r"(v) : "memory");
}
__device__ __forceinline__ void red_add(int* p, int v)
{
    asm volatile("red.global.add.s32 [%0], %1;" :: "l"(__cvta_generic_to_global(p)), "r"(v) : "memory");
}
__device__ __forceinline__ void red_add(long long* p, long long v)
{
    asm volatile("red.global.add.u64 [%0], %1;" :: "l"(__cvta_generic_to_global(p)), "l"(v) : "memory");
}
__device__ __forceinline__ void red_add(double* p, double v)
{
    asm volatile("red.global.add.f64 [%0], %1;" :: "l"(__cvta_generic_to_global(p)), "d"(v) : "memory");
}

// ---------------------------------------------------------------------------------------------
// transfers + redistribution + outputs + header accumulators of one env (lane = env).
// rsp[a * rstride]: RS_* word of agent a (incl. total_close for harvest).  contract_list.py:22-27,45-54;
// two_stage_train.py:72-99; cleanup_new.py:213-253 / harvest_new.py:183-224.
template <int KIND>
__device__ __forceinline__ void env_rewards(const GridParams& p, const StepIO& io, int env, uint8_t* hdr,
                                            const uint32_t* rsp, int rstride, double theta, int t)
{
    const int n = p.n;
    const size_t o = (size_t)env * n;
    double rj[SSD_MAXN];
#pragma unroll
    for (int a = 0; a < SSD_MAXN; a++) rj[a] = a < n ? (double)((int)rsp[a * rstride] >> RS_REWARD_SHIFT) : 0.0;
    if (p.reward_mode) {                               // shaped env rewards (map_env.py:289-301) and their f64 episode sums
        double raw_step = 0.0;                         // raw_rewards = ((0 + r0) + r1) + ... (cleanup_new.py:228-232)
        const double tm1s = (double)(t - 1);
#pragma unroll
        for (int a = 0; a < SSD_MAXN; a++) {
            if (a < n) {
                rj[a] = shaped_reward(p.reward_mode, p.alpha, p.beta, n, rsp, rstride, a);
                raw_step = __dadd_rn(raw_step, rj[a]);
                double* xs = reinterpret_cast<double*>(hdr + RO_XSUM) + a;
                double* xt = reinterpret_cast<double*>(hdr + RO_XTSUM) + a;
                *xs = __dadd_rn(*xs, rj[a]);
                *xt = __dadd_rn(*xt, __dmul_rn(tm1s, rj[a]));
            }
        }
        double* xr = reinterpret_cast<double*>(hdr + RO_XRAW);
        *xr = __dadd_rn(*xr, raw_step);
    }
    if (io.base_rew) {
#pragma unroll
        for (int a = 0; a < SSD_MAXN; a++) if (a < n) io.base_rew[o + a] = rj[a];
    }
    // A zero transfer leaves every reward bit-identical (rewards are never -0.0), so it is skipped.
    double total_tr = 0.0;
    if (p.contract != SSD_CONTRACT_NONE) {
        const double nm1 = (double)(n - 1);
        for (int i = 0; i < n; i++) {                  // rolled: one copy of the fp64 division
            {
                const uint32_t w = rsp[i * rstride];
                double tr;
                if (p.contract == SSD_CONTRACT_CLEANUP) tr = __dmul_rn(-theta, (double)(w & RS_CLEANED_MASK));
                else tr = (((w >> RS_CLOSE_SHIFT) & 31u) < 4u && (w & RS_EATEN_CLOSE)) ? theta : 0.0;
                if (io.transfers) io.transfers[o + i] = tr;
                if (tr != 0.0) {
                    const double share = __ddiv_rn(tr, nm1), neg = -tr;
#pragma unroll
                    for (int j = 0; j < SSD_MAXN; j++) rj[j] = __dadd_rn(rj[j], j == i ? neg : share);
                    total_tr = __dadd_rn(total_tr, tr);
                }
            }
        }
    } else if (io.transfers) {
        for (int i = 0; i < n; i++) io.transfers[o + i] = 0.0;
    }
    const int tm1i = t - 1;
    const double tm1 = (double)tm1i;
    uint32_t n_eaten = 0, n_close = 0;
#pragma unroll
    for (int a = 0; a < SSD_MAXN; a++) {
        if (a < n) {
            const uint32_t w = rsp[a * rstride];
            const uint32_t eaten = (w >> 2) & 1u, eclose = (w >> 3) & 1u, cleaned = w & RS_CLEANED_MASK;
            const uint32_t tclose = (w >> RS_CLOSE_SHIFT) & 31u;
            n_eaten += eaten; n_close += eclose;
            if (io.rew) io.rew[o + a] = rj[a];
            if (io.info) reinterpret_cast<uint32_t*>(io.info)[o + a] =
                eaten | ((KIND == SSD_ENV_CLEANUP ? cleaned : eclose) << 8) | (tclose << 16);
        }
    }
    // episode accumulators: fire-and-forget reductions (RED at the L2, no load round trip in this thread's
    // dependency chain).  One add per address and step, so a float64 RED rounds exactly like `*p = *p + x`.  Adding a
    // zero leaves an accumulator bit-identical (sums are never -0.0), so zero terms are skipped.
#pragma unroll
    for (int a = 0; a < SSD_MAXN; a++) {
        if (a < n) {
            const uint32_t w = rsp[a * rstride];
            const int reward = (int)w >> RS_REWARD_SHIFT;
            if (reward != 0 && !p.reward_mode) {
                red_add(reinterpret_cast<int*>(hdr + RO_SUM_RAW) + a, reward);
                red_add(reinterpret_cast<long long*>(hdr + RO_TSUM_RAW) + a, (long long)tm1i * reward);
            }
            if (p.contract != SSD_CONTRACT_NONE && rj[a] != 0.0) {
                red_add(reinterpret_cast<double*>(hdr + RO_SUM_TR) + a, rj[a]);
                red_add(reinterpret_cast<double*>(hdr + RO_TSUM_TR) + a, __dmul_rn(tm1, rj[a]));
            }
            const uint32_t da = KIND == SSD_ENV_CLEANUP ? (w & RS_CLEANED_MASK) : ((w >> 2) & 1u), db = (w >> 3) & 1u;
            if (da) red_add(reinterpret_cast<uint32_t*>(hdr + RO_AGENT_A) + a, da);
            if (KIND == SSD_ENV_HARVEST && db) red_add(reinterpret_cast<uint32_t*>(hdr + RO_AGENT_B) + a, db);
        }
    }
    if (n_eaten) red_add(reinterpret_cast<uint32_t*>(hdr + RO_APPLES), n_eaten);
    if (KIND == SSD_ENV_HARVEST && n_close) red_add(reinterpret_cast<uint32_t*>(hdr + RO_LOWDENS), n_close);
    if (total_tr != 0.0) red_add(reinterpret_cast<double*>(hdr + RO_TRANSFERS), total_tr);
    if (io.done) io.done[env] = t == p.horizon ? 1 : 0;
    if (io.c_rew8) {                                   // compact result block (ssd_step_host_async)
        io.c_done[env] = t == p.horizon ? 1 : 0;
        uint32_t lo = 0, hi = 0;
        bool fits = true;
#pragma unroll
        for (int a = 0; a < SSD_MAXN; a++) {
            if (a < n) {
                int v = 0;
                const bool f = reward_fits_i8(rj[a], v);
                fits = fits && f;
                const uint32_t b = (uint32_t)(f ? v : -128) & 255u;
                if (a < 4) lo |= b << (8 * a); else hi |= b << (8 * (a - 4));
            }
        }
        if (n == 8) *reinterpret_cast<uint2*>(io.c_rew8 + o) = make_uint2(lo, hi);       // block offsets are 64-byte aligned
        else
            for (int a = 0; a < n; a++) io.c_rew8[o + a] = (int8_t)(((a < 4 ? lo : hi) >> (8 * (a & 3))) & 255u);
        if (!fits) {
            uint8_t* rec_o = io.c_rec + (size_t)compact_slot(io.c_count) * (8 + 8 * n);
            *reinterpret_cast<int2*>(rec_o) = make_int2(env, 0);
#pragma unroll
            for (int a = 0; a < SSD_MAXN; a++) if (a < n) reinterpret_cast<double*>(rec_o + 8)[a] = rj[a];
        }
    }
}

// =============================================================================================
// LOGIC: one thread per env.  Agent state lives in registers (loops over the n <= 8 agents are fully
// unrolled).  The env's only global-memory input is its hot line; static per-cell words (wall / apple point / waste
// point + list index) sit in shared memory, and so do lane-strided copies of the env's masks and of the per-agent
// arrays for the places that index them dynamically (mask bits by point index, the warp-cooperative contested-move
// resolution, the beam walk).
// dynamic shared memory: [cell_info u16 H*Wp, padded to 16 B][per warp: apple mask [mw][32], waste mask [mw][32]]
// LAY == 1: the handle is the stock cleanup map with 8 agents, CleanupContract, plain rewards (logic_layout_id in ssd_b200.cu):
// the fields below become compile-time constants (the per-agent `a < n` tests fold away, strides become immediates).
#define LOGIC_LAY_CLEANUP8(F) F(n, 8) F(H, 25) F(W, 18) F(Wp, 20) F(mw, 4) F(rec_stride, 512) F(map_bytes, 512) F(reward_mode, 0) \
    F(contract, SSD_CONTRACT_CLEANUP)
#define LOGIC_LAY_HARVEST4(F) F(n, 4) F(H, 16) F(W, 38) F(Wp, 40) F(mw, 8) F(rec_stride, 512) F(map_bytes, 640) F(reward_mode, 0) \
    F(contract, SSD_CONTRACT_HARVEST_LOCAL)
template <int KIND, int LAY>
__global__ void __launch_bounds__(LOGIC_THREADS, LOGIC_MIN_BLOCKS) grid_logic_kernel(const GridParams p_in, const StepIO io, uint32_t* __restrict__ res_g)
{
    GridParams p_pin;
    if (LAY == 1) {
        p_pin = p_in;
#define LOGIC_PIN(field, value) p_pin.field = (value);
        LOGIC_LAY_CLEANUP8(LOGIC_PIN)
#undef LOGIC_PIN
        p_pin.beam = nullptr;                                     // the specialised variants are not launched while beams are recorded
    }
    if (LAY == 2) {
        p_pin = p_in;
#define LOGIC_PIN(field, value) p_pin.field = (value);
        LOGIC_LAY_HARVEST4(LOGIC_PIN)
#undef LOGIC_PIN
        p_pin.beam = nullptr;
    }
    const GridParams& p = LAY != 0 ? p_pin : p_in;
    __shared__ uint32_t s_arr[LOGIC_WARPS][4][SSD_MAXN * 32];     // per warp: agents, results, move targets, beam keys
    extern __shared__ __align__(16) uint8_t dsm[];
    pdl_launch_dependents();                                      // the observe kernel's CTAs may take the SM slots this grid frees
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = p.n, H = p.H, W = p.W, Wp = p.Wp, mw = p.mw;
    const int ci_bytes = (H * Wp * 2 + 15) & ~15;
    const uint16_t* ci = reinterpret_cast<const uint16_t*>(dsm);
    for (int i = threadIdx.x; i < (ci_bytes >> 2); i += LOGIC_THREADS)
        reinterpret_cast<uint32_t*>(dsm)[i] = __ldg(reinterpret_cast<const uint32_t*>(p.cell_info) + i);
    pdl_wait();                                                   // the actions (and the records) come from the preceding kernels
    uint32_t* amk = reinterpret_cast<uint32_t*>(dsm + ci_bytes) + warp * 2 * mw * 32 + lane;
    uint32_t* wmk = amk + mw * 32;
    uint32_t* agA = s_arr[warp][0]; uint32_t* mvA = s_arr[warp][2];
    uint32_t* ags = agA + lane; uint32_t* res = s_arr[warp][1] + lane; uint32_t* mvs = mvA + lane; uint32_t* key = s_arr[warp][3] + lane;
    const bool act_lane = lane < n;
    const int env0 = blockIdx.x * LOGIC_THREADS + warp * 32;       // first env of this warp
    const bool valid = env0 + lane < p.E;
    const int env = valid ? env0 + lane : p.E - 1;
    uint8_t* hdr = p.state + (size_t)env * p.rec_stride;           // this env's record

    int t = 0, hcount = 0; uint32_t episode = 0, flags = 0; double theta = 0.0;
    uint32_t err = 0, movers = 0, firem = 0, cleanm = 0;
    uint32_t ag[SSD_MAXN], tg[SSD_MAXN];
    uint32_t act_lo = 0x04040404u, act_hi = 0x04040404u;
    bool slow = false;
    if (valid) {
        const uint4 a0 = *reinterpret_cast<const uint4*>(hdr + RO_AGENTS);
        const uint4 a1 = *reinterpret_cast<const uint4*>(hdr + RO_AGENTS + 16);
        const uint4 s0 = *reinterpret_cast<const uint4*>(hdr + RO_T);        // t, episode, theta
        const uint2 s1 = *reinterpret_cast<const uint2*>(hdr + RO_FLAGS);    // flags, hcount
        for (int k = 0; k < mw; k += 4) {
            const uint4 ma = *reinterpret_cast<const uint4*>(hdr + RO_AMASK + 4 * k);
            amk[k * 32] = ma.x; amk[(k + 1) * 32] = ma.y; amk[(k + 2) * 32] = ma.z; amk[(k + 3) * 32] = ma.w;
            if (KIND == SSD_ENV_CLEANUP) {
                const uint4 mq = *reinterpret_cast<const uint4*>(hdr + RO_WMASK + 4 * k);
                wmk[k * 32] = mq.x; wmk[(k + 1) * 32] = mq.y; wmk[(k + 2) * 32] = mq.z; wmk[(k + 3) * 32] = mq.w;
            }
        }
        ag[0] = a0.x; ag[1] = a0.y; ag[2] = a0.z; ag[3] = a0.w; ag[4] = a1.x; ag[5] = a1.y; ag[6] = a1.z; ag[7] = a1.w;
        t = (int)s0.x + 1;                                                    // map_env.py:230
        episode = s0.y;
        theta = __hiloint2double((int)s0.w, (int)s0.z);
        flags = s1.x; hcount = (int)s1.y;
        // ---- packed action ids
        const uint8_t* g_act = io.actions + (size_t)env * n;
        if (n == 8 && (reinterpret_cast<uintptr_t>(io.actions) & 7u) == 0) {
            const uint2 a = *reinterpret_cast<const uint2*>(g_act); act_lo = a.x; act_hi = a.y;
        } else {
            for (int a = 0; a < n; a++) {
                const uint32_t b = g_act[a];
                if (a < 4) act_lo = (act_lo & ~(255u << (8 * a))) | (b << (8 * a));
                else act_hi = (act_hi & ~(255u << (8 * (a - 4)))) | (b << (8 * (a - 4)));
            }
        }
    }
    __syncthreads();                                             // the cell table is in place
    if (valid) {
        // ---- decode, rotations (map_env.py:514-516), candidate cells (Agent.py:8-16,161-162,198-199)
        uint32_t cand[SSD_MAXN];
        uint32_t want = 0;                                       // movers with a real candidate cell inside the map
#pragma unroll
        for (int a = 0; a < SSD_MAXN; a++) {
            cand[a] = 0;
            if (a < n) {
                const uint32_t v = ag[a];
                const int row = (int)(v & 255u), col = (int)((v >> 8) & 255u);
                int ori = (int)((v >> 16) & 3u);
                const int act = (int)(((a < 4 ? act_lo : act_hi) >> (8 * (a & 3))) & 255u);
                if (act <= 4) {
                    movers |= 1u << a;
                    if (act < 4) {
                        // egocentric -> world direction: LEFT ori+3, RIGHT ori+1, UP ori, DOWN ori+2 (rotate_action :844-853)
                        const int d = (ori + ((0x2013 >> (4 * act)) & 3)) & 3;
                        const int nr = row + ori_dr(d), nc = col + ori_dc(d);
                        if ((unsigned)nr < (unsigned)H && (unsigned)nc < (unsigned)W) {
                            want |= 1u << a;
                            cand[a] = (uint32_t)nr | ((uint32_t)nc << 8);
                        }
                    }
                } else if (act == 5) ori = (ori + 1) & 3;                            // TURN_CLOCKWISE
                else if (act == 6) ori = (ori + 3) & 3;                              // TURN_COUNTERCLOCKWISE
                else if (KIND == SSD_ENV_HARVEST) { if (act == 7) firem |= 1u << a; else { err |= 8; movers |= 1u << a; } }
                else if (act == 7) cleanm |= 1u << a;
                else if (act == 8) firem |= 1u << a;
                else { err |= 8; movers |= 1u << a; }
                ag[a] = (v & 0xFFFFu) | ((uint32_t)ori << 16);
            }
        }
#pragma unroll
        for (int a = 0; a < SSD_MAXN; a++)                       // return_valid_pos (Agent.py:111-119): walls are static
            tg[a] = (((want >> a) & 1u) && !(ci[rc_off(cand[a], Wp)] & CI_WALL)) ? cand[a] : (ag[a] & 0xFFFFu);
        // ---- fast path test: no two movers share a target and no real move targets an occupied cell
#pragma unroll
        for (int a = 0; a < SSD_MAXN; a++) {
            if ((movers >> a) & 1u) {
                const bool real = tg[a] != (ag[a] & 0xFFFFu);
#pragma unroll
                for (int b = 0; b < SSD_MAXN; b++) {
                    if (b == a || b >= n) continue;
                    if (b > a && ((movers >> b) & 1u) && tg[b] == tg[a]) slow = true;
                    if (real && (ag[b] & 0xFFFFu) == tg[a]) slow = true;
                }
            }
        }
        if (!slow) {
#pragma unroll
            for (int a = 0; a < SSD_MAXN; a++)
                if ((movers >> a) & 1u) ag[a] = (ag[a] & 0xFFFF0000u) | tg[a];
        }
#pragma unroll
        for (int a = 0; a < SSD_MAXN; a++) { ags[a * 32] = ag[a]; mvs[a * 32] = tg[a]; res[a * 32] = 0u; }
    }
    __syncwarp();
    // ---- contested moves: the literal reference ordering, one env at a time, lane = agent
    unsigned slowm = __ballot_sync(FULL, slow);
    while (slowm) {
        const int r = __ffs(slowm) - 1; slowm &= slowm - 1;
        const uint32_t movers_r = __shfl_sync(FULL, movers, r);
        const uint32_t ep_r = __shfl_sync(FULL, episode, r), t_r = (uint32_t)__shfl_sync(FULL, t, r);
        uint32_t v = 0; int ao = 0, tgt = 0; bool has_move = false;
        if (act_lane) {
            v = agA[lane * 32 + r];
            ao = (int)rc_lex(v);                             // lexicographic (row, col) cell id
            has_move = (movers_r >> lane) & 1u;
            tgt = has_move ? (int)rc_lex(mvA[lane * 32 + r]) : ao;
        }
        const uint32_t mval = has_move ? (uint32_t)tgt : (0xFFFF0000u | (uint32_t)lane);
        const unsigned same = __match_any_sync(FULL, mval);              // all lanes: not under a short-circuit
        const bool contested = has_move && (__popc(same) > 1);
        const uint32_t rr = resolve_moves_slow(lane, n, p.seed, p.first_env_id + (uint32_t)(env0 + r), ep_r, t_r,
                                               ao, has_move, tgt, movers_r, contested);
        if (act_lane) agA[lane * 32 + r] = (v & 0xFFFF0000u) | rc_lex(rr & 0xFFFFu);
        const uint32_t e2 = __reduce_or_sync(FULL, rr >> 16);
        if (lane == r) err |= e2;
    }
    __syncwarp();
    if (!valid) return;
    if (slow) {
#pragma unroll
        for (int a = 0; a < SSD_MAXN; a++) ag[a] = ags[a * 32];
    }

    // ---- cells under the agents: stale-list infos on the start-of-step map (cleanup_new.py:220-223,
    //      harvest_new.py:190-199), then consume in agent order (map_env.py:244-247): of co-located
    //      agents the lowest index eats
    uint32_t on_apple = 0, first = 0;
    uint32_t agc[SSD_MAXN];                                  // agents' cells for the beams (absent: 0xFFFF)
#pragma unroll
    for (int a = 0; a < SSD_MAXN; a++) agc[a] = a < n ? (ag[a] & 0xFFFFu) : 0xFFFFu;
#pragma unroll
    for (int a = 0; a < SSD_MAXN; a++) {
        if (a < n) {
            on_apple |= cell_has(amk, ci[rc_off(ag[a], Wp)], 14) << a;
            bool dup = false;
#pragma unroll
            for (int b = 0; b < a; b++) if ((ag[b] & 0xFFFFu) == (ag[a] & 0xFFFFu)) dup = true;
            if (!dup) first |= 1u << a;
        }
    }
    bool dirty = false;
    if (on_apple) {
        const bool stale_ok = !(flags & RF_STALE_EMPTY);
        for (uint32_t m = on_apple; m; m &= m - 1) {
            const int a = __ffs(m) - 1;
            const uint32_t v = ags[a * 32];
            uint32_t rs = 0;
            if (stale_ok) {
                rs = RS_EATEN;
                if (KIND == SSD_ENV_HARVEST &&
                    g2_count_r5(ci, amk, (int)(v & 255u), (int)((v >> 8) & 255u), H, W, Wp) < 4) rs |= RS_EATEN_CLOSE;
            }
            if ((first >> a) & 1u) rs += 1u << RS_REWARD_SHIFT;
            res[a * 32] = rs;
        }
        for (uint32_t m = on_apple & first; m; m &= m - 1) {
            const int a = __ffs(m) - 1;
            const uint32_t c = ci[rc_off(ags[a * 32], Wp)];
            amk[((c & CI_IDX) >> 5) * 32] &= ~(1u << (c & 31u));
        }
        dirty = true;
    }
    // ---- beams in shuffled agent order (map_env.py:678-693); keys only matter when >= 2 agents fire
    uint32_t rem = firem | cleanm;
    int ncleaned = 0;
    if (rem) {
        const bool multi = (rem & (rem - 1)) != 0;
        if (multi) {
            for (int b = 0; b < 2; b++)
                if (rem & (0xFu << (4 * b))) {
                    const uint4 q = draw_block_ool(p.seed, p.first_env_id + (uint32_t)env, episode, (uint32_t)t,
                                                   SITE_BEAM_ORDER, (uint32_t)b);
                    key[(4 * b) * 32] = q.x; key[(4 * b + 1) * 32] = q.y; key[(4 * b + 2) * 32] = q.z; key[(4 * b + 3) * 32] = q.w;
                }
        }
        while (rem) {
            int s = __ffs(rem) - 1;
            if (multi) {
                uint32_t best = key[s * 32];
                for (uint32_t m2 = rem & (rem - 1); m2; m2 &= m2 - 1) {
                    const int a = __ffs(m2) - 1;
                    const uint32_t kk = key[a * 32];
                    if (kk < best) { best = kk; s = a; }
                }
            }
            rem &= ~(1u << s);
            const bool clean = (cleanm >> s) & 1u;
            const int nup = g2_fire(p.beam_tab, mw, wmk, p.beam ? p.beam + (size_t)env * p.map_bytes : nullptr, ags[s * 32], agc, ags, n, res, clean, Wp);
            if (clean) { res[s * 32] |= (uint32_t)nup; ncleaned += nup; }
            else res[s * 32] -= 1u << RS_REWARD_SHIFT;                    // fire cost (Agent.py:217-219)
        }
    }
    if (KIND == SSD_ENV_CLEANUP) hcount -= ncleaned;

    // ---- hot line back (the observe kernel reads agents, t, episode, flags, hcount, masks from it)
    *reinterpret_cast<uint4*>(hdr + RO_AGENTS) = make_uint4(ag[0], ag[1], ag[2], ag[3]);
    *reinterpret_cast<uint4*>(hdr + RO_AGENTS + 16) = make_uint4(ag[4], ag[5], ag[6], ag[7]);
    *reinterpret_cast<int*>(hdr + RO_T) = t;
    *reinterpret_cast<uint2*>(hdr + RO_FLAGS) =
        make_uint2((flags & ~RF_STALE_EMPTY) | (err ? (err << RF_ERR_SHIFT) : 0u), (uint32_t)hcount);
    if (dirty)
        for (int k = 0; k < mw; k += 4)
            *reinterpret_cast<uint4*>(hdr + RO_AMASK + 4 * k) = make_uint4(amk[k * 32], amk[(k + 1) * 32], amk[(k + 2) * 32], amk[(k + 3) * 32]);
    if (KIND == SSD_ENV_CLEANUP && ncleaned) {
        for (int k = 0; k < mw; k += 4)
            *reinterpret_cast<uint4*>(hdr + RO_WMASK + 4 * k) = make_uint4(wmk[k * 32], wmk[(k + 1) * 32], wmk[(k + 2) * 32], wmk[(k + 3) * 32]);
        red_add(reinterpret_cast<uint32_t*>(hdr + RO_DIRT), (uint32_t)ncleaned);
    }
    uint4* rg = reinterpret_cast<uint4*>(res_g + (size_t)env * SSD_MAXN);
    rg[0] = make_uint4(res[0], res[32], res[64], res[96]);
    rg[1] = make_uint4(res[128], res[160], res[192], res[224]);
    // cleanup: nothing below depends on the spawn, so rewards / outputs are finished here
    if (KIND == SSD_ENV_CLEANUP) env_rewards<KIND>(p, io, env, hdr, res, 32, theta, t);
}

// harvest: rewards after the observe kernel has added total_close_apples to the result words
__global__ void __launch_bounds__(LOGIC_THREADS) grid_reward_kernel(const GridParams p, const StepIO io, const uint32_t* __restrict__ res_g)
{
    pdl_launch_dependents();                          // (auto_reset) the masked reset kernel may set up meanwhile
    pdl_wait();                                       // total_close_apples come from the observe kernel
    const int env = blockIdx.x * LOGIC_THREADS + threadIdx.x;
    if (env >= p.E) return;
    uint8_t* hdr = p.state + (size_t)env * p.rec_stride;
    const int t = *reinterpret_cast<const int*>(hdr + RO_T);
    const double theta = *reinterpret_cast<const double*>(hdr + RO_THETA);
    env_rewards<SSD_ENV_HARVEST>(p, io, env, hdr, res_g + (size_t)env * SSD_MAXN, 1, theta, t);
}

// ---------------------------------------------------------------------------------------------
// Observation gather of the observe kernel.  The kernel is bound by shared-memory wavefronts and instruction issue, so
// an output row is read as 5 aligned WORDS: every output row of color_view (map_env.py:397-411) is a run of 15
// consecutive bytes, forwards or backwards, either of the row-major tile T (UP, DOWN) or of its transpose T2 (LEFT, RIGHT):
//   UP    out[i][j] = V[i][j]        T : run at origin  + i S,          forwards
//   DOWN  out[i][j] = V[14-i][14-j]  T : run at origin  + (14 - i) S,   backwards
//   LEFT  out[i][j] = V[j][14-i]     T2: run at origin2 + (14 - i) S2,  forwards
//   RIGHT out[i][j] = V[14-j][i]     T2: run at origin2 + i S2,         backwards
// with V[a][b] = T[origin + a S + b] = T2[origin2 + b S2 + a].  T2 is not rebuilt per env: both tiles live in the warp's
// shared memory for the whole kernel and only their dynamic cells are rewritten (apply_masks, paint).
// ao: the agent's cell in T.  `tile` is the base of [T | T2]; vdesc entries hold offsets relative to it.
__device__ __forceinline__ void gather_obs2(const GridParams& p, int lane, const uint8_t* tile, uint8_t* stage,
                                            const uint32_t* sm_pal, int4* vdesc, int ao, int ori, uint8_t* gdst)
{
    const int n = p.n;
    const int L = n * SSD_OBS_BYTES;
    const uint32_t gaddr = (uint32_t)(reinterpret_cast<uintptr_t>(gdst) & 15u);
    const bool word_ok = (gaddr & 3u) == 0;
    const int shift = word_ok ? (int)gaddr : 0;          // staged stream is congruent to gdst modulo 16
    uint32_t* sw = reinterpret_cast<uint32_t*>(stage + shift);
    if (lane < n) vdesc[lane] = view_desc2(p, ao, ori);
    if (lane == 0) bulk_wait_read<0>();                  // the previous env's store has drained `stage`
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
            uint32_t bw[4];
            run_bytes15(tile, d.x + i * d.y, d.z, bw);        // the row's 15-byte run (lowest byte d.x + i d.y)
#pragma unroll
            for (int j = 0; j < SSD_OBSW; j++)               // a tile byte IS the byte offset of its palette entry
                col[15 * q + j] = *reinterpret_cast<const uint32_t*>(
                    reinterpret_cast<const uint8_t*>(sm_pal) + __byte_perm(bw[j >> 2], 0u, 0x4440u + (uint32_t)(j & 3)));
        }
        uint32_t* dst = sw + 45 * lane;
#pragma unroll
        for (int g4 = 0; g4 < 15; g4++) pack4(dst + 3 * g4, col[4 * g4], col[4 * g4 + 1], col[4 * g4 + 2], col[4 * g4 + 3]);
    }
    obs_stream_store(lane, stage, shift, word_ok, L, gdst);
}

// =============================================================================================
// OBSERVE: one warp per env.  Spawn + observation windows.  Per warp: [T | T2 | stage (obs staging, aliased
// by the spawn scratch) | misc].  Lane l prefetches word l of the NEXT env's hot line (one coalesced 128-byte load) while
// the current env is processed: words 0-7 agents, 8 t, 9 episode, 12 flags, 13 #waste, 16.. apple mask, 24.. waste mask.
// LAY: 0 = every layout value is read from the kernel parameters; 1 = the handle was checked (obs_layout_id in ssd_b200.cu) to be
// the stock cleanup map with 8 agents, and the layout values below are compile-time constants for the optimiser (row
// strides become shifts / immediates, the per-agent loops lose their bounds): same code, fewer instructions and registers.
#define OBS_LAY_CLEANUP8(F) F(S, 36) F(S2, 44) F(tile2_off, 1408) F(g2_stage, 2912) F(g2_misc, 8336) F(g2_warp_bytes, 8464) \
    F(sm_thr, 64) F(sm_won, 544) F(sm_apple_rc, 672) F(sm_waste_rc, 880) F(sm_warp0, 1120) F(n, 8) F(obs_items, 30) \
    F(n_apple, 103) F(n_waste, 119) F(rec_stride, 512) F(H, 25) F(W, 18) F(Wp, 20)
// LAY == 2: the stock harvest map with 4 agents (BASELINE configs[1])
#define OBS_LAY_HARVEST4(F) F(S, 56) F(S2, 32) F(tile2_off, 1696) F(g2_stage, 3440) F(g2_misc, 6512) F(g2_warp_bytes, 6640) \
    F(sm_thr, 64) F(sm_won, 80) F(sm_apple_rc, 96) F(sm_waste_rc, 416) F(sm_warp0, 416) F(n, 4) F(obs_items, 15) \
    F(n_apple, 155) F(n_waste, 0) F(rec_stride, 512) F(H, 16) F(W, 38) F(Wp, 40)
// FORM: the observation form (OBS_U8: uint8 windows at io.obs; a policy form: the policy's image tensor, io.obs_stride bytes per env).
template <int KIND, int MW, bool FEAT, int LAY, int FORM = OBS_U8>
__global__ void __maxnreg__(OBS_MAXREG) grid_obs_kernel(const GridParams p_in, const StepIO io_in, uint32_t* __restrict__ res_g)
{
    GridParams p_pin; StepIO io_pin;                  // LAY == 1: a copy (scalar-replaced by the compiler) with the layout fields pinned
    if (LAY == 1) {
        p_pin = p_in; io_pin = io_in;
#define OBS_PIN(field, value) p_pin.field = (value);
        OBS_LAY_CLEANUP8(OBS_PIN)
#undef OBS_PIN
        p_pin.s_magic = 119304648u;
        io_pin.obs_stride = 5400 * (int)sizeof(typename ObsForm<FORM>::T);
    }
    if (LAY == 2) {
        p_pin = p_in; io_pin = io_in;
#define OBS_PIN(field, value) p_pin.field = (value);
        OBS_LAY_HARVEST4(OBS_PIN)
#undef OBS_PIN
        p_pin.s_magic = 76695845u;
        io_pin.obs_stride = 2700 * (int)sizeof(typename ObsForm<FORM>::T);
    }
    const GridParams& p = LAY != 0 ? p_pin : p_in;
    const StepIO& io = LAY != 0 ? io_pin : io_in;
    extern __shared__ __align__(16) uint8_t smem[];
    const SharedTables tb = load_shared_tables(p, smem, FEAT);
    if constexpr (FORM != OBS_U8) load_policy_palette<typename ObsForm<FORM>::T>(p);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* tile = smem + p.sm_warp0 + warp * p.g2_warp_bytes;
    uint8_t* tile2 = tile + p.tile2_off;
    uint8_t* stage = tile + p.g2_stage;
    uint32_t* scratch = reinterpret_cast<uint32_t*>(stage);
    int4* vdesc = reinterpret_cast<int4*>(tile + p.g2_misc + MISC_VDESC);
    const PointRegs<MW> pr = load_point_regs<MW>(p, lane);
    init_warp_tiles(p, tile, lane);
    __syncthreads();                                  // tables visible
    const int n = p.n, S = p.S, S2 = p.S2;
    const bool act_lane = lane < n;
    const int env_stride = gridDim.x * OBS_WARPS;
    const uint32_t rot3 = (uint32_t)(lane - 3) & 31u, rot2 = (uint32_t)(lane - 2) & 31u;

    // Schedule.  An env costs 3-7 us depending on whether its spawn is active, and a one-wave persistent grid ends with its
    // slowest warp (ncu, static schedule: 21 of 24 resident warps active on average).  So every warp takes its first
    // obs_static_iters envs from the static grid-stride schedule and the rest, one at a time, from a global counter
    // (requested two envs ahead, so the atomic's latency hides behind an env's work; the last CTA to finish rearms it).
    const int nwarps = env_stride, wid = blockIdx.x * OBS_WARPS + warp;
    const int dyn0 = p.obs_static_iters * nwarps;          // first env of the dynamic pool
    int it = 0;
    auto next_env = [&]() -> int {
        int e;
        if (it < p.obs_static_iters) e = wid + it * nwarps;
        else {
            e = 0;
            if (lane == 0) e = dyn0 + (int)atomicAdd(p.obs_ctr, 1u);
            e = __shfl_sync(FULL, e, 0);
        }
        it++;
        return e;
    };
    pdl_launch_dependents();                                   // the masked reset behind the step (auto_reset) may set up early
    pdl_wait();                                                // the hot lines are the logic kernel's output
    int env = next_env(), env_n = next_env();
    uint32_t hw_next = 0;
    if (env < p.E) hw_next = reinterpret_cast<const uint32_t*>(p.state + (size_t)env * p.rec_stride)[lane];
    for (; env < p.E; env = env_n, env_n = next_env()) {
        uint8_t* g_rec = p.state + (size_t)env * p.rec_stride;
        uint8_t* g_obs = io.obs + (size_t)env * (size_t)io.obs_stride;
        const uint32_t hw = hw_next;
        if (env_n < p.E) hw_next = reinterpret_cast<const uint32_t*>(p.state + (size_t)env_n * p.rec_stride)[lane];
        // ---- dynamic cells of T and T2 from the masks; header scalars
        uint32_t am[MW], wm[MW];
#pragma unroll
        for (int q = 0; q < MW; q++) {
            am[q] = __shfl_sync(FULL, hw, RO_AMASK / 4 + q);
            wm[q] = KIND == SSD_ENV_CLEANUP ? __shfl_sync(FULL, hw, RO_WMASK / 4 + q) : 0u;
        }
        apply_masks<MW, true>(p, tile, pr, am, wm, rot3, rot2);
        const uint32_t t = __shfl_sync(FULL, hw, RO_T / 4);               // already incremented by the logic kernel
        const uint32_t episode = __shfl_sync(FULL, hw, RO_EPISODE / 4);
        int hcount = (int)__shfl_sync(FULL, hw, RO_HCOUNT / 4);
        const EnvRng g = { p.seed, p.first_env_id + (uint32_t)env, episode, t };
        int ao = 0, ao2 = 0, ori = 0;
        if (act_lane) {
            const int row = (int)(hw & 255u), col = (int)((hw >> 8) & 255u);
            ao = (row + SSD_VIEW) * S + 8 + col;
            ao2 = (col + SSD_VIEW) * S2 + 8 + row;
            ori = (int)((hw >> 16) & 3u);
        }
        __syncwarp();
        uint32_t old = 0;
        if (act_lane) {                               // spawn eligibility: "no agent there" (co-located lanes write the same value)
            old = tile[ao] & CODE_MASK;
            tile[ao] = (uint8_t)(old | OCC_BIT);
        }
        __syncwarp();
        // ---- spawn
        bool changed = false;
#ifndef OBS_SKIP_SPAWN         // OBS_SKIP_*: timing experiments only (tools/sweep_obs_parts.sh), results are wrong
        if (KIND == SSD_ENV_CLEANUP) {
            if (cleanup_spawn_active(tb, hcount)) {
                if (lane == 0) bulk_wait_read<0>();   // the previous observation store has drained `stage` (= scratch)
                __syncwarp();
                changed = cleanup_spawn<MW>(p, tb, lane, tile, true, scratch, g, t, hcount, pr, am, wm);
            }
        } else {
            if (lane == 0) bulk_wait_read<0>();
            __syncwarp();
            changed = harvest_spawn<MW>(p, lane, tile, true, scratch, g, t, pr, am);
        }
        if (changed) {                                // the masks (and #waste) go back only when the spawn changed them
            uint32_t* hot = reinterpret_cast<uint32_t*>(g_rec);
#pragma unroll
            for (int q = 0; q < MW; q++)
                if (lane == q) {
                    hot[RO_AMASK / 4 + q] = am[q];
                    if (KIND == SSD_ENV_CLEANUP) hot[RO_WMASK / 4 + q] = wm[q];
                }
            if (KIND == SSD_ENV_CLEANUP && lane == 0) hot[RO_HCOUNT / 4] = (uint32_t)hcount;
        }
#endif
        int total_close = 0;
        if (KIND == SSD_ENV_HARVEST && act_lane) {
            total_close = count_apples_r5(tile, ao, S);
            res_g[(size_t)env * SSD_MAXN + lane] |= (uint32_t)total_close << RS_CLOSE_SHIFT;
        }
        if (FEAT) {
            const int cleaned = (KIND == SSD_ENV_CLEANUP && act_lane) ? (int)(res_g[(size_t)env * SSD_MAXN + lane] & RS_CLEANED_MASK) : 0;
            write_features<KIND, MW>(p, tb, lane, hw, am, wm, cleaned, total_close, hcount, io.feat + (size_t)env * n * p.F);
        }
        // ---- paint agents in agent order: the highest index wins a shared cell (map_env.py:257-261)
        const unsigned grp = __match_any_sync(FULL, act_lane ? (uint32_t)ao : (0x40000000u | (uint32_t)lane));
        __syncwarp();
        if (act_lane && lane == 31 - __clz(grp)) { tile[ao] = (uint8_t)PAINT_CODE(lane); tile2[ao2] = (uint8_t)PAINT_CODE(lane); }
        __syncwarp();
        // gather_obs2 / gather_policy wait (lane 0) until the previous observation store has drained `stage`, then sync the warp
#ifndef OBS_SKIP_GATHER
        if constexpr (FORM == OBS_U8) gather_obs2(p, lane, tile, stage, tb.pal, vdesc, ao, ori, g_obs);
        else gather_policy<FORM, true>(p, lane, tile, stage, vdesc, ao, ori, g_obs);
#endif
        // the agents' cells back to their code (the gather ends behind a warp barrier after its last tile read)
        if (act_lane) { tile[ao] = (uint8_t)old; tile2[ao2] = (uint8_t)old; }
        __syncwarp();
    }
    if (lane == 0) bulk_wait_read<0>();      // smem must outlive the async bulk reads
    __syncthreads();
    if (threadIdx.x == 0) {                  // every warp of this CTA has taken its last env: rearm the counter behind the last CTA
        __threadfence();
        if (atomicAdd(p.obs_ctr + 1, 1u) == gridDim.x - 1) { p.obs_ctr[0] = 0u; p.obs_ctr[1] = 0u; }
    }
}

// =============================================================================================
// FEATURE FORM (ssd_set_feature_output): the observation is infos['feature_obs'] (cleanup_new.py:235-251,
// harvest_new.py:208-222), written in output form OUT: SSD_FEATURE_F64 (double [E][n][F]) or SSD_POLICY_* (the policy's
// flat rows T [E n][width], features ++ [theta, 0] under a contract).  No observation windows are built.
template <int OUT> struct FeatureElem : PolicyElem<1 + OUT> {};
template <> struct FeatureElem<SSD_FEATURE_F64> { typedef double T; };

// columns F, F + 1 of a policy row under a contract: [theta, 0] (two_stage_train.py:113-121)
template <typename T>
__device__ __forceinline__ void feature_theta_cols(T* rows, const GridParams& p, int lane, int width, double theta)
{
    if (width > p.F && lane < p.n) { feat_put(rows + (size_t)lane * width, p.F, theta); feat_put(rows + (size_t)lane * width, p.F + 1, 0.0); }
}

// STEP, in place of the observe kernel behind the logic kernel: one warp per env, grid-stride.  What the observe kernel
// does for an env apart from painting and the window gather — the env's tile T from the masks, the same spawn on the
// same draws (masks and #waste written back when it changes them), harvest's total_close_apples into res_g for
// grid_reward_kernel — then write_features' values.  Shared memory: the observe kernel's layout (T2 unused).
template <int KIND, int MW, int OUT>
__global__ void __launch_bounds__(OBS_WARPS * 32) grid_feature_kernel(const GridParams p, uint32_t* __restrict__ res_g, void* out, int width)
{
    typedef typename FeatureElem<OUT>::T T;
    extern __shared__ __align__(16) uint8_t smem[];
    const SharedTables tb = load_shared_tables(p, smem, true);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* tile = smem + p.sm_warp0 + warp * p.g2_warp_bytes;
    uint32_t* scratch = reinterpret_cast<uint32_t*>(tile + p.g2_stage);
    const PointRegs<MW> pr = load_point_regs<MW>(p, lane);
    init_warp_tiles(p, tile, lane);
    __syncthreads();                                  // tables visible
    const int n = p.n, S = p.S;
    const bool act_lane = lane < n;
    const uint32_t rot3 = (uint32_t)(lane - 3) & 31u, rot2 = (uint32_t)(lane - 2) & 31u;
    pdl_launch_dependents();                          // the reward / masked reset kernel behind the step may set up early
    pdl_wait();                                       // the hot lines and res_g are the logic kernel's output
    for (int env = blockIdx.x * OBS_WARPS + warp; env < p.E; env += gridDim.x * OBS_WARPS) {
        uint32_t* hot = reinterpret_cast<uint32_t*>(p.state + (size_t)env * p.rec_stride);
        const uint32_t hw = hot[lane];
        uint32_t am[MW], wm[MW];
#pragma unroll
        for (int q = 0; q < MW; q++) {
            am[q] = __shfl_sync(FULL, hw, RO_AMASK / 4 + q);
            wm[q] = KIND == SSD_ENV_CLEANUP ? __shfl_sync(FULL, hw, RO_WMASK / 4 + q) : 0u;
        }
        apply_masks<MW, false>(p, tile, pr, am, wm, rot3, rot2);
        const uint32_t t = __shfl_sync(FULL, hw, RO_T / 4);               // already incremented by the logic kernel
        const uint32_t episode = __shfl_sync(FULL, hw, RO_EPISODE / 4);
        int hcount = (int)__shfl_sync(FULL, hw, RO_HCOUNT / 4);
        const double theta = __hiloint2double((int)__shfl_sync(FULL, hw, RO_THETA / 4 + 1), (int)__shfl_sync(FULL, hw, RO_THETA / 4));
        const EnvRng g = { p.seed, p.first_env_id + (uint32_t)env, episode, t };
        const int ao = act_lane ? ((int)(hw & 255u) + SSD_VIEW) * S + 8 + (int)((hw >> 8) & 255u) : 0;
        __syncwarp();
        uint32_t old = 0;
        if (act_lane) {                               // spawn eligibility: "no agent there" (co-located lanes write the same value)
            old = tile[ao] & CODE_MASK;
            tile[ao] = (uint8_t)(old | OCC_BIT);
        }
        __syncwarp();
        bool changed = false;
        if (KIND == SSD_ENV_CLEANUP) {
            if (cleanup_spawn_active(tb, hcount)) changed = cleanup_spawn<MW>(p, tb, lane, tile, false, scratch, g, t, hcount, pr, am, wm);
        } else {
            changed = harvest_spawn<MW>(p, lane, tile, false, scratch, g, t, pr, am);
        }
        if (changed) {                                // the masks (and #waste) go back only when the spawn changed them
#pragma unroll
            for (int q = 0; q < MW; q++)
                if (lane == q) {
                    hot[RO_AMASK / 4 + q] = am[q];
                    if (KIND == SSD_ENV_CLEANUP) hot[RO_WMASK / 4 + q] = wm[q];
                }
            if (KIND == SSD_ENV_CLEANUP && lane == 0) hot[RO_HCOUNT / 4] = (uint32_t)hcount;
        }
        int total_close = 0, cleaned = 0;
        if (KIND == SSD_ENV_HARVEST && act_lane) {
            total_close = count_apples_r5(tile, ao, S);
            res_g[(size_t)env * SSD_MAXN + lane] |= (uint32_t)total_close << RS_CLOSE_SHIFT;
        }
        if (KIND == SSD_ENV_CLEANUP && act_lane) cleaned = (int)(res_g[(size_t)env * SSD_MAXN + lane] & RS_CLEANED_MASK);
        T* rows = reinterpret_cast<T*>(out) + (size_t)env * n * width;
        write_features<KIND, MW, T>(p, tb, lane, hw, am, wm, cleaned, total_close, hcount, rows, width);
        feature_theta_cols(rows, p, lane, width, theta);
        __syncwarp();                                 // every lane's spawn / count reads of T are done
        if (act_lane) tile[ao] = (uint8_t)old;
        __syncwarp();
    }
}

// RESET ROWS, behind grid_reset_kernel<KIND, 0> (no windows) on the same mask: the reset observation of each reset env from
// its fresh record (GridWorldEnv._reset_feature_obs, cleanup_new.py:193-202, harvest_new.py:160-168).  One warp per env.
//   cleanup: custom_reset fills the apple / waste caches BEFORE the reset-time spawn (map_env.py:319-320): no apples
//            (closest apple [0, 0], 0 apples), the waste list is the map's initial 'H' cells, #waste their count, nothing
//            cleaned;
//   harvest: the map after the reset: the record's apples, count_apples_in_radius(5) (j*j + k*k <= 5) as total_close.
// The theta column (policy rows under a contract) is the record's theta: the negotiated one behind an auto-reset.
template <int KIND, int OUT>
__global__ void __launch_bounds__(GRID_THREADS) grid_reset_features_kernel(const GridParams p, const uint8_t* mask, void* out, int width)
{
    typedef typename FeatureElem<OUT>::T T;
    constexpr int MW = MAX_POINT_ROUNDS;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int env0 = blockIdx.x * GRID_WARPS + warp, estride = gridDim.x * GRID_WARPS;
    const SharedTables tb = { nullptr, nullptr, nullptr, p.apple_rc, p.waste_rc };   // write_features reads only the point lists
    for (int i0 = 0; env0 + (long long)i0 * estride < p.E; i0 += 32) {
        const long long el = env0 + (long long)(i0 + lane) * estride;
        unsigned todo = __ballot_sync(FULL, el < p.E && (!mask || mask[el]));
        while (todo) {
            const int env = env0 + (i0 + __ffs(todo) - 1) * estride;
            todo &= todo - 1;
            const uint32_t hw = reinterpret_cast<const uint32_t*>(p.state + (size_t)env * p.rec_stride)[lane];
            uint32_t am[MW], wm[MW];
#pragma unroll
            for (int q = 0; q < MW; q++) {
                am[q] = KIND == SSD_ENV_HARVEST ? __shfl_sync(FULL, hw, RO_AMASK / 4 + q) : 0u;
                wm[q] = KIND == SSD_ENV_CLEANUP ? p.reset_wmask[q] : 0u;
            }
            int total_close = 0;
            if (KIND == SSD_ENV_HARVEST) {
                const int my_r = (int)(hw & 255u), my_c = (int)((hw >> 8) & 255u);
                for (int a = 0; a < p.n; a++) {
                    const int ar = __shfl_sync(FULL, my_r, a), ac = __shfl_sync(FULL, my_c, a);
                    int cnt = 0;
#pragma unroll
                    for (int q = 0; q < MW; q++) {
                        bool near = false;
                        if ((am[q] >> lane) & 1u) {
                            const uint32_t rc = __ldg(p.apple_rc + lane + 32 * q);
                            const int dr = (int)(rc >> 8) - ar, dc = (int)(rc & 255u) - ac;
                            near = dr * dr + dc * dc <= 5;
                        }
                        cnt += __popc(__ballot_sync(FULL, near));
                    }
                    if (lane == a) total_close = cnt;
                }
            }
            const double theta = __hiloint2double((int)__shfl_sync(FULL, hw, RO_THETA / 4 + 1), (int)__shfl_sync(FULL, hw, RO_THETA / 4));
            T* rows = reinterpret_cast<T*>(out) + (size_t)env * p.n * width;
            write_features<KIND, MW, T>(p, tb, lane, hw, am, wm, 0, total_close, p.n_waste_start, rows, width);
            feature_theta_cols(rows, p, lane, width, theta);
        }
    }
}

// =============================================================================================
// GLOBAL FORM (ssd_set_global_output): the observation is JointEnv's global view, MapEnv.global_view() (map_env.py:394-395;
// global_view_kernel's output), written in output form OUT: SSD_GLOBAL_U8 (uint8 [E][H][W][3]) or SSD_POLICY_* (T
// [E][3][H][W], T(float32(u8 / 255.0)): get_global_obs() as VisionNetwork.forward feeds it).  No observation windows are built.
template <int OUT> struct GlobalElem : PolicyElem<1 + OUT> {};
template <> struct GlobalElem<SSD_GLOBAL_U8> { typedef uint8_t T; };

// One env's view from a map of cell codes (cell (r, c) at m[r * stride + c]; an agent painted as PAINT_CODE; OCC_BIT ignored)
// to `dst`, the env's block.  inv_w = 1.0f / W: (cell + 0.5) * inv_w stays within 4e-4 of the exact quotient for the
// cells of a 48 x 64 map, so its truncation is cell / W.  Stores are coalesced:
//   uint8: the 3 H W bytes as aligned words (lane = word; a word spans two cells: its four bytes are picked from their
//          colours with one byte permute), the unaligned head and tail as bytes — a block starts on any byte;
//   T:     three planes of H W elements, lane = cell, the palette's T entries (load_policy_palette) per channel.
template <int OUT>
__device__ __forceinline__ void write_global_view(const GridParams& p, int lane, const uint8_t* m, int stride, float inv_w,
                                                  const uint32_t* pal, void* dst)
{
    typedef typename GlobalElem<OUT>::T T;
    const int W = p.W, HW = p.H * p.W;
    auto cell_off = [&](int cell, int& c) -> int {
        const int r = __float2int_rz(__fmul_rn(__int2float_rn(cell) + 0.5f, inv_w));
        c = cell - r * W;
        return r * stride + c;
    };
    if constexpr (OUT == SSD_GLOBAL_U8) {
        const uint8_t* pb = reinterpret_cast<const uint8_t*>(pal);     // a code is the byte offset of its palette entry
        uint8_t* g = reinterpret_cast<uint8_t*>(dst);
        const int L = 3 * HW;
        const int head = min((int)((0u - (uint32_t)reinterpret_cast<uintptr_t>(g)) & 3u), L);
        const int nw = (L - head) >> 2, tail0 = head + 4 * nw;
        auto byte_at = [&](int b) -> uint8_t {
            const int cell = (int)(((uint32_t)b * 0xAAABu) >> 17), ch = b - 3 * cell;     // b / 3 for b < 2^17
            int c;
            return pb[(m[cell_off(cell, c)] & CODE_MASK) + ch];
        };
        if (lane < head) g[lane] = byte_at(lane);
        if (lane < L - tail0) g[tail0 + lane] = byte_at(tail0 + lane);
        uint32_t* gw = reinterpret_cast<uint32_t*>(g + head);
        for (int w = lane; w < nw; w += 32) {
            const int b0 = head + 4 * w;
            const int cell = (int)(((uint32_t)b0 * 0xAAABu) >> 17), ch = b0 - 3 * cell;
            int c;
            const int o0 = cell_off(cell, c), o1 = c + 1 < W ? o0 + 1 : o0 - c + stride;   // the next cell (next row's first)
            const uint32_t c0 = pal[(m[o0] & CODE_MASK) >> 2], c1 = pal[(m[o1] & CODE_MASK) >> 2];
            gw[w] = __byte_perm(c0 | (c1 << 24), c1 >> 8, 0x3210u + 0x1111u * (uint32_t)ch);    // bytes ch .. ch + 3 of c0 ++ c1
        }
    } else {
        const T* ppal = policy_palette<T>();
        T* o = reinterpret_cast<T*>(dst);
        for (int cell = lane; cell < HW; cell += 32) {
            int c;
            const int code = m[cell_off(cell, c)] & CODE_MASK;
            o[cell] = ppal[code]; o[HW + cell] = ppal[code + 1]; o[2 * HW + cell] = ppal[code + 2];
        }
    }
}

// STEP, in place of the observe kernel behind the logic kernel: one warp per env, grid-stride.  grid_feature_kernel's env
// work — the env's tile T from the masks, the same spawn on the same draws (masks and #waste written back when it changes
// them), harvest's total_close_apples into res_g for grid_reward_kernel — then the agents painted into T in agent order
// (the highest index wins a shared cell; t > 0 after a step, so they always show) and the view written from T's map rows.
// Shared memory: the observe kernel's layout (T2 unused).  `width` is unused (grid_feature_kernel's signature).
template <int KIND, int MW, int OUT>
__global__ void __launch_bounds__(OBS_WARPS * 32) grid_global_kernel(const GridParams p, uint32_t* __restrict__ res_g, void* out, int width)
{
    typedef typename GlobalElem<OUT>::T T;
    extern __shared__ __align__(16) uint8_t smem[];
    const SharedTables tb = load_shared_tables(p, smem, false);
    if constexpr (OUT != SSD_GLOBAL_U8) load_policy_palette<T>(p);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* tile = smem + p.sm_warp0 + warp * p.g2_warp_bytes;
    uint32_t* scratch = reinterpret_cast<uint32_t*>(tile + p.g2_stage);
    const PointRegs<MW> pr = load_point_regs<MW>(p, lane);
    init_warp_tiles(p, tile, lane);
    __syncthreads();                                  // tables visible
    const int n = p.n, S = p.S;
    const bool act_lane = lane < n;
    const uint32_t rot3 = (uint32_t)(lane - 3) & 31u, rot2 = (uint32_t)(lane - 2) & 31u;
    const float inv_w = __frcp_rn((float)p.W);
    const size_t env_elems = (size_t)3 * p.H * p.W;
    pdl_launch_dependents();                          // the reward / masked reset kernel behind the step may set up early
    pdl_wait();                                       // the hot lines and res_g are the logic kernel's output
    for (int env = blockIdx.x * OBS_WARPS + warp; env < p.E; env += gridDim.x * OBS_WARPS) {
        uint32_t* hot = reinterpret_cast<uint32_t*>(p.state + (size_t)env * p.rec_stride);
        const uint32_t hw = hot[lane];
        uint32_t am[MW], wm[MW];
#pragma unroll
        for (int q = 0; q < MW; q++) {
            am[q] = __shfl_sync(FULL, hw, RO_AMASK / 4 + q);
            wm[q] = KIND == SSD_ENV_CLEANUP ? __shfl_sync(FULL, hw, RO_WMASK / 4 + q) : 0u;
        }
        apply_masks<MW, false>(p, tile, pr, am, wm, rot3, rot2);
        const uint32_t t = __shfl_sync(FULL, hw, RO_T / 4);               // already incremented by the logic kernel
        const uint32_t episode = __shfl_sync(FULL, hw, RO_EPISODE / 4);
        int hcount = (int)__shfl_sync(FULL, hw, RO_HCOUNT / 4);
        const EnvRng g = { p.seed, p.first_env_id + (uint32_t)env, episode, t };
        const int ao = act_lane ? ((int)(hw & 255u) + SSD_VIEW) * S + 8 + (int)((hw >> 8) & 255u) : 0;
        __syncwarp();
        uint32_t old = 0;
        if (act_lane) {                               // spawn eligibility: "no agent there" (co-located lanes write the same value)
            old = tile[ao] & CODE_MASK;
            tile[ao] = (uint8_t)(old | OCC_BIT);
        }
        __syncwarp();
        bool changed = false;
        if (KIND == SSD_ENV_CLEANUP) {
            if (cleanup_spawn_active(tb, hcount)) changed = cleanup_spawn<MW>(p, tb, lane, tile, false, scratch, g, t, hcount, pr, am, wm);
        } else {
            changed = harvest_spawn<MW>(p, lane, tile, false, scratch, g, t, pr, am);
        }
        if (changed) {                                // the masks (and #waste) go back only when the spawn changed them
#pragma unroll
            for (int q = 0; q < MW; q++)
                if (lane == q) {
                    hot[RO_AMASK / 4 + q] = am[q];
                    if (KIND == SSD_ENV_CLEANUP) hot[RO_WMASK / 4 + q] = wm[q];
                }
            if (KIND == SSD_ENV_CLEANUP && lane == 0) hot[RO_HCOUNT / 4] = (uint32_t)hcount;
        }
        if (KIND == SSD_ENV_HARVEST && act_lane)
            res_g[(size_t)env * SSD_MAXN + lane] |= (uint32_t)count_apples_r5(tile, ao, S) << RS_CLOSE_SHIFT;
        // ---- paint agents in agent order: the highest index wins a shared cell (map_env.py:257-261)
        const unsigned grp = __match_any_sync(FULL, act_lane ? (uint32_t)ao : (0x40000000u | (uint32_t)lane));
        __syncwarp();                                 // every lane's spawn / count reads of T are done
        if (act_lane && lane == 31 - __clz(grp)) tile[ao] = (uint8_t)PAINT_CODE(lane);
        __syncwarp();
        write_global_view<OUT>(p, lane, tile + SSD_VIEW * S + 8, S, inv_w, tb.pal, reinterpret_cast<T*>(out) + (size_t)env * env_elems);
        __syncwarp();                                 // the view's reads of T are done
        if (act_lane) tile[ao] = (uint8_t)old;
        __syncwarp();
    }
}

// RESET VIEW, behind grid_reset_kernel<KIND, 0> (no windows) on the same mask: the view of each reset env from its fresh
// record — the static map with the record's apples and (cleanup) waste, no agents (t == 0: MapEnv.reset does not paint them).  One
// warp per env; dynamic shared memory: one map (map_bytes, rows of Wp cells) per warp.  `width` is unused.
template <int KIND, int OUT>
__global__ void __launch_bounds__(GRID_THREADS) grid_reset_global_kernel(const GridParams p, const uint8_t* mask, void* out, int width)
{
    typedef typename GlobalElem<OUT>::T T;
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ uint32_t s_pal[16];
    if (threadIdx.x < 16) s_pal[threadIdx.x] = __ldg(p.pal + threadIdx.x);
    if constexpr (OUT != SSD_GLOBAL_U8) load_policy_palette<T>(p);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int env0 = blockIdx.x * GRID_WARPS + warp, estride = gridDim.x * GRID_WARPS;
    uint8_t* m = smem + warp * p.map_bytes;
    const float inv_w = __frcp_rn((float)p.W);
    const size_t env_elems = (size_t)3 * p.H * p.W;
    for (int i0 = 0; env0 + (long long)i0 * estride < p.E; i0 += 32) {
        const long long el = env0 + (long long)(i0 + lane) * estride;
        unsigned todo = __ballot_sync(FULL, el < p.E && (!mask || mask[el]));
        while (todo) {
            const int env = env0 + (i0 + __ffs(todo) - 1) * estride;
            todo &= todo - 1;
            const uint32_t hw = reinterpret_cast<const uint32_t*>(p.state + (size_t)env * p.rec_stride)[lane];
            for (int i = lane; i < (p.map_bytes >> 4); i += 32)
                reinterpret_cast<uint4*>(m)[i] = __ldg(reinterpret_cast<const uint4*>(p.base_map) + i);
            __syncwarp();
#pragma unroll
            for (int q = 0; q < MAX_POINT_ROUNDS; q++) {   // point 32 q + lane: the cell takes its code when its mask bit is set
                const uint32_t aq = __shfl_sync(FULL, hw, RO_AMASK / 4 + q);
                const uint32_t wq = KIND == SSD_ENV_CLEANUP ? __shfl_sync(FULL, hw, RO_WMASK / 4 + q) : 0u;
                const int j = 32 * q + lane;
                if (j < p.n_apple && ((aq >> lane) & 1u)) m[__ldg(p.apple_c + j)] = (uint8_t)C_APPLE;
                if (KIND == SSD_ENV_CLEANUP && j < p.n_waste && ((wq >> lane) & 1u)) m[__ldg(p.waste_c + j)] = (uint8_t)C_WASTE;
            }
            __syncwarp();
            write_global_view<OUT>(p, lane, m, p.Wp, inv_w, s_pal, reinterpret_cast<T*>(out) + (size_t)env * env_elems);
            __syncwarp();                                  // the view's reads of m are done
        }
    }
}
