// ssd_selfdrive.cuh — sm_100a kernels for SelfAcceleratingCarEnv (+ SelfdriveContractDistprop subgame wrapper).
//
// Reference behaviour restated here (paths relative to the reference root):
//   environments/self_driving_car_accelerate.py  reset :49-79, step :151-250, update_rel_rank :110-125,
//       update_infos :127-149, make_new_pos_consistent :92-108 (collision_on=False)
//   contract/contract_list.py :66-102 ; environments/two_stage_train.py :62-121, :159-187
//
// Mapping (round 2): EIGHT LANES PER ENV (lane = car), four envs per warp.  The kinematics are a handful of float64
// operations per car; the dominant cost is the 2n+5-double observation row per car (n (2n+5) 8 B per env), a pure function
// of the 2n positions / velocities.  Round 1 ran one thread per env and expanded the rows of a warp's 32 envs with lanes =
// row elements: 513 warp-instructions per env, most of them the flat-index bookkeeping of that expansion (0.155 ms per
// step at 131072 envs = 23 % of HBM).  Here every lane builds its own car's row in a warp-private staging area and the
// warp copies the four envs' rows out as one contiguous run of 16-byte stores; the cross-car parts of the step — crossing
// order, dist_to_front, make_new_pos_consistent, the contract's redistribution — happen on a few percent of the steps and
// run as plain scalar code on the octet's positions in shared memory.  State stays struct-of-arrays ([car][env]: a warp's
// loads touch whole 32-byte sectors).  CTAs are persistent and request a warp's next four envs' inputs before they process the
// current four (+4 %).  Everything is float64 and rounds like the reference (-fmad=false).
#pragma once
#include "ssd_common.cuh"

#ifndef CAR_WARPS
#define CAR_WARPS 8
#endif
#ifndef CAR_MIN_BLOCKS
#define CAR_MIN_BLOCKS 4
#endif
#define CAR_THREADS (CAR_WARPS * 32)
#define CAR_ENVS_PER_CTA (CAR_WARPS * 4)
#define CAR_OCT_DOUBLES 24              // per octet: old positions [8], new positions [8], velocities [8]

struct CarParams {
    int E, n, D, contract;
    int warp_doubles;       // shared memory per warp: 4 n D staged observation doubles (rounded up to even) + 4 octets' scratch
    double low_bound, high_bound, start_vel, start_vel_amb, theta_low, theta_high, null_prob;
    uint32_t seed, first_env_id;
    // state, struct of arrays
    double* pos;        // [n][E]
    double* vel;        // [n][E]
    double* theta;      // [E]
    double* m_transfers;// [E]
    double* dist_front; // [E]  dist_to_front['a{n-1}'] (:144)
    uint32_t* crossed;  // [E]  crossed_agents, 4 bits per entry
    uint32_t* meta;     // [E]  n_crossed | done mask << 8 | all_done << 16 | initialised << 31
    int32_t* t;         // [E]
    uint32_t* episode;  // [E]
    EpisodeLog elog;    // optional: ssd_set_episode_log ring buffer (appended to by the resets of car_kernel)
};

struct CarIO {
    const float* actions;   // [E][n]
    void* obs;              // double [E][n][D] (OBS_F64), or the policy's rows T [E n][W] (1 + SSD_POLICY_*: see car_kernel)
    double* rew; double* base_rew; double* transfers;   // [E][n]
    double* info;           // [E][n][4]: just_passed, active, ambulance_rank, ambulance_dist_to_front (row of the first acting agent)
    uint8_t* done;          // [E][n+1]
    int auto_reset;         // next-step auto-reset (see car_kernel)
    // compact result block of ssd_selfdrive_step_host_async (all null otherwise): int8 rewards, dones [E][n+1], and records
    // { int32 env; int32 0; double rew[n] } for the envs whose rewards are not all integers in [-127, 127]
    int8_t* c_rew8; uint8_t* c_done; uint32_t* c_count; uint8_t* c_rec;
};

__device__ __forceinline__ double py_min(double x, double y) { return y < x ? y : x; }   // Python min([x, y])
__device__ __forceinline__ double py_max(double x, double y) { return y > x ? y : x; }
__device__ __forceinline__ double car_u01(const CarParams& p, uint32_t env_id, uint32_t episode, uint32_t site, uint32_t idx)
{
    return __dmul_rn((double)draw_u32(p.seed, env_id, episode, 0u, site, 0u, idx), 1.0 / 4294967296.0);
}

#define CAR_FULL 0xffffffffu

// update_infos (:127-149) for the cars that crossed in this step, in index order: dist_to_front of the LAST of them stays
// in the env; the ambulance's own crossing also sets the infos of the step.  Scalar code, identical in the octet's lanes.
__device__ __noinline__ void car_update_infos(const CarParams& p, const double* o_new, uint32_t justm, uint32_t active_m,
                                              uint32_t crossed, int n_crossed, double& dist, double& info2, double& info3)
{
    const int n = p.n;
    for (int k = 0; k < n; k++) {
        if (!((justm >> k) & 1u)) continue;
        const double nk = o_new[k];
        double d = 0.0;
        for (int i = 0; i < n; i++) {
            if (i == k) continue;
            const bool act_i = (active_m >> i) & 1u;
            const double ni = o_new[i];
            if (!act_i) { if (__dsub_rn(p.high_bound, nk) > d) d = __dsub_rn(__dadd_rn(p.high_bound, 1.0), nk); }
            else if (ni > nk) { if (__dsub_rn(ni, nk) > d) d = __dsub_rn(ni, ni); }      // sic (:143)
        }
        dist = d;
        if (k == 0) {
            int c0 = 0;
            for (int i = 0; i < n_crossed; i++) if (((crossed >> (4 * i)) & 15u) == 0u) c0 = i;
            info2 = (double)(c0 + 1); info3 = d;
        }
    }
}

// make_new_pos_consistent (:92-108), run by ONE lane on the octet's effective positions (new for the acting cars, old for
// the others) when a crossed car stands behind the car that crossed after it: the later car is put 0.01 behind, cars
// pushed back below 0 leave the crossing order.  vmask: the pairs (i, i + 1) of the order that are inconsistent before any
// change — a pair needs a look only if it is one of them or its front car has just been moved.
__device__ __noinline__ void car_make_consistent(double* o_eff, uint32_t active_m, uint32_t vmask, uint32_t& crossed, int& n_crossed)
{
    uint32_t pre = 0u;
    int i = __ffs(vmask) - 1;
    while (i >= 0 && i + 1 < n_crossed) {
        const int f = (int)((crossed >> (4 * i)) & 15u), b = (int)((crossed >> (4 * i + 4)) & 15u);
        const double pf = o_eff[f], pb = o_eff[b];
        if (pf < pb && ((active_m >> f) & (active_m >> b) & 1u)) {
            const double nb = __dsub_rn(pf, 0.01);
            o_eff[b] = nb;
            if (nb < 0) pre |= 1u << b;
            i++;                                                           // its front car has moved: the next pair needs a look
        } else {
            vmask &= ~((2u << i) - 1u);                                    // on to the next pair that was inconsistent to begin with
            i = __ffs(vmask) - 1;
        }
    }
    if (pre) {
        uint32_t kept = 0u; int m = 0;
        for (int i = 0; i < n_crossed; i++) {
            const uint32_t a = (crossed >> (4 * i)) & 15u;
            if (!((pre >> a) & 1u)) { kept |= a << (4 * m); m++; }
        }
        crossed = kept; n_crossed = m;
    }
}

// SelfdriveContractDistprop (contract_list.py:66-102) + redistribution (two_stage_train.py:71-92) on the step the ambulance
// crosses: scalar code over the octet's final positions, every lane keeps its own car's reward / transfer.
__device__ __noinline__ void car_contract(const CarParams& p, const double* o_pos, uint32_t active_m, double theta, int k,
                                          double& rew, double& tr, double& total)
{
    const int n = p.n;
    const double x0 = o_pos[0];
    uint32_t behind = 0u;
    double sum = 0.0, rew0 = rew;                       // rew0: car 0's running reward (meaningful in lane 0)
    for (int i = 1; i < n; i++) {
        const double rel = __dsub_rn(o_pos[i], x0);
        if (rel < 0) { behind |= 1u << i; sum = __dadd_rn(sum, -rel); }
    }
    total = 0.0;
    if (behind) {
        const double v0 = __dmul_rn(theta, sum);
        if (k == 0) tr = v0;
        rew0 = __dsub_rn(rew0, v0); total = __dadd_rn(total, v0);
        if (k > 0 && k < n && ((behind >> k) & 1u) && ((active_m >> k) & 1u)) {
            const double dj = -__dsub_rn(o_pos[k], x0);
            rew = __dadd_rn(rew, __dmul_rn(v0, __ddiv_rn(dj, sum)));
        }
    }
    for (int i = 1; i < n; i++) {
        if (!((active_m >> i) & 1u) || ((behind >> i) & 1u)) continue;
        const double vi = __dmul_rn(theta, __dsub_rn(o_pos[i], x0));
        if (i == k) { tr = vi; rew = __dsub_rn(rew, vi); }
        total = __dadd_rn(total, vi);
        rew0 = __dadd_rn(rew0, vi);
    }
    if (k == 0) rew = rew0;
}

// Episode log of the resets of one car_kernel round (all 32 lanes; `mine`: this octet resets an initialised env): one atomic
// for the warp's up to four records, then the octet writes its env's record — metrics [transfers, 0, ...] —, lane k the
// vectors k, k + 8, ...  Reads the env's state before the reset rewrites it.  Out of line, off the step's hot path.
__device__ __noinline__ void car_log_episode(EpisodeLog log, const double* theta, const double* m_transfers, const int32_t* t,
                                             const uint32_t* episode, int env, uint32_t env_id, bool mine, bool ended, int lane)
{
    const int k = lane & 7, obase = lane & 24;
    const uint32_t lm = __ballot_sync(CAR_FULL, mine && k == 0);
    if (!lm) return;
    const int leader = __ffs(lm) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(log.count, (unsigned long long)__popc(lm));
    base = __shfl_sync(CAR_FULL, base, leader);
    if (!mine) return;
    const unsigned long long slot = (base + (unsigned long long)__popc(lm & ((1u << obase) - 1u))) % log.capacity;
    uint4* rec = log.records + slot * EPREC_VECS;
#pragma unroll 1
    for (int v = k; v < EPREC_VECS; v += 8) {
        uint4 w;
        if (v == 0) w = eprec_head(env_id, episode[env], t[env], ended);
        else if (v == 1) w = eprec_pair(theta[env], 0.0);
        else w = eprec_pair(v == 2 ? m_transfers[env] : 0.0, 0.0);
        rec[v] = w;
    }
}

// An env's staged rows, L bytes, to global memory in the widest units that divide L: the staged run and its destination
// start at multiples of L from 16-byte aligned bases, so both are aligned to the unit (16 bytes for n = 8 in every form).
__device__ __forceinline__ void car_copy_run(uint8_t* dst, const uint8_t* src, int L, int lane)
{
    if ((L & 15) == 0) for (int f = lane; 16 * f < L; f += 32) reinterpret_cast<uint4*>(dst)[f] = reinterpret_cast<const uint4*>(src)[f];
    else if ((L & 7) == 0) for (int f = lane; 8 * f < L; f += 32) reinterpret_cast<uint2*>(dst)[f] = reinterpret_cast<const uint2*>(src)[f];
    else if ((L & 3) == 0) for (int f = lane; 4 * f < L; f += 32) reinterpret_cast<uint32_t*>(dst)[f] = reinterpret_cast<const uint32_t*>(src)[f];
    else for (int f = lane; 2 * f < L; f += 32) reinterpret_cast<uint16_t*>(dst)[f] = reinterpret_cast<const uint16_t*>(src)[f];
}

// One launch = one step (or, RESET_ONLY, one masked reset) of every env.
// Next-step auto-reset (ssd_selfdrive_io.auto_reset): an env whose episode ended in the previous step starts its next
// episode in this one — reset observation, zero rewards, dones cleared, the actions of this step ignored.
// FORM: OBS_F64 (float64 rows [E][n][D]) or 1 + SSD_POLICY_*: the policy's rows T [E n][W], each car's D values ++ [theta, 0]
// with a contract (W = D + 2), else the D values alone (W = D), each T(float32(x)).  Either form is built in the staging
// area exactly as it goes out (an env's n rows contiguous, the warp's four envs one after the other) and copied out by
// car_copy_run.
template <bool RESET_ONLY, int FORM>
__global__ void __launch_bounds__(CAR_THREADS, CAR_MIN_BLOCKS) car_kernel(const CarParams p, const CarIO io, const uint8_t* __restrict__ mask)
{
    extern __shared__ __align__(16) double csm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, k = lane & 7, oct = lane >> 3, obase = lane & 24;
    const int n = p.n, D = p.D, nD = n * D;
    double* w_stage = csm + (size_t)warp * p.warp_doubles;
    double* o_pos = w_stage + (p.warp_doubles - 4 * CAR_OCT_DOUBLES) + oct * CAR_OCT_DOUBLES;
    double* o_new = o_pos + 8;
    double* o_vel = o_pos + 16;
    const bool kv = k < n;
    // Persistent CTAs; the inputs of a warp's NEXT four envs are requested before the current four are processed, so the
    // one round of global loads a step needs (its only long-latency wait) overlaps a whole round of work.
    struct In { uint32_t meta, crossed; double theta, pos, vel, dist; float act; int t; int env; bool live; };
    auto fetch = [&](int g) {
        In in = { 0u, 0u, 0.0, 0.0, 0.0, -1.0, 0.0f, 0, p.E - 1, false };
        const int e_raw = (g * CAR_WARPS + warp) * 4 + oct;
        in.live = e_raw < p.E;
        in.env = in.live ? e_raw : p.E - 1;
        if (RESET_ONLY && mask) in.live = in.live && mask[in.env] != 0;
        if (in.live) {
            in.meta = p.meta[in.env];
            if (!RESET_ONLY) {
                in.crossed = p.crossed[in.env]; in.theta = p.theta[in.env];
                if (kv) {
                    const size_t so_ = (size_t)k * p.E + in.env;
                    in.pos = p.pos[so_]; in.vel = p.vel[so_]; in.act = io.actions[(size_t)in.env * n + k];
                }
                if (k == 0) in.t = p.t[in.env];
                if (n == 1) in.dist = p.dist_front[in.env];
            }
        }
        return in;
    };
    const int ngroups = (p.E + CAR_ENVS_PER_CTA - 1) / CAR_ENVS_PER_CTA;
    In cur = fetch(blockIdx.x < ngroups ? (int)blockIdx.x : 0);
#pragma unroll 1
    for (int grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
    const int grp_next = grp + (int)gridDim.x;
    const In nxt = fetch(grp_next < ngroups ? grp_next : grp);
    const bool live = cur.live;
    const int env = cur.env;
    const size_t so = (size_t)k * p.E + env;
    const uint32_t meta0 = cur.meta;
    const uint32_t crossed_in = cur.crossed; const double theta_in = cur.theta, pos_in = cur.pos, vel_in = cur.vel, dist_in = cur.dist;
    const float act_in = cur.act; const int t_in = cur.t;
    if (!RESET_ONLY || __any_sync(CAR_FULL, live)) {
    const bool doreset = RESET_ONLY ? live : (live && io.auto_reset && ((meta0 >> 16) & 1u));
    const bool stepping = !RESET_ONLY && live && !doreset;
    double x = 0.0, v = 0.0;                            // this car's position / velocity after the step (or the reset)
    double row_theta = theta_in;                        // the policy form's theta column (after a reset: lane 0's new theta)

    if (p.elog.records && __any_sync(CAR_FULL, doreset))     // hand the finished episodes over before the reset rewrites them
        car_log_episode(p.elog, p.theta, p.m_transfers, p.t, p.episode, env, p.first_env_id + (uint32_t)env,
                        doreset && (meta0 & 0x80000000u), (meta0 >> 16) & 1u, lane);
    if (doreset) {
        // self_driving_car_accelerate.py:49-79 + two_stage_train.py:159-187
        const uint32_t episode = (meta0 & 0x80000000u) ? p.episode[env] + 1u : 0u;
        const uint32_t env_id = p.first_env_id + (uint32_t)env;
        if (kv) {
            const double u = car_u01(p, env_id, episode, SITE_SELFDRIVE_RESET, (uint32_t)k);
            if (k == 0) {        // random.random() * low / 2 + low / 2  (:53)
                x = __dadd_rn(__ddiv_rn(__dmul_rn(u, p.low_bound), 2.0), __ddiv_rn(p.low_bound, 2.0));
                v = p.start_vel_amb;
            } else {             // random.random() * low / 16 + low * 3 / 16  (:57)
                x = __dadd_rn(__ddiv_rn(__dmul_rn(u, p.low_bound), 16.0), __ddiv_rn(__dmul_rn(p.low_bound, 3.0), 16.0));
                v = p.start_vel;
            }
            p.pos[so] = x; p.vel[so] = v;
        }
        if (k == 0) {
            double theta = 0.0;
            if (p.contract != SSD_CONTRACT_NONE) {       // two_stage_train.py:163-166
                const double u0 = car_u01(p, env_id, episode, SITE_CONTRACT, 0u), u1 = car_u01(p, env_id, episode, SITE_CONTRACT, 1u);
                theta = (u0 > p.null_prob) ? __dadd_rn(p.theta_low, __dmul_rn(__dsub_rn(p.theta_high, p.theta_low), u1)) : p.theta_low;
            }
            p.theta[env] = theta; p.m_transfers[env] = 0.0; p.dist_front[env] = -1.0;
            row_theta = theta;
            p.crossed[env] = 0u; p.meta[env] = 0x80000000u; p.t[env] = 0; p.episode[env] = episode;
        }
    }

    if (!RESET_ONLY) {
        int n_crossed = (int)(meta0 & 0xFFu);
        uint32_t done_mask = (meta0 >> 8) & 0xFFu;
        bool all_done = (meta0 >> 16) & 1u;
        uint32_t crossed = stepping ? crossed_in : 0u;
        const double theta = theta_in;
        const double pos0 = stepping ? pos_in : 0.0, vel0 = stepping ? vel_in : 0.0;
        const uint32_t active_m = (!stepping || all_done) ? 0u : (~done_mask & ((1u << n) - 1u));   // done agents stop acting (RLlib)
        const bool on = active_m != 0u, act = (active_m >> k) & 1u;
        const int first = active_m ? __ffs(active_m) - 1 : -1;
        double rew = 0.0, tr = 0.0, info2 = 0.0, info3 = 0.0;
        double newx = pos0;
        if (stepping) { x = pos0; v = vel0; }
        if (act) {
            const double a = (double)act_in;
            v = py_max(py_min(__dadd_rn(py_max(py_min(a, 0.1), -0.1), vel0), k == 0 ? 1.0 : 0.25), 0.0);      // :172-174
            newx = __dadd_rn(v, pos0);                                                                         // :180
        }
        const bool just = act && pos0 < 0.0 && newx > 0.0;
        const uint32_t justm = (__ballot_sync(CAR_FULL, just) >> obase) & 0xFFu;
        if (on) {
            if (k == 0) p.t[env] = t_in + 1;
            // infos defaults (:183-189)
            int ci = -1;                                                  // the ambulance's place in the crossing order
            {   // lowest zero nibble of the order (a car appears once; the lowest flag of the zero-in-word test is exact)
                const uint32_t z = (crossed - 0x11111111u) & ~crossed & 0x88888888u;
                const int i0 = z ? (__ffs(z) - 1) >> 2 : 8;
                if (i0 < n_crossed) ci = i0;
            }
            info2 = ci >= 0 ? (double)(ci + 1) : (double)n;
            { const double d0 = dist_in; info3 = d0 > -1.0 ? d0 : __dsub_rn(p.high_bound, p.low_bound); }
            // update_rel_rank (:110-125): crossers appended in index order
            for (uint32_t jm = justm; jm; jm &= jm - 1) { crossed |= (uint32_t)(__ffs(jm) - 1) << (4 * n_crossed); n_crossed++; }
        }
        o_new[k] = newx;
        __syncwarp();
        if (__any_sync(CAR_FULL, justm != 0u)) {                           // a few percent of the steps
            if (justm) {
                double dist = 0.0;
                car_update_infos(p, o_new, justm, active_m, crossed, n_crossed, dist, info2, info3);
                if (k == 0) p.dist_front[env] = dist;
            }
        }
        {   // make_new_pos_consistent changes something only if a crossed car stands behind its successor in the order
            bool viol = false;                                             // (o_new: new positions of the acting cars, old ones of the others)
            if (on && k + 1 < n_crossed) {
                const int f = (int)((crossed >> (4 * k)) & 15u), b = (int)((crossed >> (4 * k + 4)) & 15u);
                viol = ((active_m >> f) & (active_m >> b) & 1u) && o_new[f] < o_new[b];
            }
            const uint32_t vm = __ballot_sync(CAR_FULL, viol);
            if (vm) {
                const uint32_t vo = (vm >> obase) & 0xFFu;
                if (vo && k == 0) car_make_consistent(o_new, active_m, vo, crossed, n_crossed);
                __syncwarp();
                crossed = __shfl_sync(CAR_FULL, crossed, 0, 8);
                n_crossed = __shfl_sync(CAR_FULL, n_crossed, 0, 8);
                newx = o_new[k];
            }
        }
        if (on) {
            // new positions, rewards, dones (:216-238)
            x = act ? newx : pos0;
            if (act) rew = k == 0 ? __dsub_rn(-1.0, 99.0) : -1.0;
        }
        const bool over = on && kv && x > p.high_bound;
        if (over) x = __dadd_rn(p.high_bound, 1.0);
        done_mask |= (__ballot_sync(CAR_FULL, over) >> obase) & 0xFFu;
        if (on) {
            all_done = (active_m & ~done_mask) == 0u;
            if (kv) { p.pos[so] = x; p.vel[so] = v; }
        }
        const double base_rew = rew;
        __syncwarp();
        o_pos[k] = x;                                                      // final positions (contract, observation rows)
        __syncwarp();
        const bool deal = stepping && p.contract == SSD_CONTRACT_SELFDRIVE_DISTPROP && (active_m & 1u) && (justm & 1u);
        if (__any_sync(CAR_FULL, deal)) {
            if (deal) {
                double total = 0.0;
                car_contract(p, o_pos, active_m, theta, k, rew, tr, total);
                if (k == 0) p.m_transfers[env] = __dadd_rn(p.m_transfers[env], total);
            }
        }
        if (stepping && k == 0) {
            p.crossed[env] = crossed;
            p.meta[env] = 0x80000000u | (uint32_t)n_crossed | (done_mask << 8) | ((all_done ? 1u : 0u) << 16);
        }
        if (live && kv) {                                                  // (a restarting env: zeros)
            const size_t o = (size_t)env * n + k;
            if (io.rew) io.rew[o] = rew;
            if (io.base_rew) io.base_rew[o] = base_rew;
            if (io.transfers) io.transfers[o] = tr;
            if (io.info)
                reinterpret_cast<double4*>(io.info)[o] = stepping ? make_double4(just ? 1.0 : 0.0, act ? 1.0 : 0.0, k == first ? info2 : 0.0, k == first ? info3 : 0.0)
                                                                  : make_double4(0.0, 0.0, 0.0, 0.0);
            if (io.done) io.done[(size_t)env * (n + 1) + k] = stepping ? (uint8_t)((done_mask >> k) & 1u) : (uint8_t)0;
        }
        if (live && k == 0 && io.done) io.done[(size_t)env * (n + 1) + n] = (stepping && all_done) ? 1 : 0;
        if (io.c_rew8) {                                                   // the pipelined host path's lossless result block
            int vi = 0;
            const bool mine = live && kv, fits = reward_fits_i8(rew, vi);
            if (mine) {
                io.c_rew8[(size_t)env * n + k] = fits ? (int8_t)vi : (int8_t)0;
                io.c_done[(size_t)env * (n + 1) + k] = stepping ? (uint8_t)((done_mask >> k) & 1u) : (uint8_t)0;
            }
            if (live && k == 0) io.c_done[(size_t)env * (n + 1) + n] = (stepping && all_done) ? 1 : 0;
            const uint32_t badm = __ballot_sync(CAR_FULL, mine && !fits);
            if (badm) {                                                    // one record per env with such a reward, one atomic per warp
                const bool need = ((badm >> obase) & 0xFFu) != 0u;
                const uint32_t needm = __ballot_sync(CAR_FULL, need && k == 0);
                const int leader = __ffs(needm) - 1;
                uint32_t base = 0u;
                if (lane == leader) base = atomicAdd(io.c_count, (uint32_t)__popc(needm));
                base = __shfl_sync(CAR_FULL, base, leader);
                if (need) {
                    uint8_t* rec = io.c_rec + (size_t)(base + (uint32_t)__popc(needm & ((1u << obase) - 1u))) * (size_t)(8 + 8 * n);
                    if (k == 0) { reinterpret_cast<int32_t*>(rec)[0] = env; reinterpret_cast<int32_t*>(rec)[1] = 0; }
                    if (kv) reinterpret_cast<double*>(rec + 8)[k] = rew;
                }
            }
        }
    } else {
        o_pos[k] = x;
    }
    o_vel[k] = v;
    __syncwarp();

    // ---- observation rows (:244-249): [pos, vel, pos_q - pos (q < n), vel_q (q < n), pos_0 > 0, pos > 0, 0], built by the
    // car's lane in the staging area, then copied out as one contiguous run per env
    if (io.obs) {
        if constexpr (FORM == OBS_F64) {
            if (kv) {
                double* row = w_stage + (size_t)(oct * n + k) * D;
                row[0] = x; row[1] = v;
                for (int q = 0; q < n; q++) { row[2 + q] = __dsub_rn(o_pos[q], x); row[2 + n + q] = o_vel[q]; }
                row[2 + 2 * n] = o_pos[0] > 0 ? 1.0 : 0.0;
                row[3 + 2 * n] = x > 0 ? 1.0 : 0.0;
                row[4 + 2 * n] = 0.0;
            }
            __syncwarp();
            const uint32_t lv = __ballot_sync(CAR_FULL, live);
            for (int q = 0; q < 4; q++) {
                if (!((lv >> (8 * q)) & 1u)) continue;                    // (uniform)
                const int e = (grp * CAR_WARPS + warp) * 4 + q;
                double* dst = static_cast<double*>(io.obs) + (size_t)e * nD;
                const double* src = w_stage + (size_t)q * nD;
                if ((nD & 1) == 0) {                                       // 16-byte aligned runs
                    for (int f = lane; 2 * f < nD; f += 32) reinterpret_cast<double2*>(dst)[f] = reinterpret_cast<const double2*>(src)[f];
                } else {
                    for (int f = lane; f < nD; f += 32) dst[f] = src[f];
                }
            }
        } else {
            // the same values as T, and theta (lane 0's of the octet: after a reset the new one) and 0 after them
            typedef typename PolicyElem<FORM>::T T;
            const bool con = p.contract != SSD_CONTRACT_NONE;
            const int W = D + (con ? 2 : 0), L = n * W * (int)sizeof(T);
            const double th = __shfl_sync(CAR_FULL, row_theta, obase);
            if (kv) {
                T* row = reinterpret_cast<T*>(w_stage) + (size_t)(oct * n + k) * W;
                auto put = [&](int i, double val) { row[i] = policy_cast<T>(__double2float_rn(val)); };
                put(0, x); put(1, v);
                for (int q = 0; q < n; q++) { put(2 + q, __dsub_rn(o_pos[q], x)); put(2 + n + q, o_vel[q]); }
                put(2 + 2 * n, o_pos[0] > 0 ? 1.0 : 0.0);
                put(3 + 2 * n, x > 0 ? 1.0 : 0.0);
                put(4 + 2 * n, 0.0);
                if (con) { put(D, th); put(D + 1, 0.0); }
            }
            __syncwarp();
            const uint32_t lv = __ballot_sync(CAR_FULL, live);
            for (int q = 0; q < 4; q++) {
                if (!((lv >> (8 * q)) & 1u)) continue;                    // (uniform)
                const int e = (grp * CAR_WARPS + warp) * 4 + q;
                car_copy_run(static_cast<uint8_t*>(io.obs) + (size_t)e * L, reinterpret_cast<const uint8_t*>(w_stage) + (size_t)q * L, L, lane);
            }
        }
    }
    }
    cur = nxt;
    __syncwarp();                                       // the warp's staging area is rewritten by the next round
    }
}

__global__ void car_random_actions_kernel(const CarParams p, uint32_t step_index, uint32_t* counter, float lo, float hi,
                                          float* actions)
{
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (counter) step_index = *reinterpret_cast<volatile uint32_t*>(counter);
    if (env < p.E) {
        const uint32_t env_id = p.first_env_id + (uint32_t)env;
        for (int b = 0; b * 4 < p.n; b++) {
            Philox4 q = philox4x32_10((uint32_t)b, SITE_ACTIONS, step_index, 0u, p.seed, env_id);
            uint32_t w[4] = { q.x, q.y, q.z, q.w };
            for (int j = 0; j < 4 && b * 4 + j < p.n; j++)
                actions[(size_t)env * p.n + b * 4 + j] = lo + (hi - lo) * ((float)(w[j] >> 8) * (1.0f / 16777216.0f));
        }
    }
    if (counter) counter_finish(counter, step_index);
}

__global__ void car_get_state_kernel(const CarParams p, double* pos, double* vel, double* theta, double* m_transfers, int32_t* t)
{
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.E) return;
    for (int k = 0; k < p.n; k++) {
        if (pos) pos[(size_t)env * p.n + k] = p.pos[(size_t)k * p.E + env];
        if (vel) vel[(size_t)env * p.n + k] = p.vel[(size_t)k * p.E + env];
    }
    if (theta) theta[env] = p.theta[env];
    if (m_transfers) m_transfers[env] = p.m_transfers[env];
    if (t) t[env] = p.t[env];
}
