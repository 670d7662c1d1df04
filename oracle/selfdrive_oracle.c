/*
 * selfdrive_oracle.c — CPU restatement of SelfAcceleratingCarEnv + SelfdriveContractDistprop + the contract
 * wrapper's redistribution, for E independent envs.
 *
 * TEST INFRASTRUCTURE (oracle/): used by tests/, bench.py's cpu_baseline / `--impl reference` leg and
 * __graft_entry__.smoke() only — never by the product path.  Pinned against the unmodified reference by
 * tests/golden/selfdrive_*.npz (oracle/make_golden.py runs the reference under RNG injection).
 *
 * Reference (paths relative to the reference root):
 *   environments/self_driving_car_accelerate.py  reset :49-79, step :151-250, update_rel_rank :110-125,
 *       update_infos :127-149, make_new_pos_consistent :92-108 (collision_on=False, the default)
 *   contract/contract_list.py SelfdriveContractDistprop.compute_transfer :66-102
 *   environments/two_stage_train.py SeparateContractEnv.step :62-121, SeparateContractSubgameStage.reset :159-187
 *
 * Acting set: RLlib stops querying an agent once its done flag has been returned, so the agents acting at a
 * step are those not done at its start ("active").  Everything is float64 like the reference's Python floats
 * (actions are float32 values widened exactly).  Draws: Philox site 9 (selfdrive reset), index = agent;
 * site 7 (contract sample) as for the gridworlds.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define MAXN 8
#define SITE_CONTRACT 7
#define SITE_SELFDRIVE_RESET 9

#define ACCEL_LOW (-0.1)
#define ACCEL_HIGH 0.1
#define VEL_LOW 0.0
#define VEL_HIGH 0.25
#define VEL_HIGH_AMB 1.0

typedef struct {
    int n, contract;
    double low_bound, high_bound, start_vel, start_vel_amb, theta_low, theta_high, null_prob;
    uint32_t seed, env_id, episode;
    double pos[MAXN], vel[MAXN];
    int done[MAXN], all_done;
    int crossed[2 * MAXN], n_crossed;      /* crossed_agents, in order */
    double dist_to_front_last;             /* dist_to_front['a{n-1}'] (the only key ever written, :144) */
    double theta, m_transfers;
    int t;
} car_env;

typedef struct { int E, n; car_env* envs; } car_batch;

static void philox(const uint32_t c_in[4], const uint32_t k_in[2], uint32_t out[4])
{
    uint32_t c0 = c_in[0], c1 = c_in[1], c2 = c_in[2], c3 = c_in[3], k0 = k_in[0], k1 = k_in[1];
    for (int i = 0; i < 10; i++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1; c3 = (uint32_t)p0; c0 = n0; c2 = n2;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
static double draw_f64(const car_env* e, uint32_t t, int site, uint32_t call, uint32_t idx)
{
    uint32_t ctr[4] = { idx >> 2, (uint32_t)site | (call << 8), t, e->episode };
    uint32_t key[2] = { e->seed, e->env_id }, out[4];
    philox(ctr, key, out);
    return (double)out[idx & 3] * (1.0 / 4294967296.0);
}

/* Python's min([x, y]) / max([x, y]): the first extremal element wins ties */
static double py_min(double x, double y) { return y < x ? y : x; }
static double py_max(double x, double y) { return y > x ? y : x; }

static int obs_dim(int n) { return 2 * (n + 1) + 3; }

/* observation row of agent k (:75-79, :244-249); crashed flag is always 0.0 with collision_on=False */
static void write_obs(const car_env* e, int k, double* o)
{
    int n = e->n;
    o[0] = e->pos[k]; o[1] = e->vel[k];
    for (int i = 0; i < n; i++) { o[2 + i] = e->pos[i] - e->pos[k]; o[2 + n + i] = e->vel[i]; }
    o[2 + 2 * n] = e->pos[0] > 0 ? 1.0 : 0.0;
    o[3 + 2 * n] = e->pos[k] > 0 ? 1.0 : 0.0;
    o[4 + 2 * n] = 0.0;
}

static void env_reset(car_env* e, uint32_t episode)
{
    e->episode = episode;
    for (int k = 0; k < e->n; k++) {
        double u = draw_f64(e, 0, SITE_SELFDRIVE_RESET, 0, (uint32_t)k);
        if (k == 0) { e->pos[k] = u * e->low_bound / 2 + e->low_bound / 2; e->vel[k] = e->start_vel_amb; }   /* :53-54 */
        else { e->pos[k] = u * e->low_bound / 16 + e->low_bound * 3 / 16; e->vel[k] = e->start_vel; }       /* :57-58 */
        e->done[k] = 0;
    }
    e->all_done = 0; e->n_crossed = 0; e->dist_to_front_last = -1; e->m_transfers = 0; e->t = 0;
    e->theta = 0;
    if (e->contract) {                     /* two_stage_train.py:163-166 */
        double u0 = draw_f64(e, 0, SITE_CONTRACT, 0, 0);
        if (u0 > e->null_prob) { double u1 = draw_f64(e, 0, SITE_CONTRACT, 0, 1); e->theta = e->theta_low + (e->theta_high - e->theta_low) * u1; }
        else e->theta = e->theta_low;
    }
}

static int crossed_index(const car_env* e, int a)
{
    for (int i = 0; i < e->n_crossed; i++) if (e->crossed[i] == a) return i;
    return -1;
}

/* info: [n][4] doubles = just_passed, active (acted this step), ambulance_rank, ambulance_dist_to_front
 * (the last two only meaningful in the row of the first acting agent, like the reference's infos[key_lst[0]]) */
static void env_step(car_env* e, const float* acts, double* obs, double* rew, double* base_rew, double* transfers,
                     double* info, uint8_t* done)
{
    const int n = e->n, D = obs_dim(n);
    int active[MAXN], first = -1;
    double newpos[MAXN];
    for (int k = 0; k < n; k++) { active[k] = !e->done[k] && !e->all_done; if (active[k] && first < 0) first = k; }
    for (int k = 0; k < n; k++) { rew[k] = 0; base_rew[k] = 0; transfers[k] = 0; for (int j = 0; j < 4; j++) info[k * 4 + j] = 0; }
    if (first < 0) {                        /* episode over: frozen until reset (the reference would raise, :160) */
        for (int k = 0; k < n; k++) { write_obs(e, k, obs + k * D); done[k] = (uint8_t)e->done[k]; }
        done[n] = 1;
        return;
    }
    e->t++;
    for (int k = 0; k < n; k++) {
        newpos[k] = e->pos[k];
        if (!active[k]) continue;
        double a = (double)acts[k];
        double v = py_max(py_min(py_max(py_min(a, ACCEL_HIGH), ACCEL_LOW) + e->vel[k], k == 0 ? VEL_HIGH_AMB : VEL_HIGH), VEL_LOW);   /* :172-174 */
        e->vel[k] = v;
        newpos[k] = e->vel[k] + e->pos[k];                                                                                          /* :180 */
    }
    /* infos defaults (:183-189) */
    { int ci = crossed_index(e, 0);
      info[first * 4 + 2] = ci >= 0 ? ci + 1 : n;
      double d0 = n == 1 ? e->dist_to_front_last : -1;        /* dist_to_front['a0'] is only ever written when n == 1 */
      info[first * 4 + 3] = d0 > -1 ? d0 : e->high_bound - e->low_bound; }
    /* update_rel_rank (:110-125): crossers are appended sorted by the digit of their name = index order */
    int just[MAXN];
    for (int k = 0; k < n; k++) {
        just[k] = active[k] && e->pos[k] < 0.0 && newpos[k] > 0.0;
        if (just[k]) e->crossed[e->n_crossed++] = k;
    }
    /* update_infos (:127-149) */
    for (int k = 0; k < n; k++) {
        if (!just[k]) continue;
        info[k * 4 + 0] = 1;
        double d = 0.0;
        for (int i = 0; i < n; i++) {
            if (i == k) continue;
            if (!active[i] || newpos[i] > newpos[k]) {
                if (!active[i]) { if (e->high_bound - newpos[k] > d) d = e->high_bound + 1 - newpos[k]; }
                else { if (newpos[i] - newpos[k] > d) d = newpos[i] - newpos[i]; }      /* sic (:143): always 0.0 */
            }
        }
        e->dist_to_front_last = d;
        if (k == 0) { info[first * 4 + 2] = crossed_index(e, 0) + 1; info[first * 4 + 3] = d; }
    }
    /* make_new_pos_consistent (:92-108) */
    { int pre[2 * MAXN], npre = 0;
      for (int i = 0; i + 1 < e->n_crossed; i++) {
          int f = e->crossed[i], b = e->crossed[i + 1];
          double pf = active[f] ? newpos[f] : e->pos[f], pb = active[b] ? newpos[b] : e->pos[b];
          if (pf < pb && active[f] && active[b]) {
              newpos[b] = pf - 0.01;
              if (newpos[b] < 0) pre[npre++] = b;
          }
      }
      if (npre) {
          int m = 0;
          for (int i = 0; i < e->n_crossed; i++) {
              int keep = 1;
              for (int j = 0; j < npre; j++) if (pre[j] == e->crossed[i]) keep = 0;
              if (keep) e->crossed[m++] = e->crossed[i];
          }
          e->n_crossed = m;
      } }
    for (int k = 0; k < n; k++) if (active[k]) e->pos[k] = newpos[k];
    for (int k = 0; k < n; k++) if (active[k]) { double r = -1.0; if (k == 0) r -= 99.0; rew[k] = r; base_rew[k] = r; info[k * 4 + 1] = 1; }
    for (int i = 0; i < n; i++) if (e->pos[i] > e->high_bound) { e->pos[i] = e->high_bound + 1; e->done[i] = 1; }   /* :228-231 */
    { int all = 1; for (int k = 0; k < n; k++) if (active[k] && !e->done[k]) all = 0; e->all_done = all; }
    for (int k = 0; k < n; k++) write_obs(e, k, obs + k * D);

    /* SelfdriveContractDistprop (contract_list.py:66-102) + redistribution (two_stage_train.py:71-92) */
    if (e->contract && active[0] && just[0]) {
        const double* o0 = obs;                  /* obs['a0'] */
        int behind[MAXN], any = 0;
        double dist[MAXN], sum = 0;
        for (int i = 1; i < n; i++) { behind[i] = o0[2 + i] < 0; if (behind[i]) { any = 1; dist[i] = -o0[2 + i]; sum += dist[i]; } }
        double total = 0;
        /* i = 0 */
        if (any) {
            double v0 = e->theta * sum;
            transfers[0] = v0;
            rew[0] -= v0; total += v0;
            for (int j = 1; j < n; j++) if (behind[j] && active[j]) rew[j] += v0 * (dist[j] / sum);
        }
        for (int i = 1; i < n; i++) {
            if (!active[i] || behind[i]) continue;
            double vi = e->theta * o0[2 + i];
            transfers[i] = vi;
            rew[i] -= vi; total += vi;
            rew[0] += vi * 1;
        }
        e->m_transfers += total;
    }
    for (int k = 0; k < n; k++) done[k] = (uint8_t)e->done[k];
    done[n] = (uint8_t)e->all_done;
}

/* ------------------------------------------------------------------ C API (ctypes: oracle/oracle.py) */
void* car_oracle_create(int E, int n, int contract, double low_bound, double high_bound, double start_vel,
                        double start_vel_amb, double theta_low, double theta_high, double null_prob, uint32_t seed,
                        uint32_t first_env_id)
{
    if (n < 1 || n > MAXN || E < 1) return NULL;
    car_batch* b = (car_batch*)calloc(1, sizeof(car_batch));
    b->E = E; b->n = n;
    b->envs = (car_env*)calloc((size_t)E, sizeof(car_env));
    for (int i = 0; i < E; i++) {
        car_env* e = &b->envs[i];
        e->n = n; e->contract = contract; e->low_bound = low_bound; e->high_bound = high_bound; e->start_vel = start_vel;
        e->start_vel_amb = start_vel_amb; e->theta_low = theta_low; e->theta_high = theta_high; e->null_prob = null_prob;
        e->seed = seed; e->env_id = first_env_id + (uint32_t)i;
        for (int k = 0; k < n; k++) { e->pos[k] = low_bound; e->vel[k] = start_vel; }
        e->dist_to_front_last = -1;
    }
    return b;
}
void car_oracle_destroy(void* h) { car_batch* b = (car_batch*)h; if (b) { free(b->envs); free(b); } }
int car_oracle_obs_dim(void* h) { return obs_dim(((car_batch*)h)->n); }

void car_oracle_reset(void* h, const uint8_t* mask, const uint32_t* episode, double* obs)
{
    car_batch* b = (car_batch*)h;
    int D = obs_dim(b->n);
    for (int i = 0; i < b->E; i++) {
        if (mask && !mask[i]) continue;
        env_reset(&b->envs[i], episode[i]);
        if (obs) for (int k = 0; k < b->n; k++) write_obs(&b->envs[i], k, obs + ((size_t)i * b->n + k) * D);
    }
}
/* acts float32 [E][n]; obs [E][n][D]; rew/base_rew/transfers [E][n]; info [E][n][4]; done u8 [E][n+1] */
void car_oracle_step(void* h, const float* acts, double* obs, double* rew, double* base_rew, double* transfers,
                     double* info, uint8_t* done)
{
    car_batch* b = (car_batch*)h;
    int n = b->n, D = obs_dim(n);
#pragma omp parallel for schedule(static) if (b->E > 1)   /* a one-env batch (the live differential tests) stays on the calling thread */
    for (int i = 0; i < b->E; i++)
        env_step(&b->envs[i], acts + (size_t)i * n, obs + (size_t)i * n * D, rew + (size_t)i * n, base_rew + (size_t)i * n,
                 transfers + (size_t)i * n, info + (size_t)i * n * 4, done + (size_t)i * (n + 1));
}
/* car_oracle_step with a per-env skip byte: an env with skip[i] != 0 is not stepped and its output rows are left as the
   caller passed them (a batch's next-step auto-reset: reset the done envs with a mask, then step the others). */
void car_oracle_step_skip(void* h, const float* acts, double* obs, double* rew, double* base_rew, double* transfers,
                          double* info, uint8_t* done, const uint8_t* skip)
{
    car_batch* b = (car_batch*)h;
    int n = b->n, D = obs_dim(n);
#pragma omp parallel for schedule(static) if (b->E > 1)
    for (int i = 0; i < b->E; i++) {
        if (skip && skip[i]) continue;
        env_step(&b->envs[i], acts + (size_t)i * n, obs + (size_t)i * n * D, rew + (size_t)i * n, base_rew + (size_t)i * n,
                 transfers + (size_t)i * n, info + (size_t)i * n * 4, done + (size_t)i * (n + 1));
    }
}
/* state: pos [E][n], vel [E][n], theta [E], transfers metric [E], t [E] */
void car_oracle_get_state(void* h, double* pos, double* vel, double* theta, double* m_transfers, int32_t* t)
{
    car_batch* b = (car_batch*)h;
    for (int i = 0; i < b->E; i++) {
        car_env* e = &b->envs[i];
        for (int k = 0; k < b->n; k++) { pos[(size_t)i * b->n + k] = e->pos[k]; vel[(size_t)i * b->n + k] = e->vel[k]; }
        theta[i] = e->theta; m_transfers[i] = e->m_transfers; t[i] = e->t;
    }
}
void car_oracle_set_theta(void* h, const double* theta)
{
    car_batch* b = (car_batch*)h;
    for (int i = 0; i < b->E; i++) b->envs[i].theta = theta[i];
}
