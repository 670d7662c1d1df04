/*
 * features_oracle.c — CPU restatement of CleanupFeatures / HarvestFeatures (the 'Cleanup' / 'Harvest' tags) and the
 * contract wrapper's redistribution on top of them, for E independent envs.
 *
 * TEST INFRASTRUCTURE (oracle/): used by tests/, bench.py's cpu_baseline and __graft_entry__.smoke() only — never by
 * the product path.  Pinned against the unmodified reference by tests/golden/features_*.npz.
 *
 * Reference (paths relative to the reference root):
 *   environments/cleanup_features.py  step :156-254, reset :256-284, initialize_arrays :70-101,
 *       initialize_players :103-109, spawn_apples_and_waste :111-125, compute_closest_* :127-154,
 *       compute_probabilities :286-303
 *   environments/harvest_features.py  step :173-287, reset :289-336, spawn_apples :139-151,
 *       count_apples_in_radius :128-137
 *   contract/contract_list.py :22-27, :45-54 ; environments/two_stage_train.py :62-121, :159-187
 *
 * The current apple / waste lists are kept as a birth stamp per map point (0 = absent): list order = stamp order,
 * which is what decides np.argmin ties in compute_closest_*.  Draws: site 10 (spawn-index shuffle), 11 (rotation,
 * call = agent), 12 (k-th random.random() of a step / reset), 7 (contract sample).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define MAXN 8
#define MAXH 48
#define MAXW 64
#define MAXP 256
#define KIND_CLEANUP 0
#define KIND_HARVEST 1
#define SITE_CONTRACT 7
#define SITE_FEAT_ORDER 10
#define SITE_FEAT_ROT 11
#define SITE_FEAT_SPAWN 12
#define CONTRACT_CLEANUP 1
#define CONTRACT_HARVEST_LOCAL 2

typedef struct { int r, c; } pt;

typedef struct {
    int kind, H, W;
    char map[MAXH][MAXW];
    pt spawn[MAXP]; int n_spawn;
    pt apple[MAXP]; int n_apple;
    pt waste[MAXP]; int n_waste; int waste_is_start[MAXP];
    int apple_idx[MAXH][MAXW], waste_idx[MAXH][MAXW];     /* -1 or index into the point list */
    int potential_waste_area;
} fstatic;

typedef struct {
    int n, horizon, contract;
    double theta_low, theta_high, null_prob;
    uint32_t seed, env_id, episode;
    const fstatic* s;
    pt pos[MAXN]; int ori[MAXN];
    uint32_t apple_stamp[MAXP], waste_stamp[MAXP], next_apple, next_waste;
    int n_cur_apple, n_cur_waste;
    int t;
    double theta;
    double m_dirt, m_raw, m_transfers, m_apples, m_low_density;
    double sum_raw[MAXN], tsum_raw[MAXN], sum_tr[MAXN], tsum_tr[MAXN];
} fenv;

typedef struct { int E, n, F; fstatic st; fenv* envs; } fbatch;

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
static uint32_t draw_u32(const fenv* e, uint32_t t, int site, uint32_t call, uint32_t idx)
{
    uint32_t ctr[4] = { idx >> 2, (uint32_t)site | (call << 8), t, e->episode };
    uint32_t key[2] = { e->seed, e->env_id }, out[4];
    philox(ctr, key, out);
    return out[idx & 3];
}
static double draw_f64(const fenv* e, uint32_t t, int site, uint32_t call, uint32_t idx)
{
    return (double)draw_u32(e, t, site, call, idx) * (1.0 / 4294967296.0);
}

static const int MOVE_ACTIONS[4][2] = { { 0, -1 }, { 0, 1 }, { -1, 0 }, { 1, 0 } };
static const int FIRE_DIRECTIONS[4][2] = { { -1, 0 }, { 0, 1 }, { 1, 0 }, { 0, -1 } };

static int is_wall(const fstatic* s, int r, int c) { return r >= 0 && r < s->H && c >= 0 && c < s->W && s->map[r][c] == '@'; }
static int apple_at(const fenv* e, int r, int c)
{
    const fstatic* s = e->s;
    if (r < 0 || r >= s->H || c < 0 || c >= s->W) return -1;
    int i = s->apple_idx[r][c];
    return (i >= 0 && e->apple_stamp[i]) ? i : -1;
}
static int waste_at(const fenv* e, int r, int c)
{
    const fstatic* s = e->s;
    if (r < 0 || r >= s->H || c < 0 || c >= s->W) return -1;
    int i = s->waste_idx[r][c];
    return (i >= 0 && e->waste_stamp[i]) ? i : -1;
}
static int agent_on(const fenv* e, int r, int c)
{
    for (int a = 0; a < e->n; a++) if (e->pos[a].r == r && e->pos[a].c == c) return 1;
    return 0;
}
/* count_apples_in_radius: j*j + k*k <= radius (sic: not squared) over the live list */
static int count_apples_in_radius(const fenv* e, int radius, pt loc)
{
    int cnt = 0;
    for (int j = -radius; j <= radius; j++)
        for (int k = -radius; k <= radius; k++)
            if (j * j + k * k <= radius && apple_at(e, loc.r + j, loc.c + k) >= 0) cnt++;
    return cnt;
}

/* cleanup_features.py:286-303 */
static void compute_probabilities(const fenv* e, double* p_apple, double* p_waste)
{
    const fstatic* s = e->s;
    double waste_density = 0;
    if (s->potential_waste_area > 0) {
        int free_area = s->potential_waste_area - e->n_cur_waste;
        waste_density = 1 - (double)free_area / (double)s->potential_waste_area;
    }
    if (waste_density >= 0.4) { *p_apple = 0; *p_waste = 0; }
    else {
        *p_waste = 0.5;
        if (waste_density <= 0.0) *p_apple = 0.05;
        else *p_apple = (1 - (waste_density - 0.0) / (0.4 - 0.0)) * 0.05;
    }
}

/* cleanup_features.py:111-125 / harvest_features.py:139-151; `t` addresses the draws */
static void spawn(fenv* e, uint32_t t)
{
    const fstatic* s = e->s;
    uint32_t k = 0;
    if (s->kind == KIND_CLEANUP) {
        double pa, pw;
        compute_probabilities(e, &pa, &pw);
        for (int i = 0; i < s->n_apple; i++) {
            if (!e->apple_stamp[i] && !agent_on(e, s->apple[i].r, s->apple[i].c)) {
                double r = draw_f64(e, t, SITE_FEAT_SPAWN, 0, k++);
                if (r < pa) { e->apple_stamp[i] = e->next_apple++; e->n_cur_apple++; }
            }
        }
        for (int i = 0; i < s->n_waste; i++) {
            if (!e->waste_stamp[i]) {
                double r = draw_f64(e, t, SITE_FEAT_SPAWN, 0, k++);
                if (r < pw) { e->waste_stamp[i] = e->next_waste++; e->n_cur_waste++; break; }
            }
        }
    } else {
        static const double SPAWN_PROB[4] = { 0, 0.005, 0.02, 0.05 };
        for (int i = 0; i < s->n_apple; i++) {
            if (!e->apple_stamp[i] && !agent_on(e, s->apple[i].r, s->apple[i].c)) {
                int num = count_apples_in_radius(e, 2, s->apple[i]);      /* live list: sees this loop's earlier spawns */
                double r = draw_f64(e, t, SITE_FEAT_SPAWN, 0, k++);
                if (r < SPAWN_PROB[num < 3 ? num : 3]) { e->apple_stamp[i] = e->next_apple++; e->n_cur_apple++; }
            }
        }
    }
}

/* np.argmin over the list in birth order: smallest (L1 distance, stamp) */
static pt closest(const pt* pts, const uint32_t* stamp, int n, pt p)
{
    pt best = { 0, 0 };
    long bd = -1; uint32_t bs = 0;
    for (int i = 0; i < n; i++) {
        if (!stamp[i]) continue;
        long d = labs((long)pts[i].r - p.r) + labs((long)pts[i].c - p.c);
        if (bd < 0 || d < bd || (d == bd && stamp[i] < bs)) { bd = d; bs = stamp[i]; best = pts[i]; }
    }
    return best;
}

static int feat_dim(int kind, int n) { return kind == KIND_CLEANUP ? 12 + n : 10 + 2 * n; }

static void write_obs(const fenv* e, const int* cleaned, double* obs)
{
    const fstatic* s = e->s;
    const int n = e->n, F = feat_dim(s->kind, n);
    for (int a = 0; a < n; a++) {
        double* o = obs + a * F;
        int cp = a == 0 ? (n > 1 ? 1 : 0) : 0;            /* compute_closest_pos quirk: distances are 0 for every other agent */
        pt ca = closest(s->apple, e->apple_stamp, s->n_apple, e->pos[a]);
        o[0] = e->pos[a].r; o[1] = e->pos[a].c; o[2] = e->ori[a];
        o[3] = e->pos[cp].r; o[4] = e->pos[cp].c; o[5] = e->ori[cp];
        o[6] = ca.r; o[7] = ca.c;
        if (s->kind == KIND_CLEANUP) {
            pt cw = closest(s->waste, e->waste_stamp, s->n_waste, e->pos[a]);
            o[8] = cw.r; o[9] = cw.c; o[10] = e->n_cur_apple; o[11] = e->n_cur_waste;
            for (int i = 0; i < n; i++) o[12 + i] = cleaned ? cleaned[i] : 0;
        } else {
            o[8] = count_apples_in_radius(e, 5, e->pos[a]); o[9] = e->n_cur_apple;
            for (int i = 0; i < 2 * n; i++) o[10 + i] = 0;
        }
    }
}

static void env_reset(fenv* e, uint32_t episode)
{
    const fstatic* s = e->s;
    e->episode = episode;
    /* initialize_arrays */
    memset(e->apple_stamp, 0, sizeof(e->apple_stamp)); memset(e->waste_stamp, 0, sizeof(e->waste_stamp));
    e->next_apple = 1; e->next_waste = 1; e->n_cur_apple = 0; e->n_cur_waste = 0;
    if (s->kind == KIND_CLEANUP) { for (int i = 0; i < s->n_waste; i++) if (s->waste_is_start[i]) { e->waste_stamp[i] = e->next_waste++; e->n_cur_waste++; } }
    else { for (int i = 0; i < s->n_apple; i++) { e->apple_stamp[i] = e->next_apple++; e->n_cur_apple++; } }
    /* initialize_players: random.shuffle(list(range(n_spawn))) -> stable argsort of one key per index */
    { uint32_t keys[MAXP]; int order[MAXP];
      for (int i = 0; i < s->n_spawn; i++) { keys[i] = draw_u32(e, 0, SITE_FEAT_ORDER, 0, (uint32_t)i); order[i] = i; }
      for (int i = 1; i < s->n_spawn; i++) { int o = order[i], j = i - 1; while (j >= 0 && keys[order[j]] > keys[o]) { order[j + 1] = order[j]; j--; } order[j + 1] = o; }
      for (int a = 0; a < e->n; a++) { e->pos[a] = s->spawn[order[a]]; e->ori[a] = (int)(draw_u32(e, 0, SITE_FEAT_ROT, (uint32_t)a, 0) >> 30); } }
    spawn(e, 0);
    e->t = 0;
    e->m_dirt = e->m_raw = e->m_transfers = e->m_apples = e->m_low_density = 0;
    for (int a = 0; a < MAXN; a++) e->sum_raw[a] = e->tsum_raw[a] = e->sum_tr[a] = e->tsum_tr[a] = 0;
    e->theta = 0;
    if (e->contract) {
        double u0 = draw_f64(e, 0, SITE_CONTRACT, 0, 0);
        if (u0 > e->null_prob) { double u1 = draw_f64(e, 0, SITE_CONTRACT, 0, 1); e->theta = e->theta_low + (e->theta_high - e->theta_low) * u1; }
        else e->theta = e->theta_low;
    }
}

/* info [n][4]: cleanup (cleaned_squares, 0, 0, 0); harvest (eaten_apples, eaten_close_apples, 0, 0) */
static void env_step(fenv* e, const int32_t* acts, double* obs, double* rew, double* base_rew, double* transfers,
                     int32_t* info, uint8_t* done)
{
    const fstatic* s = e->s;
    const int n = e->n;
    const uint32_t t_draw = (uint32_t)e->t + 1;
    pt claim[MAXN]; int has[MAXN], order[MAXN], n_order = 0;
    double rewards[MAXN]; int cleaned[MAXN], eaten[MAXN], eaten_close[MAXN];
    for (int a = 0; a < n; a++) { has[a] = 0; rewards[a] = 0.0; cleaned[a] = eaten[a] = eaten_close[a] = 0; }
    /* stay first (cleanup: act == 4; harvest: every act > 3) */
    for (int a = 0; a < n; a++) {
        int stay = s->kind == KIND_CLEANUP ? acts[a] == 4 : acts[a] > 3;
        if (stay) { claim[a] = e->pos[a]; has[a] = 1; order[n_order++] = a; }
    }
    for (int a = 0; a < n; a++) {
        if (acts[a] < 0 || acts[a] > 3) continue;
        pt tmp = { e->pos[a].r + MOVE_ACTIONS[acts[a]][0], e->pos[a].c + MOVE_ACTIONS[acts[a]][1] };
        int taken = 0;
        for (int b = 0; b < n; b++) if (has[b] && claim[b].r == tmp.r && claim[b].c == tmp.c) taken = 1;
        claim[a] = (taken || is_wall(s, tmp.r, tmp.c)) ? e->pos[a] : tmp;
        has[a] = 1; order[n_order++] = a;
    }
    for (int a = 0; a < n; a++) if (has[a]) e->pos[a] = claim[a];
    /* consume in move_squares insertion order */
    for (int k = 0; k < n_order; k++) {
        int a = order[k];
        int i = apple_at(e, e->pos[a].r, e->pos[a].c);
        if (i < 0) continue;
        rewards[a] += 1;
        if (s->kind == KIND_HARVEST) {
            eaten[a] += 1;
            if (count_apples_in_radius(e, 5, e->pos[a]) < 4) { eaten_close[a] += 1; e->m_low_density += 1; }
            e->m_apples += 1;
        }
        e->apple_stamp[i] = 0; e->n_cur_apple--;
    }
    for (int a = 0; a < n; a++) {
        if (acts[a] == 5) e->ori[a] = (e->ori[a] + 1) % 4;
        if (acts[a] == 6) e->ori[a] = ((e->ori[a] - 1) % 4 + 4) % 4;
    }
    if (s->kind == KIND_CLEANUP) {
        for (int a = 0; a < n; a++) {
            if (acts[a] != 7 && acts[a] != 8) continue;
            const int* dir = FIRE_DIRECTIONS[e->ori[a]];
            const int* side = FIRE_DIRECTIONS[(e->ori[a] + 1) % 4];
            pt start[3] = { e->pos[a], { e->pos[a].r + side[0], e->pos[a].c + side[1] }, { e->pos[a].r - side[0], e->pos[a].c - side[1] } };
            for (int b = 0; b < 3; b++)
                for (int j = 0; j < 6; j++) {
                    int r = start[b].r + j * dir[0], c = start[b].c + j * dir[1];
                    if (is_wall(s, r, c)) break;
                    if (acts[a] == 7) {
                        int w = waste_at(e, r, c);
                        if (w >= 0) { e->waste_stamp[w] = 0; e->n_cur_waste--; cleaned[a]++; e->m_dirt += 1; }
                    }
                }
        }
    }
    spawn(e, t_draw);
    write_obs(e, cleaned, obs);
    e->t += 1;
    *done = (uint8_t)(e->t == e->horizon);
    { double raw = 0; for (int a = 0; a < n; a++) raw += rewards[a]; e->m_raw += raw; }
    /* contract transfers + redistribution (two_stage_train.py:71-92) */
    double tr[MAXN], r[MAXN], total = 0;
    const int F = feat_dim(s->kind, n);
    for (int a = 0; a < n; a++) {
        r[a] = rewards[a];
        tr[a] = 0;
        if (e->contract == CONTRACT_CLEANUP) tr[a] = -e->theta * cleaned[a];
        else if (e->contract == CONTRACT_HARVEST_LOCAL) tr[a] = (obs[a * F + 8] < 4 && eaten_close[a] > 0) ? e->theta : 0;
    }
    if (e->contract) {
        for (int i = 0; i < n; i++) {
            r[i] -= tr[i]; total += tr[i];
            for (int j = 0; j < n; j++) if (i != j) r[j] += tr[i] / (n - 1);
        }
        e->m_transfers += total;
    }
    for (int a = 0; a < n; a++) {
        rew[a] = r[a]; base_rew[a] = rewards[a]; transfers[a] = tr[a];
        info[a * 4 + 0] = s->kind == KIND_CLEANUP ? cleaned[a] : eaten[a];
        info[a * 4 + 1] = s->kind == KIND_CLEANUP ? 0 : eaten_close[a];
        info[a * 4 + 2] = info[a * 4 + 3] = 0;
        e->sum_raw[a] += rewards[a]; e->tsum_raw[a] += (double)(e->t - 1) * rewards[a];
        e->sum_tr[a] += r[a]; e->tsum_tr[a] += (double)(e->t - 1) * r[a];
    }
}

static int static_init(fstatic* s, int kind, int H, int W, const char* ascii)
{
    memset(s, 0, sizeof(*s));
    s->kind = kind; s->H = H; s->W = W;
    for (int r = 0; r < H; r++)
        for (int c = 0; c < W; c++) {
            char ch = ascii[r * W + c];
            s->map[r][c] = ch; s->apple_idx[r][c] = -1; s->waste_idx[r][c] = -1;
            pt p = { r, c };
            if (ch == 'P') { if (s->n_spawn >= MAXP) return -1; s->spawn[s->n_spawn++] = p; }
            if (ch == (kind == KIND_CLEANUP ? 'B' : 'A')) { if (s->n_apple >= MAXP) return -1; s->apple_idx[r][c] = s->n_apple; s->apple[s->n_apple++] = p; }
            if (kind == KIND_CLEANUP && (ch == 'H' || ch == 'R')) {
                if (s->n_waste >= MAXP) return -1;
                s->waste_idx[r][c] = s->n_waste; s->waste_is_start[s->n_waste] = ch == 'H'; s->waste[s->n_waste++] = p;
                s->potential_waste_area++;
            }
        }
    return 0;
}

/* ------------------------------------------------------------------ C API (ctypes: oracle/oracle.py) */
void* feat_oracle_create(int kind, int E, int n, int H, int W, const char* ascii, int horizon, int contract,
                         double theta_low, double theta_high, double null_prob, uint32_t seed, uint32_t first_env_id)
{
    if (n < 1 || n > MAXN || H < 1 || H > MAXH || W < 1 || W > MAXW || E < 1) return NULL;
    fbatch* b = (fbatch*)calloc(1, sizeof(fbatch));
    b->E = E; b->n = n; b->F = feat_dim(kind, n);
    if (static_init(&b->st, kind, H, W, ascii) != 0 || b->st.n_spawn < n) { free(b); return NULL; }
    b->envs = (fenv*)calloc((size_t)E, sizeof(fenv));
    for (int i = 0; i < E; i++) {
        fenv* e = &b->envs[i];
        e->n = n; e->horizon = horizon; e->contract = contract; e->theta_low = theta_low; e->theta_high = theta_high;
        e->null_prob = null_prob; e->seed = seed; e->env_id = first_env_id + (uint32_t)i; e->s = &b->st;
    }
    return b;
}
void feat_oracle_destroy(void* h) { fbatch* b = (fbatch*)h; if (b) { free(b->envs); free(b); } }
int feat_oracle_dim(void* h) { return ((fbatch*)h)->F; }

void feat_oracle_reset(void* h, const uint8_t* mask, const uint32_t* episode, double* obs)
{
    fbatch* b = (fbatch*)h;
    for (int i = 0; i < b->E; i++) {
        if (mask && !mask[i]) continue;
        env_reset(&b->envs[i], episode[i]);
        if (obs) write_obs(&b->envs[i], NULL, obs + (size_t)i * b->n * b->F);
    }
}
void feat_oracle_step(void* h, const int32_t* acts, double* obs, double* rew, double* base_rew, double* transfers,
                      int32_t* info, uint8_t* done)
{
    fbatch* b = (fbatch*)h;
    int n = b->n;
#pragma omp parallel for schedule(static) if (b->E > 1)   /* a one-env batch (the live differential tests) stays on the calling thread */
    for (int i = 0; i < b->E; i++)
        env_step(&b->envs[i], acts + (size_t)i * n, obs + (size_t)i * n * b->F, rew + (size_t)i * n, base_rew + (size_t)i * n,
                 transfers + (size_t)i * n, info + (size_t)i * n * 4, done + i);
}
/* feat_oracle_step with a per-env skip byte: an env with skip[i] != 0 is not stepped and its output rows are left as the
   caller passed them (a batch's next-step auto-reset: reset the done envs with a mask, then step the others). */
void feat_oracle_step_skip(void* h, const int32_t* acts, double* obs, double* rew, double* base_rew, double* transfers,
                           int32_t* info, uint8_t* done, const uint8_t* skip)
{
    fbatch* b = (fbatch*)h;
    int n = b->n;
#pragma omp parallel for schedule(static) if (b->E > 1)
    for (int i = 0; i < b->E; i++) {
        if (skip && skip[i]) continue;
        env_step(&b->envs[i], acts + (size_t)i * n, obs + (size_t)i * n * b->F, rew + (size_t)i * n, base_rew + (size_t)i * n,
                 transfers + (size_t)i * n, info + (size_t)i * n * 4, done + i);
    }
}
/* metrics [E][8 + 4*8]: dirt, raw, transfers, apples, low_density, 0, 0, 0, sum_raw[8], tsum_raw[8], sum_tr[8], tsum_tr[8] */
void feat_oracle_get_metrics(void* h, double* out)
{
    fbatch* b = (fbatch*)h;
    for (int i = 0; i < b->E; i++) {
        fenv* e = &b->envs[i];
        double* o = out + (size_t)i * 40;
        o[0] = e->m_dirt; o[1] = e->m_raw; o[2] = e->m_transfers; o[3] = e->m_apples; o[4] = e->m_low_density; o[5] = o[6] = o[7] = 0;
        for (int a = 0; a < MAXN; a++) { o[8 + a] = e->sum_raw[a]; o[16 + a] = e->tsum_raw[a]; o[24 + a] = e->sum_tr[a]; o[32 + a] = e->tsum_tr[a]; }
    }
}
/* state: pos [E][n][2], ori [E][n], apple / waste presence by map cell [E][H][W] (1 apple, 2 waste), theta [E], t [E] */
void feat_oracle_get_state(void* h, int32_t* pos, int32_t* ori, uint8_t* cells, double* theta, int32_t* t)
{
    fbatch* b = (fbatch*)h;
    const fstatic* s = &b->st;
    for (int i = 0; i < b->E; i++) {
        fenv* e = &b->envs[i];
        for (int a = 0; a < b->n; a++) { pos[((size_t)i * b->n + a) * 2] = e->pos[a].r; pos[((size_t)i * b->n + a) * 2 + 1] = e->pos[a].c; ori[(size_t)i * b->n + a] = e->ori[a]; }
        if (cells) {
            uint8_t* c = cells + (size_t)i * s->H * s->W;
            memset(c, 0, (size_t)s->H * s->W);
            for (int k = 0; k < s->n_apple; k++) if (e->apple_stamp[k]) c[s->apple[k].r * s->W + s->apple[k].c] = 1;
            for (int k = 0; k < s->n_waste; k++) if (e->waste_stamp[k]) c[s->waste[k].r * s->W + s->waste[k].c] = 2;
        }
        theta[i] = e->theta; t[i] = e->t;
    }
}
