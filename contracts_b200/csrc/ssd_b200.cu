// ssd_b200.cu — C ABI of libssd_b200.so (see include/ssd_b200.h) and host-side setup.
//
// Build (see __graft_entry__.build / contracts_b200/build.py):
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -fmad=false \
//        -Xcompiler -fPIC -shared -I include -o contracts_b200/libssd_b200.so contracts_b200/csrc/ssd_b200.cu
// -fmad=false: reward / transfer arithmetic must round like the reference's float64 ops.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/ssd_b200.h"
#include "ssd_grid.cuh"
#include "ssd_grid2.cuh"
#include "ssd_grid3.cuh"
#include "ssd_views.cuh"
#include "ssd_selfdrive.cuh"
#include "ssd_features.cuh"
#include "ssd_checkpoint.cuh"
#include "ssd_solver.cuh"

static thread_local char g_create_error[512] = "";

struct ssd_handle {
    ssd_config cfg;
    std::string ascii;
    GridParams gp;
    CarParams cp;
    FeatParams fp;
    int grid_blocks;
    int feat_smem;           // dynamic shared memory of the feature-env kernels
    int car_smem;            // dynamic shared memory of the selfdrive kernels
    int obs_blocks;          // grid of the observe kernel (persistent: CTAs per SM x SMs, or fewer for small batches)
    int logic_smem;          // dynamic shared memory of the logic kernel (cell table + per-warp mask copies)
    bool pdl;                // programmatic dependent launch of the observe / reset kernels behind the logic / observe kernels
    int obs_lay;             // observe kernel specialisation the handle qualifies for (obs_layout_id)
    int logic_lay;           // logic kernel specialisation (logic_layout_id)
    bool logic8;             // the eight-lanes-per-env logic kernel (ssd_grid3.cuh): small batches; SSD_LOGIC8=0 / 1 forces the choice
    int logic8_smem, logic8_blocks;
    cudaEvent_t tev[3];      // ssd_enable_timing: before the logic kernel / between / after the observe (+ reward) kernel
    bool timing;
    uint32_t* d_res;         // u32 [E][8] per-agent result words passed between the step's kernels
    uint8_t* d_beam;         // ssd_record_beams: [E][map_bytes] beam overlay of the last step
    cudaStream_t side;       // ssd_step_host: copy stream + its events (created on first use)
    cudaEvent_t ev_rew, ev_copied;
    // ssd_step_host_async: two slots, each with a device action buffer and a device result block
    struct Slot {
        uint8_t* d_actions; uint8_t* d_block;
        cudaEvent_t ev_up, ev_rew, ev_copied, ev_logic;
        void* host_block; int64_t ticket; bool busy; uint32_t copied_records;
    } slot[2];
    cudaStream_t s_in, s_out;
    int64_t next_ticket;
    uint32_t recent_count[2];
    ssd_host_layout lay;
    uint32_t* d_counter;     // device step counter for SSD_STEP_AUTO: [0] index, [1] CTAs finished
    bool rounds4;            // point lists fit 4 rounds of 32 (selects the observe-kernel variant)
    int64_t launches;
    CkParams ck;             // ssd_checkpoint_*: where each part of an env's row lives (ssd_checkpoint.cuh)
    uint64_t config_tag;     // ssd_checkpoint_get_layout: hash of everything that gives a row its meaning
    // ssd_set_policy_output / ssd_set_flat_policy_output: the one observation form the handle's kernels write
    int form;                // 0: the native form (OBS_U8 / OBS_F64); else 1 + SSD_POLICY_*
    void* pol_rows;          //   the policy image T [E n][3][15][15] (grid worlds) or the flat rows T [E n][W]
    ThetaRows theta_rows;    //   the rows that carry theta: a grid world's contract rows, flat rows under a contract
    int feat_form;           // ssd_set_feature_output (grid worlds, form 0): 1 + its dtype (SSD_FEATURE_F64 / SSD_POLICY_*), rows at
                             // pol_rows; 0: off
    // ssd_solver_enable: the solver queue (ssd_solver.cuh)
    bool solver_on;
    uint32_t* d_resolved;    //   [E] episode whose contract the solver chose, SQ_NONE: none
    uint32_t* d_sq_blocks;   //   [ceil(E / SQ_BLOCK)] pending envs per block of the scan
    uint8_t* d_sq_ok;        //   checkpoint_load without row_ok_dev: the rows that loaded, [sq_ok_cap]
    int sq_ok_cap;
    char err[512];
    std::vector<void*> dev_allocs;
};

// f(std::integral_constant<int, FORM>()) for a runtime observation form: 0, the native form (OBS_U8 / OBS_F64), or
// 1 + SSD_POLICY_*
template <typename F>
static auto by_form(int form, F f)
{
    if (form == 1 + SSD_POLICY_F32) return f(std::integral_constant<int, 1 + SSD_POLICY_F32>());
    if (form == 1 + SSD_POLICY_F16) return f(std::integral_constant<int, 1 + SSD_POLICY_F16>());
    if (form == 1 + SSD_POLICY_BF16) return f(std::integral_constant<int, 1 + SSD_POLICY_BF16>());
    return f(std::integral_constant<int, 0>());
}
typedef void (*obs_kernel_t)(const GridParams, const StepIO, uint32_t*);
// lay: 0, or 1 when the handle matches OBS_LAY_CLEANUP8 (stock cleanup map, 8 agents, dense observation tensor, no feature_obs);
// form: OBS_U8 or the policy form of ssd_set_policy_output (1 + SSD_POLICY_*)
static obs_kernel_t obs_kernel_fn(int kind, bool rounds4, bool feat, int lay = 0, int form = OBS_U8)
{
    return by_form(form, [&](auto F) -> obs_kernel_t {
        constexpr int FORM = decltype(F)::value;
        if (lay == 1 && kind == SSD_ENV_CLEANUP && rounds4 && !feat) return grid_obs_kernel<SSD_ENV_CLEANUP, 4, false, 1, FORM>;
        if (lay == 2 && kind == SSD_ENV_HARVEST && !rounds4 && !feat) return grid_obs_kernel<SSD_ENV_HARVEST, MAX_POINT_ROUNDS, false, 2, FORM>;
        if (kind == SSD_ENV_CLEANUP) {
            if (rounds4) return feat ? grid_obs_kernel<SSD_ENV_CLEANUP, 4, true, 0, FORM> : grid_obs_kernel<SSD_ENV_CLEANUP, 4, false, 0, FORM>;
            return feat ? grid_obs_kernel<SSD_ENV_CLEANUP, MAX_POINT_ROUNDS, true, 0, FORM> : grid_obs_kernel<SSD_ENV_CLEANUP, MAX_POINT_ROUNDS, false, 0, FORM>;
        }
        if (rounds4) return feat ? grid_obs_kernel<SSD_ENV_HARVEST, 4, true, 0, FORM> : grid_obs_kernel<SSD_ENV_HARVEST, 4, false, 0, FORM>;
        return feat ? grid_obs_kernel<SSD_ENV_HARVEST, MAX_POINT_ROUNDS, true, 0, FORM> : grid_obs_kernel<SSD_ENV_HARVEST, MAX_POINT_ROUNDS, false, 0, FORM>;
    });
}
typedef void (*reset_kernel_t)(const GridParams, const uint8_t*, uint8_t*, long long, const StepIO, void*);
static reset_kernel_t reset_kernel_fn(int kind, int form)
{
    return by_form(form, [&](auto F) -> reset_kernel_t {
        constexpr int FORM = decltype(F)::value;
        return kind == SSD_ENV_CLEANUP ? grid_reset_kernel<SSD_ENV_CLEANUP, FORM> : grid_reset_kernel<SSD_ENV_HARVEST, FORM>;
    });
}
// f(std::integral_constant<int, OUT>()) for the dtype of ssd_set_feature_output (SSD_FEATURE_F64 or SSD_POLICY_*)
template <typename F>
static auto by_feature_dtype(int dtype, F f)
{
    if (dtype == SSD_POLICY_F32) return f(std::integral_constant<int, SSD_POLICY_F32>());
    if (dtype == SSD_POLICY_F16) return f(std::integral_constant<int, SSD_POLICY_F16>());
    if (dtype == SSD_POLICY_BF16) return f(std::integral_constant<int, SSD_POLICY_BF16>());
    return f(std::integral_constant<int, SSD_FEATURE_F64>());
}
typedef void (*feature_kernel_t)(const GridParams, uint32_t*, void*, int);
static feature_kernel_t feature_kernel_fn(int kind, bool rounds4, int dtype)
{
    return by_feature_dtype(dtype, [&](auto O) -> feature_kernel_t {
        constexpr int OUT = decltype(O)::value;
        if (kind == SSD_ENV_CLEANUP) return rounds4 ? grid_feature_kernel<SSD_ENV_CLEANUP, 4, OUT> : grid_feature_kernel<SSD_ENV_CLEANUP, MAX_POINT_ROUNDS, OUT>;
        return rounds4 ? grid_feature_kernel<SSD_ENV_HARVEST, 4, OUT> : grid_feature_kernel<SSD_ENV_HARVEST, MAX_POINT_ROUNDS, OUT>;
    });
}
typedef void (*reset_features_kernel_t)(const GridParams, const uint8_t*, void*, int);
static reset_features_kernel_t reset_features_kernel_fn(int kind, int dtype)
{
    return by_feature_dtype(dtype, [&](auto O) -> reset_features_kernel_t {
        constexpr int OUT = decltype(O)::value;
        return kind == SSD_ENV_CLEANUP ? grid_reset_features_kernel<SSD_ENV_CLEANUP, OUT> : grid_reset_features_kernel<SSD_ENV_HARVEST, OUT>;
    });
}
typedef void (*feat_kernel_t)(const FeatParams, const FeatIO, const uint8_t*);
// form: OBS_F64 or the flat policy form of ssd_set_flat_policy_output (1 + SSD_POLICY_*)
static feat_kernel_t feat_kernel_fn(bool cleanup, bool reset_only, int form)
{
    return by_form(form, [&](auto F) -> feat_kernel_t {
        constexpr int FORM = decltype(F)::value;
        if (cleanup) return reset_only ? feat_kernel<true, true, FORM> : feat_kernel<true, false, FORM>;
        return reset_only ? feat_kernel<false, true, FORM> : feat_kernel<false, false, FORM>;
    });
}
typedef void (*car_kernel_t)(const CarParams, const CarIO, const uint8_t*);
static car_kernel_t car_kernel_fn(bool reset_only, int form)
{
    return by_form(form, [&](auto F) -> car_kernel_t {
        constexpr int FORM = decltype(F)::value;
        return reset_only ? car_kernel<true, FORM> : car_kernel<false, FORM>;
    });
}
// bytes of one env's block of the policy image tensor
static long long policy_env_bytes(const GridParams& p, int form)
{
    return (long long)p.n * SSD_OBS_BYTES * (form == 1 + SSD_POLICY_F32 ? 4 : 2);
}
typedef void (*logic_kernel_t)(const GridParams, const StepIO, uint32_t*);
static logic_kernel_t logic_kernel_fn(int kind, int lay)
{
    if (kind == SSD_ENV_CLEANUP) return lay == 1 ? grid_logic_kernel<SSD_ENV_CLEANUP, 1> : grid_logic_kernel<SSD_ENV_CLEANUP, 0>;
    return lay == 2 ? grid_logic_kernel<SSD_ENV_HARVEST, 2> : grid_logic_kernel<SSD_ENV_HARVEST, 0>;
}
static int logic_layout_id(const GridParams& p)
{
    if (const char* e = getenv("SSD_LOGIC_GENERIC")) if (atoi(e)) return 0;
    bool ok = p.kind == SSD_ENV_CLEANUP, ok2 = p.kind == SSD_ENV_HARVEST;
#define LOGIC_CHECK(field, value) ok = ok && p.field == (value);
    LOGIC_LAY_CLEANUP8(LOGIC_CHECK)
#undef LOGIC_CHECK
#define LOGIC_CHECK(field, value) ok2 = ok2 && p.field == (value);
    LOGIC_LAY_HARVEST4(LOGIC_CHECK)
#undef LOGIC_CHECK
    return ok ? 1 : (ok2 ? 2 : 0);
}
// does the handle have the layout the specialised observe kernel assumes?
static int obs_layout_id(const GridParams& p)
{
    if (const char* e = getenv("SSD_OBS_GENERIC")) if (atoi(e)) return 0;
    bool ok = p.kind == SSD_ENV_CLEANUP && p.s_magic == 119304648u, ok2 = p.kind == SSD_ENV_HARVEST && p.s_magic == 76695845u;
#define OBS_CHECK(field, value) ok = ok && p.field == (value);
    OBS_LAY_CLEANUP8(OBS_CHECK)
#undef OBS_CHECK
#define OBS_CHECK(field, value) ok2 = ok2 && p.field == (value);
    OBS_LAY_HARVEST4(OBS_CHECK)
#undef OBS_CHECK
    return ok ? 1 : (ok2 ? 2 : 0);
}

static int fail(ssd_handle* h, int code, const char* fmt, ...)
{
    char* buf = h ? h->err : g_create_error;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, 512, fmt, ap);
    va_end(ap);
    return code;
}
#define CUDA_TRY(h, call)                                                                         \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) return fail(h, SSD_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Every entry point runs on the handle's device whatever the caller's current device is, and leaves the caller's
// current device as it found it.
struct DeviceGuard {
    int prev; bool switched;
    explicit DeviceGuard(int dev) : prev(-1), switched(false)
    {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};
#define ON_DEVICE(h) DeviceGuard device_guard_((h)->cfg.device)

// ceil(p * 2^32) clamped: (u32 * 2^-32 < p) <=> (u32 < T)
static uint32_t prob_threshold(double p)
{
    if (!(p > 0.0)) return 0u;
    double x = ceil(p * 4294967296.0);
    if (x >= 4294967295.0) return 0xFFFFFFFFu;
    return (uint32_t)x;
}

// DEFAULT_COLOURS (map_env.py:24-42) + CLEANUP_COLORS (cleanup_new.py:42-47), packed r | g << 8 | b << 16
static uint32_t rgb(int r, int g, int b) { return (uint32_t)r | ((uint32_t)g << 8) | ((uint32_t)b << 16); }
static void build_palette(uint32_t* pal)   // index = tile byte value: cell codes 0..5, 6 + i = agent i, 15 = outside
{
    const uint32_t v[16] = { rgb(0, 0, 0), rgb(180, 180, 180), rgb(0, 255, 0), rgb(99, 156, 194), rgb(113, 75, 24),
                             rgb(113, 75, 24),
                             rgb(0, 0, 255), rgb(2, 81, 154), rgb(204, 0, 204), rgb(216, 30, 54), rgb(254, 151, 0),
                             rgb(100, 255, 255), rgb(99, 99, 255), rgb(250, 204, 255),
                             0, rgb(0, 0, 0) };
    for (int i = 0; i < 16; i++) pal[i] = v[i];
}

template <typename T>
static int upload(ssd_handle* h, const std::vector<T>& v, const T** out)
{
    void* d = nullptr;
    size_t bytes = (v.size() ? v.size() : 1) * sizeof(T);
    CUDA_TRY(h, cudaMalloc(&d, bytes));
    h->dev_allocs.push_back(d);
    if (v.size()) CUDA_TRY(h, cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = reinterpret_cast<const T*>(d);
    return SSD_OK;
}

// spawn probabilities by #waste cells as integer thresholds, computed with the reference's float64 arithmetic
// (cleanup_new.py:351-368 == cleanup_features.py:286-303; thresholdDepletion 0.4, thresholdRestoration 0.0, 0.5, 0.05)
static void cleanup_probability_table(int area, std::vector<uint32_t>& thr_apple, std::vector<uint8_t>& waste_on)
{
    thr_apple.assign(area + 1, 0u);
    waste_on.assign(area + 1, 0);
    for (int k = 0; k <= area; k++) {
        volatile double waste_density = 0;
        if (area > 0) {
            volatile double ratio = (double)(area - k) / (double)area;
            waste_density = 1 - ratio;
        }
        double pa, pw;
        if (waste_density >= 0.4) { pa = 0; pw = 0; }
        else {
            pw = 0.5;
            if (waste_density <= 0.0) pa = 0.05;
            else {
                volatile double frac = (waste_density - 0.0) / (0.4 - 0.0);
                volatile double one_minus = 1 - frac;
                pa = one_minus * 0.05;
            }
        }
        thr_apple[k] = prob_threshold(pa);
        waste_on[k] = pw != 0;
    }
}

template <typename T>
static int dev_zalloc(ssd_handle* h, size_t count, T** out)
{
    void* d = nullptr;
    CUDA_TRY(h, cudaMalloc(&d, (count ? count : 1) * sizeof(T)));
    h->dev_allocs.push_back(d);
    CUDA_TRY(h, cudaMemset(d, 0, (count ? count : 1) * sizeof(T)));
    *out = reinterpret_cast<T*>(d);
    return SSD_OK;
}

// the dynamic shared-memory limit of every kernel of the handle's step and reset in observation form `form` (0 at create,
// the policy form when an output is set)
static int set_form_smem(ssd_handle* h, int form)
{
    const int kind = h->cfg.env_kind;
    if (kind == SSD_ENV_SELFDRIVE) {
        for (int q = 0; q < 2; q++)
            CUDA_TRY(h, cudaFuncSetAttribute((const void*)car_kernel_fn(q != 0, form), cudaFuncAttributeMaxDynamicSharedMemorySize, h->car_smem));
    } else if (kind == SSD_ENV_CLEANUP_FEATURES || kind == SSD_ENV_HARVEST_FEATURES) {
        for (int q = 0; q < 2; q++)
            CUDA_TRY(h, cudaFuncSetAttribute((const void*)feat_kernel_fn(kind == SSD_ENV_CLEANUP_FEATURES, q != 0, form),
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, h->feat_smem));
    } else {
        const int smem = h->gp.g2_smem_bytes;
        CUDA_TRY(h, cudaFuncSetAttribute((const void*)reset_kernel_fn(kind, form), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        for (int feat = 0; feat < 2; feat++)
            CUDA_TRY(h, cudaFuncSetAttribute((const void*)obs_kernel_fn(kind, h->rounds4, feat != 0, 0, form),
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        if (h->obs_lay) CUDA_TRY(h, cudaFuncSetAttribute((const void*)obs_kernel_fn(kind, h->rounds4, false, h->obs_lay, form),
                                                         cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    }
    return SSD_OK;
}

// ---------------------------------------------------------------------------------------------
static int setup_grid(ssd_handle* h)
{
    const ssd_config& c = h->cfg;
    GridParams& p = h->gp;
    memset(&p, 0, sizeof(p));
    const int H = c.map_h, W = c.map_w, n = c.num_agents;
    if (H < 1 || W < 1 || H > 48 || W > 64) return fail(h, SSD_EINVAL, "map size %dx%d out of range (max 48x64)", H, W);
    if (!c.ascii_map || (int)h->ascii.size() != H * W) return fail(h, SSD_EINVAL, "ascii_map must hold map_h*map_w chars");
    const bool cleanup = c.env_kind == SSD_ENV_CLEANUP;
    p.E = c.num_envs; p.n = n; p.H = H; p.W = W;
    p.Wp = round_up(W, 4); p.S = 8 + p.Wp + 8; p.TH = H + 2 * SSD_VIEW;
    const int Hp = round_up(H, 4);
    p.S2 = 8 + Hp + 8;
    p.s_magic = (uint32_t)((4294967296ull + p.S - 1) / p.S);
    p.map_bytes = round_up(H * p.Wp, 16);
    p.reward_mode = c.flags & (SSD_FLAG_COLLECTIVE_REWARD | SSD_FLAG_INEQUITY_AVERSE);
    if (c.flags & ~(SSD_FLAG_COLLECTIVE_REWARD | SSD_FLAG_INEQUITY_AVERSE)) return fail(h, SSD_EINVAL, "unknown flags 0x%x", c.flags);
    if ((p.reward_mode & RM_INEQUITY) && n < 2)          // assert self.num_agents > 1 (map_env.py:294)
        return fail(h, SSD_EINVAL, "inequity_averse_reward needs more than one agent");
    p.alpha = c.env_params[0]; p.beta = c.env_params[1];
    p.hdr_bytes = p.reward_mode ? RO_XSIZE : RO_SIZE;
    p.rec_stride = round_up(p.hdr_bytes, 128);           // 512 (640 shaped): every env's hot line is one aligned 128-byte line
    p.kind = c.env_kind; p.contract = c.contract_kind; p.horizon = c.horizon;
    p.seed = c.seed; p.first_env_id = c.first_env_id;
    p.theta_low = c.theta_low; p.theta_high = c.theta_high; p.null_prob = c.null_prob;
    p.F = cleanup ? 12 + n : 10 + 2 * n;

    // parse the map like MapEnv.__init__ / CleanupEnv.__init__ / HarvestEnv.__init__.  Static part: walls, river, stream;
    // dynamic part: apple points ('B' cleanup, 'A' harvest) and waste points ('H' / 'R'), in row-major (canonical) order.
    p.tile_r16 = round_up(p.TH * p.S + 1, 16);                          // + a spare sink byte behind T and behind T2 (see below)
    const int tile2_bytes = round_up((p.Wp + 2 * SSD_VIEW) * p.S2 + 1, 16);
    p.tile2_off = p.tile_r16;
    p.g2_stage = p.tile2_off + tile2_bytes;
    std::vector<uint16_t> spawn, apple_rc, waste_rc, apple_c, waste_c, cell_info(round_up(H * p.Wp, 8), 0);
    // point slots beyond a list point at the spare bytes behind T / T2: rewriting "their" cell is harmless
    const uint32_t sink = (uint32_t)(p.TH * p.S) | ((uint32_t)(p.tile2_off + (p.Wp + 2 * SSD_VIEW) * p.S2) << 16);
    std::vector<uint32_t> apple_pt(32 * MAX_POINT_ROUNDS, sink), waste_pt(32 * MAX_POINT_ROUNDS, sink);
    std::vector<uint8_t> base_map(p.map_bytes, (uint8_t)C_OUTSIDE), tile0(p.g2_stage, (uint8_t)C_OUTSIDE);
    auto rc16 = [](int r, int col) { return (uint16_t)((r << 8) | col); };
    auto off = [&](int r, int col) { return (uint32_t)((r + SSD_VIEW) * p.S + 8 + col); };
    auto off2 = [&](int r, int col) { return (uint32_t)((col + SSD_VIEW) * p.S2 + 8 + r); };           // within T2
    int n_spawn_unique = 0, n_waste_start = 0, na = 0, nw = 0;
    for (int r = 0; r < H; r++)
        for (int col = 0; col < W; col++) {
            const char ch = h->ascii[r * W + col];
            uint8_t code = C_EMPTY;                       // the cell's code with its dynamic content OFF
            uint16_t info = 0;
            if (ch == '@') { code = C_WALL; info = CI_WALL; }
            if (ch == 'P') { spawn.push_back((uint16_t)off(r, col)); n_spawn_unique++; if (cleanup) spawn.push_back((uint16_t)off(r, col)); }
            const bool apple_point = cleanup ? ch == 'B' : ch == 'A';
            const bool waste_point = cleanup && (ch == 'H' || ch == 'R');
            if (cleanup && ch == 'S') code = C_STREAM;
            if (apple_point || waste_point) {
                if ((apple_point ? na : nw) >= 32 * MAX_POINT_ROUNDS)
                    return fail(h, SSD_EUNSUPPORTED, "more than %d apple or waste points", 32 * MAX_POINT_ROUNDS);
                const uint32_t packed = off(r, col) | ((p.tile2_off + off2(r, col)) << 16);       // both relative to the T base
                if (apple_point) {
                    if (!cleanup) p.reset_amask[na >> 5] |= 1u << (na & 31);       // harvest starts with every apple (harvest_new.py:143-156)
                    apple_pt[na] = packed; apple_rc.push_back(rc16(r, col)); apple_c.push_back((uint16_t)(r * p.Wp + col));
                    info = (uint16_t)(CI_APPLE | na); na++;
                } else {
                    code = C_RIVER;
                    if (ch == 'H') { p.reset_wmask[nw >> 5] |= 1u << (nw & 31); n_waste_start++; }
                    waste_pt[nw] = packed; waste_rc.push_back(rc16(r, col)); waste_c.push_back((uint16_t)(r * p.Wp + col));
                    info = (uint16_t)(CI_WASTE | nw); nw++;
                }
            }
            base_map[r * p.Wp + col] = code;
            cell_info[r * p.Wp + col] = info;
            tile0[off(r, col)] = code;
            tile0[p.tile2_off + off2(r, col)] = code;
        }
    // canonical spawn order is the sorted list (row-major offsets are already sorted; duplicates adjacent)
    if (n_spawn_unique < n) return fail(h, SSD_EINVAL, "map has %d spawn points for %d agents", n_spawn_unique, n);
    if ((int)spawn.size() > 128) return fail(h, SSD_EUNSUPPORTED, "more than 128 spawn-list entries");
    if (p.g2_stage > 0xFFFF) return fail(h, SSD_EUNSUPPORTED, "tile offsets exceed 16 bits");
    p.n_apple = na; p.n_waste = nw; p.n_spawn = (int)spawn.size();
    p.n_waste_start = n_waste_start;
    h->rounds4 = p.n_apple <= 128 && p.n_waste <= 128;
    p.mw = h->rounds4 ? 4 : MAX_POINT_ROUNDS;

    std::vector<uint32_t> thr_apple;
    std::vector<uint8_t> waste_on;
    cleanup_probability_table(p.n_waste, thr_apple, waste_on);
    const double SPAWN_PROB[4] = { 0, 0.005, 0.02, 0.05 };           // harvest_new.py:34
    for (int i = 0; i < 4; i++) p.thr_harvest[i] = prob_threshold(SPAWN_PROB[i]);
    p.thr_waste = prob_threshold(0.5);

    std::vector<uint32_t> pal(16);
    build_palette(pal.data());

    int rc;
    if ((rc = upload(h, pal, &p.pal))) return rc;
    if ((rc = upload(h, apple_pt, &p.apple_pt))) return rc;
    if ((rc = upload(h, waste_pt, &p.waste_pt))) return rc;
    if ((rc = upload(h, spawn, &p.spawn_pts))) return rc;
    if ((rc = upload(h, apple_rc, &p.apple_rc))) return rc;
    if ((rc = upload(h, waste_rc, &p.waste_rc))) return rc;
    if ((rc = upload(h, apple_c, &p.apple_c))) return rc;
    if ((rc = upload(h, waste_c, &p.waste_c))) return rc;
    if ((rc = upload(h, thr_apple, &p.thr_apple))) return rc;
    if ((rc = upload(h, waste_on, &p.waste_on))) return rc;
    if ((rc = upload(h, tile0, &p.tile0))) return rc;
    if ((rc = upload(h, cell_info, &p.cell_info))) return rc;
    {   // the static part of a beam fired from (cell, orientation): update_map_fire (map_env.py:721-814) walks three rays —
        // centre: along 1..5; right / left: beside the shooter, along 0..4 — and a ray stops at a wall or outside the map
        std::vector<uint4> beam_tab((size_t)H * p.Wp * 4 * 2, make_uint4(0u, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu));
        const int RAYPOS[3] = { 0, 9, 16 };                               // RAY_L, RAY_C, RAY_R (ssd_grid2.cuh)
        for (int r = 0; r < H; r++)
            for (int col = 0; col < W; col++)
                for (int o = 0; o < 4; o++) {
                    const int dr = o == ORI_UP ? -1 : (o == ORI_DOWN ? 1 : 0), dc = o == ORI_RIGHT ? 1 : (o == ORI_LEFT ? -1 : 0);
                    const int o1 = (o + 1) & 3;                           // right = clockwise of the firing direction
                    const int rr = o1 == ORI_UP ? -1 : (o1 == ORI_DOWN ? 1 : 0), rcl = o1 == ORI_RIGHT ? 1 : (o1 == ORI_LEFT ? -1 : 0);
                    uint32_t wall = 0;
                    uint8_t widx[16];
                    memset(widx, 0xFF, sizeof(widx));
                    for (int b = 0; b < 3; b++)                           // left, centre, right
                        for (int i = 0; i < 5; i++) {
                            const int along = b == 1 ? i + 1 : i, across = b == 0 ? -1 : (b == 1 ? 0 : 1);
                            const int cr = r + along * dr + across * rr, cc = col + along * dc + across * rcl;
                            uint16_t info = CI_WALL;
                            if (cr >= 0 && cr < H && cc >= 0 && cc < W) info = cell_info[cr * p.Wp + cc];
                            if (info & CI_WALL) wall |= 1u << (RAYPOS[b] + i);
                            if (info & CI_WASTE) widx[5 * b + i] = (uint8_t)(info & CI_IDX);
                        }
                    uint32_t w4[4];
                    memcpy(w4, widx, 16);
                    uint4* e = &beam_tab[((size_t)(r * p.Wp + col) * 4 + o) * 2];
                    e[0] = make_uint4(wall, w4[0], w4[1], w4[2]);
                    e[1] = make_uint4(w4[3], 0u, 0u, 0u);
                }
        if ((rc = upload(h, beam_tab, &p.beam_tab))) return rc;
    }
    if ((rc = upload(h, base_map, &p.base_map))) return rc;

    // shared memory of the observe / reset kernels: CTA tables, then per warp [T | T2 | stage | misc]
    p.obs_items = (SSD_OBSW * n + 3) / 4;
    p.stage_r16 = round_up(p.obs_items * 180 + 16, 16);
    if (p.stage_r16 < (SCRATCH_DRAWS + 2 * SCRATCH_KEYS) * 4) p.stage_r16 = (SCRATCH_DRAWS + 2 * SCRATCH_KEYS) * 4;
    p.sm_thr = 64;
    p.sm_won = p.sm_thr + round_up((p.n_waste + 1) * 4, 16);
    p.sm_apple_rc = p.sm_won + round_up(p.n_waste + 1, 16);
    p.sm_waste_rc = p.sm_apple_rc + round_up(p.n_apple * 2, 16);
    p.sm_warp0 = p.sm_waste_rc + round_up(p.n_waste * 2, 16);
    p.g2_misc = p.g2_stage + p.stage_r16;
    p.g2_warp_bytes = p.g2_misc + MISC_BYTES;
    p.g2_smem_bytes = p.sm_warp0 + OBS_WARPS * p.g2_warp_bytes;
    static_assert(OBS_WARPS == GRID_WARPS, "the reset kernel shares the observe kernel's shared-memory layout");

    void* st = nullptr;
    size_t bytes = (size_t)p.E * p.rec_stride;
    CUDA_TRY(h, cudaMalloc(&st, bytes));
    h->dev_allocs.push_back(st);
    CUDA_TRY(h, cudaMemset(st, 0, bytes));
    p.state = (uint8_t*)st;

    int sms = 0, per_sm = 0;
    CUDA_TRY(h, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c.device));
    h->obs_lay = obs_layout_id(p);
    if ((rc = set_form_smem(h, 0))) return rc;
    CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)reset_kernel_fn(c.env_kind, OBS_U8), GRID_THREADS,
                                                              p.g2_smem_bytes));
    if (per_sm < 1) return fail(h, SSD_EUNSUPPORTED, "reset kernel does not fit on an SM (smem %d B)", p.g2_smem_bytes);
    int want = (p.E + GRID_WARPS - 1) / GRID_WARPS;
    h->grid_blocks = want < sms * per_sm ? want : sms * per_sm;

    // observe kernel: persistent grid at the achievable occupancy; logic kernel: cell table + per-warp mask copies
    int per_sm2 = 0;
    CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm2, (const void*)obs_kernel_fn(c.env_kind, h->rounds4, false),
                                                              OBS_WARPS * 32, p.g2_smem_bytes));
    if (per_sm2 < 1) return fail(h, SSD_EUNSUPPORTED, "observe kernel does not fit on an SM (smem %d B)", p.g2_smem_bytes);
    const int want_obs = (p.E + OBS_WARPS - 1) / OBS_WARPS;
    h->obs_blocks = want_obs < sms * per_sm2 ? want_obs : sms * per_sm2;
    h->logic_smem = round_up(H * p.Wp * 2, 16) + LOGIC_WARPS * 2 * p.mw * 32 * 4;
    h->logic_lay = logic_layout_id(p);
    {   // eight lanes per env: persistent CTAs, as many as are resident at once
        // Measured (1 x B200): at E = 16384 (n = 4) the octet kernel takes 13.6 us against 15.8 us for the thread-per-env kernel, whose
        // time there is the latency of one warp's chain; at E = 131072 (n = 8) 75 us against 45 us — it executes ~3 x the warp-
        // instructions per env (sequential beams four envs per warp-iteration instead of 32) and loses once the GPU is full.
        const char* e8 = getenv("SSD_LOGIC8");
        h->logic8 = e8 ? e8[0] != '0' : p.E <= 24576;
        h->logic8_smem = round_up(H * p.Wp * 2, 16) + L8_ENVS_PER_CTA * L8_OCT_WORDS * 4;
        const void* fn8 = cleanup ? (const void*)grid_logic8_kernel<SSD_ENV_CLEANUP> : (const void*)grid_logic8_kernel<SSD_ENV_HARVEST>;
        CUDA_TRY(h, cudaFuncSetAttribute(fn8, cudaFuncAttributeMaxDynamicSharedMemorySize, h->logic8_smem));
        int dev8 = 0, sms8 = 0, per_sm8 = 0;
        CUDA_TRY(h, cudaGetDevice(&dev8));
        CUDA_TRY(h, cudaDeviceGetAttribute(&sms8, cudaDevAttrMultiProcessorCount, dev8));
        CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm8, fn8, L8_THREADS, (size_t)h->logic8_smem));
        h->logic8_blocks = std::max(1, std::min((p.E + L8_ENVS_PER_CTA - 1) / L8_ENVS_PER_CTA, sms8 * std::max(per_sm8, 1)));
    }
    CUDA_TRY(h, cudaFuncSetAttribute((const void*)logic_kernel_fn(c.env_kind, 0), cudaFuncAttributeMaxDynamicSharedMemorySize, h->logic_smem));
    if (h->logic_lay)
        CUDA_TRY(h, cudaFuncSetAttribute((const void*)logic_kernel_fn(c.env_kind, h->logic_lay), cudaFuncAttributeMaxDynamicSharedMemorySize, h->logic_smem));
    if (getenv("SSD_DEBUG")) fprintf(stderr, "[ssd] observe kernel: %d warps/CTA, %d CTAs/SM, %d B smem/CTA, grid %d; logic smem %d B\n",
                                     OBS_WARPS, per_sm2, p.g2_smem_bytes, h->obs_blocks, h->logic_smem);
    if ((rc = dev_zalloc(h, (size_t)p.E * SSD_MAXN, &h->d_res))) return rc;
    if ((rc = dev_zalloc(h, 2, &p.obs_ctr))) return rc;
    h->pdl = !(getenv("SSD_NO_PDL") && atoi(getenv("SSD_NO_PDL")) != 0);
    {   // observe kernel schedule: ~5/8 of every warp's envs static, the tail dynamic (SSD_OBS_STATIC_PCT overrides, 100 = all static)
        const int per_warp = p.E / (h->obs_blocks * OBS_WARPS);
        int pct = 62;
        if (const char* e = getenv("SSD_OBS_STATIC_PCT")) pct = std::max(0, std::min(100, atoi(e)));
        p.obs_static_iters = pct >= 100 ? (p.E + h->obs_blocks * OBS_WARPS - 1) / (h->obs_blocks * OBS_WARPS) : per_warp * pct / 100;
    }
    return SSD_OK;
}

// ---------------------------------------------------------------------------------------------
static int setup_selfdrive(ssd_handle* h)
{
    const ssd_config& c = h->cfg;
    CarParams& p = h->cp;
    memset(&p, 0, sizeof(p));
    p.E = c.num_envs; p.n = c.num_agents; p.D = 2 * (c.num_agents + 1) + 3; p.contract = c.contract_kind;
    p.low_bound = c.env_params[0]; p.high_bound = c.env_params[1]; p.start_vel = c.env_params[2]; p.start_vel_amb = c.env_params[3];
    if (!(p.low_bound < p.high_bound)) return fail(h, SSD_EINVAL, "selfdrive: env_params must hold low_bound < high_bound");
    p.theta_low = c.theta_low; p.theta_high = c.theta_high; p.null_prob = c.null_prob;
    p.seed = c.seed; p.first_env_id = c.first_env_id;
    const size_t E = (size_t)p.E;
    int rc;
    if ((rc = dev_zalloc(h, E * p.n, &p.pos))) return rc;
    if ((rc = dev_zalloc(h, E * p.n, &p.vel))) return rc;
    if ((rc = dev_zalloc(h, E, &p.theta))) return rc;
    if ((rc = dev_zalloc(h, E, &p.m_transfers))) return rc;
    if ((rc = dev_zalloc(h, E, &p.dist_front))) return rc;
    if ((rc = dev_zalloc(h, E, &p.crossed))) return rc;
    if ((rc = dev_zalloc(h, E, &p.meta))) return rc;
    if ((rc = dev_zalloc(h, E, &p.t))) return rc;
    if ((rc = dev_zalloc(h, E, &p.episode))) return rc;
    p.warp_doubles = (4 * p.n * p.D + 1) / 2 * 2 + 4 * CAR_OCT_DOUBLES;
    h->car_smem = CAR_WARPS * p.warp_doubles * (int)sizeof(double);
    if ((rc = set_form_smem(h, 0))) return rc;
    {   // persistent CTAs: as many as are resident at once
        int dev = 0, sms = 0, per_sm = 0;
        CUDA_TRY(h, cudaGetDevice(&dev));
        CUDA_TRY(h, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)car_kernel_fn(false, OBS_F64), CAR_THREADS, (size_t)h->car_smem));
        h->grid_blocks = std::max(1, std::min((p.E + CAR_ENVS_PER_CTA - 1) / CAR_ENVS_PER_CTA, sms * std::max(per_sm, 1)));
        if (getenv("SSD_DEBUG")) fprintf(stderr, "[ssd] selfdrive kernel: %d CTAs/SM, %d B smem/CTA, grid %d, %d envs/round\n",
                                         per_sm, h->car_smem, h->grid_blocks, h->grid_blocks * CAR_ENVS_PER_CTA);
    }
    return SSD_OK;
}

static int setup_features(ssd_handle* h)
{
    const ssd_config& c = h->cfg;
    FeatParams& p = h->fp;
    memset(&p, 0, sizeof(p));
    const int H = c.map_h, W = c.map_w, n = c.num_agents;
    const bool cleanup = c.env_kind == SSD_ENV_CLEANUP_FEATURES;
    if (H < 1 || W < 1 || H > 255 || W > 255) return fail(h, SSD_EINVAL, "map size %dx%d out of range", H, W);
    // the closest-point search packs an L1 distance |dr| + |dc| into one key byte per agent (VABSDIFF4, ssd_features.cuh):
    // it must stay below 255, also against the (127, 127) padding entries
    if (H + W - 2 > 254) return fail(h, SSD_EUNSUPPORTED, "feature envs: map_h + map_w - 2 = %d exceeds 254 (distance keys are one byte)", H + W - 2);
    if (!c.ascii_map || (int)h->ascii.size() != H * W) return fail(h, SSD_EINVAL, "ascii_map must hold map_h*map_w chars");
    p.E = c.num_envs; p.n = n; p.kind = c.env_kind; p.H = H; p.W = W; p.horizon = c.horizon; p.contract = c.contract_kind;
    p.F = cleanup ? 12 + n : 10 + 2 * n;
    p.seed = c.seed; p.first_env_id = c.first_env_id;
    p.theta_low = c.theta_low; p.theta_high = c.theta_high; p.null_prob = c.null_prob;
    std::vector<uint8_t> wall(H * W, 0), waste_start;
    std::vector<int16_t> apple_idx(H * W, -1), waste_idx(H * W, -1);
    std::vector<uint16_t> apple_rc, waste_rc, spawn_rc;
    for (int r = 0; r < H; r++)
        for (int col = 0; col < W; col++) {
            const char ch = h->ascii[r * W + col];
            const uint16_t rc = (uint16_t)((r << 8) | col);
            if (ch == '@') wall[r * W + col] = 1;
            if (ch == 'P') spawn_rc.push_back(rc);
            if (ch == (cleanup ? 'B' : 'A')) { apple_idx[r * W + col] = (int16_t)apple_rc.size(); apple_rc.push_back(rc); }
            if (cleanup && (ch == 'H' || ch == 'R')) {
                waste_idx[r * W + col] = (int16_t)waste_rc.size(); waste_rc.push_back(rc); waste_start.push_back(ch == 'H');
            }
        }
    if ((int)spawn_rc.size() < n) return fail(h, SSD_EINVAL, "map has %d spawn points for %d agents", (int)spawn_rc.size(), n);
    if (apple_rc.size() > 32 * FEAT_MASK_WORDS || waste_rc.size() > 32 * FEAT_MASK_WORDS)
        return fail(h, SSD_EUNSUPPORTED, "more than %d apple or waste points", 32 * FEAT_MASK_WORDS);
    p.n_apple = (int)apple_rc.size(); p.n_waste = (int)waste_rc.size(); p.n_spawn = (int)spawn_rc.size(); p.potential = p.n_waste;
    p.nwa = (p.n_apple + 31) / 32; p.nww = (p.n_waste + 31) / 32;
    p.LA = std::max(16, (p.n_apple + 15) / 16 * 16); p.LW = std::max(16, (p.n_waste + 15) / 16 * 16); p.LS = p.LA + p.LW;
    p.sm_static = 2 * 2 * 32 * FEAT_MASK_WORDS; p.oct_bytes = 256 + p.LA + p.LW;     // two 256-entry uint16 point tables
    const int nwa = std::max(p.nwa, 1), nww = std::max(p.nww, 1);
    // 3x3 neighbours of an apple point (j*j + k*k <= APPLE_RADIUS = 2, harvest_features.py:139-151) as a mask over the points
    std::vector<uint32_t> nbr_mask(std::max<size_t>(apple_rc.size(), 1) * nwa, 0u);
    for (size_t i = 0; i < apple_rc.size(); i++)
        for (int j = -1; j <= 1; j++)
            for (int k = -1; k <= 1; k++) {
                if (!j && !k) continue;
                const int r = (apple_rc[i] >> 8) + j, col = (apple_rc[i] & 255) + k;
                if (r < 0 || r >= H || col < 0 || col >= W || apple_idx[r * W + col] < 0) continue;
                const int q = apple_idx[r * W + col];
                nbr_mask[i * nwa + (q >> 5)] |= 1u << (q & 31);
            }
    // count_apples_in_radius(5, cell) (harvest_features.py:128-137): the apple points with j*j + k*k <= 5 around a cell
    std::vector<uint32_t> near5((size_t)H * W * nwa, 0u);
    // cleaning beam fired from (cell, orientation) (cleanup_features.py:196-219): the waste points on its three rays — each ray
    // starts on the agent's own row / column of cells, runs 6 cells, skips cells outside the map and stops at the first wall
    std::vector<uint32_t> beam_tab((size_t)H * W * 4 * nww, 0u);
    for (int r0 = 0; r0 < H; r0++)
        for (int c0 = 0; c0 < W; c0++) {
            for (int j = -2; j <= 2; j++)
                for (int k = -2; k <= 2; k++) {
                    if (j * j + k * k > 5) continue;
                    const int r = r0 + j, col = c0 + k;
                    if (r < 0 || r >= H || col < 0 || col >= W || apple_idx[r * W + col] < 0) continue;
                    const int q = apple_idx[r * W + col];
                    near5[(size_t)(r0 * W + c0) * nwa + (q >> 5)] |= 1u << (q & 31);
                }
            if (!cleanup) continue;
            for (int o = 0; o < 4; o++) {
                const int o1 = (o + 1) & 3;
                const int dr = o == 0 ? -1 : (o == 2 ? 1 : 0), dc = o == 1 ? 1 : (o == 3 ? -1 : 0);
                const int sr = o1 == 0 ? -1 : (o1 == 2 ? 1 : 0), sc = o1 == 1 ? 1 : (o1 == 3 ? -1 : 0);
                uint32_t* row = &beam_tab[((size_t)(r0 * W + c0) * 4 + o) * nww];
                for (int b = 0; b < 3; b++) {
                    const int br = r0 + (b == 1 ? sr : (b == 2 ? -sr : 0)), bc = c0 + (b == 1 ? sc : (b == 2 ? -sc : 0));
                    for (int j = 0; j < 6; j++) {
                        const int r = br + j * dr, col = bc + j * dc;
                        if (r < 0 || r >= H || col < 0 || col >= W) continue;
                        if (wall[r * W + col]) break;
                        const int wi = waste_idx[r * W + col];
                        if (wi >= 0) row[wi >> 5] |= 1u << (wi & 31);
                    }
                }
            }
        }
    std::vector<uint32_t> start_mask(FEAT_MASK_WORDS, 0u);
    for (size_t i = 0; i < waste_start.size(); i++) if (waste_start[i]) start_mask[i >> 5] |= 1u << (i & 31);
    std::vector<uint32_t> thr_apple;
    std::vector<uint8_t> waste_on;
    cleanup_probability_table(p.potential, thr_apple, waste_on);
    const double SPAWN_PROB[4] = { 0, 0.005, 0.02, 0.05 };           // harvest_features.py:36 (increasing: the kernel ranks a draw against them)
    for (int i = 0; i < 4; i++) p.thr_harvest[i] = prob_threshold(SPAWN_PROB[i]);
    p.thr_waste = prob_threshold(0.5);
    if (apple_rc.empty()) apple_rc.push_back(0);
    if (waste_rc.empty()) waste_rc.push_back(0);
    int rc;
    if ((rc = upload(h, wall, &p.wall))) return rc;
    if ((rc = upload(h, apple_idx, &p.apple_idx))) return rc;
    if ((rc = upload(h, waste_idx, &p.waste_idx))) return rc;
    if ((rc = upload(h, apple_rc, &p.apple_rc))) return rc;
    if ((rc = upload(h, waste_rc, &p.waste_rc))) return rc;
    if ((rc = upload(h, spawn_rc, &p.spawn_rc))) return rc;
    if ((rc = upload(h, start_mask, &p.waste_start_mask))) return rc;
    if ((rc = upload(h, thr_apple, &p.thr_apple))) return rc;
    if ((rc = upload(h, waste_on, &p.waste_on))) return rc;
    if ((rc = upload(h, beam_tab, &p.beam_tab))) return rc;
    if ((rc = upload(h, near5, &p.near5))) return rc;
    if ((rc = upload(h, nbr_mask, &p.nbr_mask))) return rc;
    const size_t E = (size_t)p.E;
    if ((rc = dev_zalloc(h, E * FR_WORDS, &p.rec))) return rc;
    if ((rc = dev_zalloc(h, E * p.LS, &p.lists))) return rc;
    if ((rc = dev_zalloc(h, E * 8, &p.metrics))) return rc;
    if ((rc = dev_zalloc(h, E * n, &p.sum_raw))) return rc;
    if ((rc = dev_zalloc(h, E * n, &p.tsum_raw))) return rc;
    if ((rc = dev_zalloc(h, E * n, &p.sum_tr))) return rc;
    if ((rc = dev_zalloc(h, E * n, &p.tsum_tr))) return rc;
    h->feat_smem = p.sm_static + FEAT_ENVS_PER_CTA * p.oct_bytes;
    if (h->feat_smem > 200 * 1024) return fail(h, SSD_EUNSUPPORTED, "feature envs: %d bytes of shared memory per CTA", h->feat_smem);
    if ((rc = set_form_smem(h, 0))) return rc;
    // persistent CTAs: as many as are resident at once (a warp takes four envs per round)
    {
        int dev = 0, sms = 0, per_sm = 0;
        CUDA_TRY(h, cudaGetDevice(&dev));
        CUDA_TRY(h, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)feat_kernel_fn(cleanup, false, OBS_F64), FEAT_THREADS,
                                                              (size_t)h->feat_smem));
        const int groups = (p.E + FEAT_ENVS_PER_CTA - 1) / FEAT_ENVS_PER_CTA;
        h->grid_blocks = std::max(1, std::min(groups, sms * std::max(per_sm, 1)));
        if (getenv("SSD_DEBUG")) fprintf(stderr, "[ssd] feature kernel: %d CTAs/SM, %d B smem/CTA, grid %d, %d envs/round\n",
                                         per_sm, h->feat_smem, h->grid_blocks, h->grid_blocks * FEAT_ENVS_PER_CTA);
    }
    return SSD_OK;
}

// ---------------------------------------------------------------------------------------------
// checkpoint rows (include/ssd_b200.h documents the layout per kind)
static uint64_t fnv1a(uint64_t h, const void* data, size_t bytes)
{
    const uint8_t* b = (const uint8_t*)data;
    for (size_t i = 0; i < bytes; i++) { h ^= b[i]; h *= 1099511628211ull; }
    return h;
}
// every ssd_config field except num_envs, first_env_id, seed, device and struct_size (and the row layout's version)
static uint64_t config_tag(const ssd_handle* h)
{
    const ssd_config& c = h->cfg;
    uint64_t t = 14695981039346656037ull;
    const uint32_t version = CK_LAYOUT_VERSION;
    const int32_t ints[7] = { c.abi_version, c.env_kind, c.num_agents, c.map_h, c.map_w, c.horizon, c.contract_kind };
    t = fnv1a(t, &version, sizeof(version));
    t = fnv1a(t, ints, sizeof(ints));
    t = fnv1a(t, h->ascii.data(), h->ascii.size());
    const double dbl[3] = { c.theta_low, c.theta_high, c.null_prob };
    t = fnv1a(t, dbl, sizeof(dbl));
    t = fnv1a(t, &c.flags, sizeof(c.flags));
    t = fnv1a(t, c.env_params, sizeof(c.env_params));
    return t;
}
static void ck_col(CkParams& k, void* base, int elem, int row_off)
{
    k.col[k.ncol].base = (uint8_t*)base; k.col[k.ncol].elem = elem; k.col[k.ncol].row_off = row_off; k.ncol++;
}
static void setup_checkpoint(ssd_handle* h)
{
    CkParams& k = h->ck;
    memset(&k, 0, sizeof(k));
    const ssd_config& c = h->cfg;
    const int n = c.num_agents;
    k.E = c.num_envs; k.n = n;
    if (c.env_kind == SSD_ENV_SELFDRIVE) {                 // every array is [car][env] / [env]: columns only
        const CarParams& p = h->cp;
        k.fam = CK_CAR;
        for (int a = 0; a < n; a++) ck_col(k, p.pos + (size_t)a * p.E, 8, 8 * a);
        for (int a = 0; a < n; a++) ck_col(k, p.vel + (size_t)a * p.E, 8, 8 * (n + a));
        ck_col(k, p.theta, 8, 16 * n);
        ck_col(k, p.m_transfers, 8, 16 * n + 8);
        ck_col(k, p.dist_front, 8, 16 * n + 16);
        k.car_crossed_off = 16 * n + 24; ck_col(k, p.crossed, 4, k.car_crossed_off);
        k.car_meta_off = 16 * n + 28; ck_col(k, p.meta, 4, k.car_meta_off);
        ck_col(k, p.t, 4, 16 * n + 32);
        ck_col(k, p.episode, 4, 16 * n + 36);
        k.row_bytes = round_up(16 * n + 40, 16);
        k.zero_fill = 1;
    } else if (c.env_kind == SSD_ENV_CLEANUP_FEATURES || c.env_kind == SSD_ENV_HARVEST_FEATURES) {   // hot record + lists env-major; metrics / accumulators [k][E]
        const FeatParams& p = h->fp;
        k.fam = CK_FEAT;
        k.H = p.H; k.W = p.W; k.horizon = p.horizon; k.n_apple = p.n_apple; k.n_waste = p.n_waste; k.LA = p.LA; k.LW = p.LW;
        k.lists_off = round_up(192 + 28 * n, 16);
        k.nseg = 2;
        k.seg[0].base = (uint8_t*)p.rec; k.seg[0].stride = 4 * FR_WORDS; k.seg[0].bytes = 4 * FR_WORDS; k.seg[0].row_off = 0;
        k.seg[1].base = p.lists; k.seg[1].stride = p.LS; k.seg[1].bytes = p.LS; k.seg[1].row_off = k.lists_off;
        for (int q = 0; q < 8; q++) ck_col(k, p.metrics + (size_t)q * p.E, 8, 128 + 8 * q);
        for (int a = 0; a < n; a++) ck_col(k, p.tsum_raw + (size_t)a * p.E, 8, 192 + 8 * a);
        for (int a = 0; a < n; a++) ck_col(k, p.sum_tr + (size_t)a * p.E, 8, 192 + 8 * (n + a));
        for (int a = 0; a < n; a++) ck_col(k, p.tsum_tr + (size_t)a * p.E, 8, 192 + 8 * (2 * n + a));
        for (int a = 0; a < n; a++) ck_col(k, p.sum_raw + (size_t)a * p.E, 4, 192 + 24 * n + 4 * a);
        k.row_bytes = k.lists_off + p.LS;
        k.zero_fill = 1;
    } else {                                               // the whole record, padding included
        const GridParams& p = h->gp;
        k.fam = CK_GRID;
        k.H = p.H; k.W = p.W; k.horizon = p.horizon; k.n_apple = p.n_apple; k.n_waste = p.n_waste;
        k.nseg = 1;
        k.seg[0].base = p.state; k.seg[0].stride = p.rec_stride; k.seg[0].bytes = p.rec_stride; k.seg[0].row_off = 0;
        k.row_bytes = p.rec_stride;
    }
    h->config_tag = config_tag(h);
}

// ---------------------------------------------------------------------------------------------
// small utility kernels
__global__ void get_state_kernel(GridParams p, uint8_t* map, int32_t* pos, int32_t* ori, int32_t* t, double* theta)
{
    int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.E) return;
    const uint8_t* hdr = p.state + (size_t)env * p.rec_stride;
    const char chars[16] = { ' ', '@', 'A', 'H', 'R', 'S', '?', '?', '?', '?', '?', '?', '?', '?', '?', '?' };
    if (map) {                                             // the static map, then the dynamic cells from the masks
        uint8_t* m = map + (size_t)env * p.H * p.W;
        for (int r = 0; r < p.H; r++)
            for (int c = 0; c < p.W; c++) m[r * p.W + c] = (uint8_t)chars[(p.base_map[r * p.Wp + c] >> 2) & 15];
        const uint32_t* am = reinterpret_cast<const uint32_t*>(hdr + RO_AMASK);
        const uint32_t* wm = reinterpret_cast<const uint32_t*>(hdr + RO_WMASK);
        for (int j = 0; j < p.n_apple; j++)
            if ((am[j >> 5] >> (j & 31)) & 1u) { const int o = p.apple_c[j]; m[(o / p.Wp) * p.W + o % p.Wp] = 'A'; }
        for (int j = 0; j < p.n_waste; j++)
            if ((wm[j >> 5] >> (j & 31)) & 1u) { const int o = p.waste_c[j]; m[(o / p.Wp) * p.W + o % p.Wp] = 'H'; }
    }
    for (int a = 0; a < p.n; a++) {
        uint32_t v = reinterpret_cast<const uint32_t*>(hdr + RO_AGENTS)[a];
        if (pos) { pos[((size_t)env * p.n + a) * 2] = (int)(v & 255u); pos[((size_t)env * p.n + a) * 2 + 1] = (int)((v >> 8) & 255u); }
        if (ori) ori[(size_t)env * p.n + a] = (int)((v >> 16) & 3u);
    }
    if (t) t[env] = *reinterpret_cast<const int*>(hdr + RO_T);
    if (theta) theta[env] = *reinterpret_cast<const double*>(hdr + RO_THETA);
}

__global__ void set_state_kernel(GridParams p, const uint8_t* map, const int32_t* pos, const int32_t* ori,
                                 const int32_t* t, const double* theta)
{
    int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.E) return;
    uint8_t* hdr = p.state + (size_t)env * p.rec_stride;
    uint32_t bad = 0;
    if (map) {
        // a map can differ from the static one only by apples on apple points and waste on waste points
        const uint8_t* m = map + (size_t)env * p.H * p.W;
        const char chars[16] = { ' ', '@', 'A', 'H', 'R', 'S', '?', '?', '?', '?', '?', '?', '?', '?', '?', '?' };
        uint32_t am[MAX_POINT_ROUNDS] = {}, wm[MAX_POINT_ROUNDS] = {};
        int hc = 0;
        for (int r = 0; r < p.H; r++)
            for (int c = 0; c < p.W; c++) {
                const uint8_t ch = m[r * p.W + c];
                const uint32_t info = p.cell_info[r * p.Wp + c];
                const uint8_t stat = (uint8_t)chars[(p.base_map[r * p.Wp + c] >> 2) & 15];
                if ((info & CI_APPLE) && ch == 'A') am[(info & CI_IDX) >> 5] |= 1u << (info & 31u);
                else if ((info & CI_WASTE) && ch == 'H') { wm[(info & CI_IDX) >> 5] |= 1u << (info & 31u); hc++; }
                else if (ch != stat) bad |= 16;
            }
        for (int q = 0; q < MAX_POINT_ROUNDS; q++) {
            reinterpret_cast<uint32_t*>(hdr + RO_AMASK)[q] = am[q];
            reinterpret_cast<uint32_t*>(hdr + RO_WMASK)[q] = wm[q];
        }
        *reinterpret_cast<int*>(hdr + RO_HCOUNT) = hc;
    }
    for (int a = 0; a < p.n; a++) {
        uint32_t v = reinterpret_cast<uint32_t*>(hdr + RO_AGENTS)[a];
        if (pos) v = (v & ~0xFFFFu) | (uint32_t)(pos[((size_t)env * p.n + a) * 2] & 255) | ((uint32_t)(pos[((size_t)env * p.n + a) * 2 + 1] & 255) << 8);
        if (ori) v = (v & ~0xFF0000u) | ((uint32_t)(ori[(size_t)env * p.n + a] & 3) << 16);
        reinterpret_cast<uint32_t*>(hdr + RO_AGENTS)[a] = v;
    }
    if (t) *reinterpret_cast<int*>(hdr + RO_T) = t[env];
    if (theta) *reinterpret_cast<double*>(hdr + RO_THETA) = theta[env];
    uint32_t f = *reinterpret_cast<uint32_t*>(hdr + RO_FLAGS);
    // like oracle/ref_harness.RefGridEnv.set_state: the stale apple list is rebuilt from the map
    *reinterpret_cast<uint32_t*>(hdr + RO_FLAGS) = ((f | 0x80000000u) & ~RF_STALE_EMPTY) | (bad << RF_ERR_SHIFT);
}

// every env kind: theta where the solver reads it, then the policy output's rows that carry it
__global__ void set_theta_kernel(SolverParams p, const double* theta)
{
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.E) return;
    *reinterpret_cast<double*>(p.theta + (size_t)env * p.theta_stride) = theta[env];
    theta_rows_env(p.rows, p.n, env, theta[env]);
}

// checkpoint load with theta rows set: those of the loaded envs from their (new) theta.  Rows that failed validation kept
// their theta, so rewriting theirs changes nothing.
__global__ void theta_rows_refresh_kernel(SolverParams p, const int32_t* env_idx, int count)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= count) return;
    const int env = env_idx ? env_idx[r] : r;
    if (env < 0 || env >= p.E) return;
    theta_rows_env(p.rows, p.n, env, *reinterpret_cast<const double*>(p.theta + (size_t)env * p.theta_stride));
}

__global__ void get_metrics_kernel(GridParams p, double* out)
{
    int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.E) return;
    const uint8_t* hdr = p.state + (size_t)env * p.rec_stride;
    double* o = out + (size_t)env * SSD_METRIC_STRIDE;
    for (int q = 0; q < SSD_METRIC_STRIDE; q++) o[q] = grid_metric(p, hdr, q);
}

// SeparateContractNegotiateStage.step, agreement stage (two_stage_train.py:266-281)
__global__ void negotiate_kernel(SolverParams p, const uint8_t* mask, const double* proposals, const double* accept, uint8_t* decision)
{
    int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.E) return;
    if (mask && !mask[env]) return;
    const uint32_t episode = *reinterpret_cast<const uint32_t*>(p.episode + (size_t)env * p.episode_stride) & p.episode_mask;
    const bool dec = negotiate_agreement(p.seed, p.first_env_id + (uint32_t)env, episode, p.n, accept + (size_t)env * p.n);
    const double theta = dec ? proposals[env] : 0.0;
    *reinterpret_cast<double*>(p.theta + (size_t)env * p.theta_stride) = theta;
    if (decision) decision[env] = dec ? 1 : 0;
    theta_rows_env(p.rows, p.n, env, theta);
}

// step_index == SSD_STEP_AUTO: take the index from the handle's device counter (bumped by the last CTA to finish,
// counter_finish in ssd_common.cuh), so that a captured CUDA graph draws fresh actions at every replay
__global__ void random_actions_kernel(GridParams p, uint32_t step_index, uint32_t* counter, int num_actions, uint8_t* actions)
{
    pdl_launch_dependents();                          // a step launched behind this kernel may load its tables meanwhile
    int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (counter) step_index = *reinterpret_cast<volatile uint32_t*>(counter);
    if (env < p.E) {
        const uint32_t env_id = p.first_env_id + (uint32_t)env;
        uint32_t packed[2] = { 0u, 0u };
        for (int b = 0; b * 4 < p.n; b++) {
            Philox4 q = philox4x32_10((uint32_t)b, SITE_ACTIONS, step_index, 0u, p.seed, env_id);
            uint32_t w[4] = { q.x, q.y, q.z, q.w };
            for (int j = 0; j < 4 && b * 4 + j < p.n; j++)
                packed[b] |= (uint32_t)(((uint64_t)w[j] * (uint32_t)num_actions) >> 32) << (8 * j);
        }
        uint8_t* dst = actions + (size_t)env * p.n;
        if (p.n == 8 && (reinterpret_cast<uintptr_t>(actions) & 7u) == 0) *reinterpret_cast<uint2*>(dst) = make_uint2(packed[0], packed[1]);
        else for (int a = 0; a < p.n; a++) dst[a] = (uint8_t)(packed[a >> 2] >> (8 * (a & 3)));
    }
    if (counter) counter_finish(counter, step_index);
}

// launch `kernel` behind the previous kernel of the stream with programmatic dependent launch (see pdl_wait in ssd_grid.cuh)
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// the checks both policy-output setters make: the struct's size, its dtype and a 16-byte aligned output pointer
template <typename Out>
static int check_policy_out(ssd_handle* h, const Out* out, const char* type, const char* what, const void* ptr, const char* ptr_name)
{
    if (out->struct_size < (int32_t)sizeof(Out))
        return fail(h, SSD_EINVAL, "%s.struct_size %d < %d: the caller's declaration of %s is out of date", type, out->struct_size,
                    (int)sizeof(Out), type);
    if (out->dtype != SSD_POLICY_F32 && out->dtype != SSD_POLICY_F16 && out->dtype != SSD_POLICY_BF16)
        return fail(h, SSD_EINVAL, "%s: dtype %d is not SSD_POLICY_F32, _F16 or _BF16", what, out->dtype);
    if (!ptr || (reinterpret_cast<uintptr_t>(ptr) & 15))
        return fail(h, SSD_EINVAL, "%s: %s must be a 16-byte aligned device pointer", what, ptr_name);
    return SSD_OK;
}
// the handle's observation form and what it writes; form 0 (the native form) clears the policy output
static int set_form(ssd_handle* h, int form, void* pol_rows, ThetaRows theta_rows)
{
    if (form) { int rc = set_form_smem(h, form); if (rc) return rc; }
    h->form = form;
    h->feat_form = 0;
    h->pol_rows = pol_rows;
    h->theta_rows = theta_rows;
    return SSD_OK;
}
// elements per row of the feature output: F, + [theta, 0] for the policy dtypes under a contract
static int feature_width(const ssd_handle* h)
{
    return h->gp.F + (h->feat_form != 1 + SSD_FEATURE_F64 && h->cfg.contract_kind != SSD_CONTRACT_NONE ? 2 : 0);
}
// the feature output's reset rows of the envs `mask` selects (all when NULL), behind the reset kernel on stream s
static void launch_reset_features(ssd_handle* h, const uint8_t* mask, cudaStream_t s)
{
    reset_features_kernel_fn(h->gp.kind, h->feat_form - 1)<<<h->grid_blocks, GRID_THREADS, 0, s>>>(h->gp, mask, h->pol_rows, feature_width(h));
}

// =============================================================================================
extern "C" {

int ssd_abi_version(void) { return SSD_ABI_VERSION; }

const char* ssd_last_error(const ssd_handle* h) { return h ? h->err : g_create_error; }

void ssd_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    Philox4 q = philox4x32_10(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1]);
    out[0] = q.x; out[1] = q.y; out[2] = q.z; out[3] = q.w;
}

int ssd_create(const ssd_config* cfg, ssd_handle** out)
{
    if (!cfg || !out) return fail(nullptr, SSD_EINVAL, "null argument");
    *out = nullptr;
    if (cfg->abi_version != SSD_ABI_VERSION) return fail(nullptr, SSD_EINVAL, "abi_version %d != %d", cfg->abi_version, SSD_ABI_VERSION);
    if (cfg->struct_size != (int32_t)sizeof(ssd_config))
        return fail(nullptr, SSD_EINVAL, "ssd_config.struct_size %d != %d: the caller's declaration of ssd_config is out of date",
                    cfg->struct_size, (int)sizeof(ssd_config));
    if (cfg->num_envs < 1) return fail(nullptr, SSD_EINVAL, "num_envs must be >= 1");
    if (cfg->num_agents < 1 || cfg->num_agents > SSD_MAX_AGENTS) return fail(nullptr, SSD_EINVAL, "num_agents must be in [1, %d]", SSD_MAX_AGENTS);
    if (cfg->env_kind < SSD_ENV_CLEANUP || cfg->env_kind > SSD_ENV_SELFDRIVE)
        return fail(nullptr, SSD_EUNSUPPORTED, "env_kind %d not supported by this build", cfg->env_kind);
    if (cfg->contract_kind != SSD_CONTRACT_NONE &&
        !((cfg->env_kind == SSD_ENV_CLEANUP && cfg->contract_kind == SSD_CONTRACT_CLEANUP) ||
          (cfg->env_kind == SSD_ENV_HARVEST && cfg->contract_kind == SSD_CONTRACT_HARVEST_LOCAL) ||
          (cfg->env_kind == SSD_ENV_CLEANUP_FEATURES && cfg->contract_kind == SSD_CONTRACT_CLEANUP) ||
          (cfg->env_kind == SSD_ENV_HARVEST_FEATURES && cfg->contract_kind == SSD_CONTRACT_HARVEST_LOCAL) ||
          (cfg->env_kind == SSD_ENV_SELFDRIVE && cfg->contract_kind == SSD_CONTRACT_SELFDRIVE_DISTPROP)))
        return fail(nullptr, SSD_EINVAL, "contract_kind %d does not apply to env_kind %d", cfg->contract_kind, cfg->env_kind);
    if (cfg->contract_kind != SSD_CONTRACT_NONE && cfg->num_agents < 2 && cfg->env_kind != SSD_ENV_SELFDRIVE)
        return fail(nullptr, SSD_EINVAL, "contracts need at least 2 agents");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(nullptr, SSD_ECUDA, "no CUDA device available (this library has no CPU fallback)");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, SSD_EINVAL, "device %d out of range", cfg->device);
    ssd_handle* h = new ssd_handle();
    h->cfg = *cfg;
    ON_DEVICE(h);                                       // restores the caller's current device on return
    {
        int cur = -1;
        cudaError_t e = cudaGetDevice(&cur);
        if (e != cudaSuccess || cur != cfg->device) {
            delete h;
            return fail(nullptr, SSD_ECUDA, "cudaSetDevice(%d) failed: %s", cfg->device, cudaGetErrorString(e));
        }
    }
    h->launches = 0;
    h->timing = false;
    h->tev[0] = h->tev[1] = h->tev[2] = nullptr;
    h->err[0] = 0;
    if (cfg->ascii_map) h->ascii.assign(cfg->ascii_map, (size_t)cfg->map_h * cfg->map_w);
    h->cfg.ascii_map = h->ascii.c_str();
    const bool is_feat = cfg->env_kind == SSD_ENV_CLEANUP_FEATURES || cfg->env_kind == SSD_ENV_HARVEST_FEATURES;
    int rc = cfg->env_kind == SSD_ENV_SELFDRIVE ? setup_selfdrive(h) : (is_feat ? setup_features(h) : setup_grid(h));
    if (rc == SSD_OK) rc = dev_zalloc(h, 2, &h->d_counter);
    if (rc == SSD_OK) setup_checkpoint(h);
    if (rc != SSD_OK) {
        snprintf(g_create_error, sizeof(g_create_error), "%s", h->err);
        ssd_destroy(h);
        return rc;
    }
    *out = h;
    return SSD_OK;
}

void ssd_destroy(ssd_handle* h)
{
    if (!h) return;
    {
        ON_DEVICE(h);
        if (h->s_out) {                                 // let in-flight copies of the async host path finish
            cudaStreamSynchronize(h->s_in); cudaStreamSynchronize(h->s_out);
            for (int i = 0; i < 2; i++) {
                cudaEventDestroy(h->slot[i].ev_up); cudaEventDestroy(h->slot[i].ev_rew);
                cudaEventDestroy(h->slot[i].ev_copied); cudaEventDestroy(h->slot[i].ev_logic);
            }
            cudaStreamDestroy(h->s_in); cudaStreamDestroy(h->s_out);
        }
        for (void* d : h->dev_allocs) cudaFree(d);
        for (int i = 0; i < 3; i++) if (h->tev[i]) cudaEventDestroy(h->tev[i]);
        if (h->side) { cudaStreamDestroy(h->side); cudaEventDestroy(h->ev_rew); cudaEventDestroy(h->ev_copied); }
    }
    delete h;
}

static int check_launch(ssd_handle* h, const char* what)
{
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(h, SSD_ECUDA, "%s launch: %s", what, cudaGetErrorString(e));
    h->launches++;
    return SSD_OK;
}

#define REQUIRE_GRID(h) \
    if ((h)->cfg.env_kind != SSD_ENV_CLEANUP && (h)->cfg.env_kind != SSD_ENV_HARVEST) \
        return fail(h, SSD_EINVAL, "%s: handle is not a gridworld (env_kind %d)", __func__, (h)->cfg.env_kind)
#define IS_FEAT(h) ((h)->cfg.env_kind == SSD_ENV_CLEANUP_FEATURES || (h)->cfg.env_kind == SSD_ENV_HARVEST_FEATURES)
#define REQUIRE_FEAT(h) \
    if (!IS_FEAT(h)) return fail(h, SSD_EINVAL, "%s: handle is not a feature env (env_kind %d)", __func__, (h)->cfg.env_kind)
#define REQUIRE_CAR(h) \
    if ((h)->cfg.env_kind != SSD_ENV_SELFDRIVE) return fail(h, SSD_EINVAL, "%s: handle is not a selfdrive env", __func__)

// the rows a feature-env / selfdrive step or reset writes: obs_dev, or the flat policy rows while they are set (obs_dev
// must then be NULL: one observation form per handle)
static int flat_obs_target(ssd_handle* h, const char* what, void* obs_dev, bool required, void** out)
{
    if (h->form) {
        if (obs_dev) return fail(h, SSD_EINVAL, "%s: obs_dev must be NULL while flat policy rows are set (ssd_set_flat_policy_output)", what);
        *out = h->pol_rows;
    } else {
        if (required && !obs_dev) return fail(h, SSD_EINVAL, "actions_dev, obs_dev and rew_dev are required");
        *out = obs_dev;
    }
    return SSD_OK;
}

int ssd_reset(ssd_handle* h, const uint8_t* mask_dev, uint8_t* obs_dev, int64_t obs_env_stride, void* stream)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    const GridParams& p = h->gp;
    cudaStream_t s = (cudaStream_t)stream;
    if (h->feat_form) {                                  // one observation form per handle: the feature rows, no windows
        if (obs_dev) return fail(h, SSD_EINVAL, "reset: obs_dev must be NULL while a feature output is set (ssd_set_feature_output)");
        if (p.beam) beam_clear_kernel<<<(p.E + 3) / 4, 128, 0, s>>>(p, mask_dev);
        reset_kernel_fn(p.kind, OBS_U8)<<<h->grid_blocks, GRID_THREADS, p.g2_smem_bytes, s>>>(p, mask_dev, nullptr, 0, StepIO(), nullptr);
        int rc = check_launch(h, "reset");
        if (rc) return rc;
        launch_reset_features(h, mask_dev, s);
        return check_launch(h, "reset");
    }
    long long stride = obs_env_stride ? obs_env_stride : (long long)p.n * SSD_OBS_BYTES;
    if (h->form) {                                       // one observation form per handle: the policy output's
        if (obs_dev) return fail(h, SSD_EINVAL, "reset: obs_dev must be NULL while a policy output is set (ssd_set_policy_output)");
        obs_dev = (uint8_t*)h->pol_rows;
        stride = policy_env_bytes(p, h->form);
    }
    if (stride < (long long)p.n * SSD_OBS_BYTES) return fail(h, SSD_EINVAL, "obs_env_stride too small");
    if (p.beam) beam_clear_kernel<<<(p.E + 3) / 4, 128, 0, s>>>(p, mask_dev);                 // self.beam_pos = [] (map_env.py:316)
    reset_kernel_fn(p.kind, h->form)<<<h->grid_blocks, GRID_THREADS, p.g2_smem_bytes, s>>>(p, mask_dev, obs_dev, stride, StepIO(),
                                                                                            h->theta_rows.rows);
    return check_launch(h, "reset");
}

static int make_step_io(ssd_handle* h, const ssd_step_io* io, StepIO& k, bool async_host = false)
{
    memset(&k, 0, sizeof(k));
    if (!async_host && (!io->actions_dev || !io->rew_dev)) return fail(h, SSD_EINVAL, "actions_dev, obs_dev and rew_dev are required");
    const GridParams& p = h->gp;
    if (h->form) {                                       // one observation form per handle: the policy output's
        if (io->obs_dev) return fail(h, SSD_EINVAL, "obs_dev must be NULL while a policy output is set (ssd_set_policy_output)");
        k.obs = (uint8_t*)h->pol_rows;
        k.obs_stride = policy_env_bytes(p, h->form);
    } else if (h->feat_form) {                           // the feature rows are the observation: no windows, no second copy
        if (io->obs_dev || io->feature_obs_dev)
            return fail(h, SSD_EINVAL, "obs_dev and feature_obs_dev must be NULL while a feature output is set (ssd_set_feature_output)");
    } else {
        if (!io->obs_dev) return fail(h, SSD_EINVAL, "obs_dev is required");
        k.obs = io->obs_dev;
        k.obs_stride = io->obs_env_stride ? io->obs_env_stride : (long long)p.n * SSD_OBS_BYTES;
        if (k.obs_stride < (long long)p.n * SSD_OBS_BYTES) return fail(h, SSD_EINVAL, "obs_env_stride too small");
    }
    k.actions = (const uint8_t*)io->actions_dev;
    k.rew = io->rew_dev; k.base_rew = io->base_rew_dev; k.transfers = io->transfers_dev;
    k.info = io->info_dev; k.feat = io->feature_obs_dev; k.done = io->done_dev;
    if (k.info && (reinterpret_cast<uintptr_t>(k.info) & 3)) return fail(h, SSD_EINVAL, "info_dev must be 4-byte aligned");
    k.auto_reset = io->auto_reset != 0;
    if (k.auto_reset) {
        if ((io->neg_proposals_dev == nullptr) != (io->neg_accept_dev == nullptr))
            return fail(h, SSD_EINVAL, "neg_proposals_dev and neg_accept_dev go together");
        k.neg_prop = io->neg_proposals_dev; k.neg_acc = io->neg_accept_dev; k.neg_dec = io->neg_decision_dev;
        if (!k.done) return fail(h, SSD_EINVAL, "auto_reset needs done_dev");
    }
    return SSD_OK;
}

// ssd_step_host / ssd_step_host_async: the results go back to the host on a copy stream as soon as the kernels producing
// them are enqueued.  slot < 0: the synchronous form (dense float64 rewards + dones); else the slot's result block.
struct HostCopy { double* rew_host; uint8_t* done_host; int slot; };
static int copy_rewards(ssd_handle* h, const StepIO& k, cudaStream_t s, const HostCopy* hc)
{
    if (!hc) return SSD_OK;
    if (hc->slot >= 0) {
        ssd_handle::Slot& sl = h->slot[hc->slot];
        // the record prefix that travels: the recent maximum + 25 % + 1024 (the count of a large batch is a sum of many
        // independent envs: tens of standard deviations); ssd_step_host_wait fetches a remainder on a miss
        const uint32_t recent = std::max(h->recent_count[0], h->recent_count[1]);
        uint32_t want = recent + recent / 4u + 1024u;
        if (want > (uint32_t)h->lay.record_capacity) want = (uint32_t)h->lay.record_capacity;
        sl.copied_records = want;
        CUDA_TRY(h, cudaEventRecord(sl.ev_rew, s));
        CUDA_TRY(h, cudaStreamWaitEvent(h->s_out, sl.ev_rew, 0));
        CUDA_TRY(h, cudaMemcpyAsync(sl.host_block, sl.d_block, (size_t)h->lay.records_offset + (size_t)want * h->lay.record_bytes,
                                    cudaMemcpyDeviceToHost, h->s_out));
        CUDA_TRY(h, cudaMemsetAsync(sl.d_block + h->lay.count_offset, 0, 4, h->s_out));     // ready for the slot's next step
        CUDA_TRY(h, cudaEventRecord(sl.ev_copied, h->s_out));
        return SSD_OK;
    }
    const size_t na = (size_t)h->gp.E * h->gp.n;
    CUDA_TRY(h, cudaEventRecord(h->ev_rew, s));
    CUDA_TRY(h, cudaStreamWaitEvent(h->side, h->ev_rew, 0));
    CUDA_TRY(h, cudaMemcpyAsync(hc->rew_host, k.rew, na * sizeof(double), cudaMemcpyDeviceToHost, h->side));
    if (hc->done_host) CUDA_TRY(h, cudaMemcpyAsync(hc->done_host, k.done, (size_t)h->gp.E, cudaMemcpyDeviceToHost, h->side));
    CUDA_TRY(h, cudaEventRecord(h->ev_copied, h->side));
    return SSD_OK;
}

// the kernels of one step on stream s.  The rewards / dones are final after the logic kernel for cleanup — BEFORE the
// observe kernel — and after the reward kernel for harvest.
// (Measured and dropped in round 2: launching a step as 2-8 env chunks with chunk c's observe kernel on a second stream
// beside chunk c + 1's logic kernel, observe kernel capped at 72 registers so that a logic CTA fits beside three
// observe CTAs: 0.264 ms -> 0.29 / 0.34 / 0.39 ms for 2 / 4 / 8 chunks, and the 72-register observe kernel alone is
// 20 % slower; gpurun_out r2s sweep, DESIGN.md §4.1.)
static int launch_step(ssd_handle* h, const StepIO& k, cudaStream_t s, const HostCopy* hc)
{
    const GridParams& p = h->gp;
    if (p.beam) CUDA_TRY(h, cudaMemsetAsync(p.beam, 0, (size_t)p.E * p.map_bytes, s));       // self.beam_pos = [] (map_env.py:231)
    const int lb = (p.E + LOGIC_THREADS - 1) / LOGIC_THREADS;
    if (h->timing) cudaEventRecord(h->tev[0], s);
    if (h->logic8) {
        const logic_kernel_t fn8 = p.kind == SSD_ENV_CLEANUP ? grid_logic8_kernel<SSD_ENV_CLEANUP> : grid_logic8_kernel<SSD_ENV_HARVEST>;
        if (h->pdl && !h->timing && !p.beam)
            CUDA_TRY(h, launch_pdl(fn8, dim3(h->logic8_blocks), dim3(L8_THREADS), (size_t)h->logic8_smem, s, p, k, h->d_res));
        else fn8<<<h->logic8_blocks, L8_THREADS, h->logic8_smem, s>>>(p, k, h->d_res);
    } else if (h->pdl && !h->timing && !p.beam)
        CUDA_TRY(h, launch_pdl(logic_kernel_fn(p.kind, h->logic_lay), dim3(lb), dim3(LOGIC_THREADS), (size_t)h->logic_smem, s, p, k, h->d_res));
    else logic_kernel_fn(p.kind, p.beam ? 0 : h->logic_lay)<<<lb, LOGIC_THREADS, h->logic_smem, s>>>(p, k, h->d_res);
    h->launches++;
    if (h->timing) cudaEventRecord(h->tev[1], s);
    if (hc && hc->slot >= 0) CUDA_TRY(h, cudaEventRecord(h->slot[hc->slot].ev_logic, s));   // the slot's actions were read
    if (p.kind == SSD_ENV_CLEANUP) { int rc = copy_rewards(h, k, s, hc); if (rc) return rc; }
    // programmatic dependent launch: the observe CTAs become resident (tables, tiles) as the one-wave logic grid drains
    if (h->feat_form) {          // the feature form: spawn + feature rows in place of the observe kernel
        const feature_kernel_t fk = feature_kernel_fn(p.kind, h->rounds4, h->feat_form - 1);
        const int width = feature_width(h);
        if (h->pdl && !h->timing)
            CUDA_TRY(h, launch_pdl(fk, dim3(h->obs_blocks), dim3(OBS_WARPS * 32), (size_t)p.g2_smem_bytes, s, p, h->d_res, h->pol_rows, width));
        else fk<<<h->obs_blocks, OBS_WARPS * 32, p.g2_smem_bytes, s>>>(p, h->d_res, h->pol_rows, width);
    } else {
        const bool dense = h->form || k.obs_stride == (long long)p.n * SSD_OBS_BYTES;       // a policy image is always dense
        const int lay = (h->obs_lay != 0 && dense && !k.feat) ? h->obs_lay : 0;
        const obs_kernel_t obs_k = obs_kernel_fn(p.kind, h->rounds4, k.feat != nullptr, lay, h->form);
        if (h->pdl && !h->timing) CUDA_TRY(h, launch_pdl(obs_k, dim3(h->obs_blocks), dim3(OBS_WARPS * 32), (size_t)p.g2_smem_bytes, s, p, k, h->d_res));
        else obs_k<<<h->obs_blocks, OBS_WARPS * 32, p.g2_smem_bytes, s>>>(p, k, h->d_res);
    }
    if (p.kind == SSD_ENV_HARVEST) {
        h->launches++;
        if (h->pdl && !h->timing) CUDA_TRY(h, launch_pdl(grid_reward_kernel, dim3(lb), dim3(LOGIC_THREADS), (size_t)0, s, p, k, (const uint32_t*)h->d_res));
        else grid_reward_kernel<<<lb, LOGIC_THREADS, 0, s>>>(p, k, h->d_res);
        int rc = copy_rewards(h, k, s, hc); if (rc) return rc;
    }
    if (k.auto_reset) {          // the envs that finished restart (and negotiate) behind the step: one masked launch
        h->launches++;
        // (the copy_rewards event record of the host paths sits between the harvest reward kernel and this launch: plain launch then)
        const bool pdl_ok = h->pdl && !h->timing && (p.kind == SSD_ENV_CLEANUP || !hc);
        const reset_kernel_t reset_k = reset_kernel_fn(p.kind, h->form);
        if (pdl_ok)
            CUDA_TRY(h, launch_pdl(reset_k, dim3(h->grid_blocks), dim3(GRID_THREADS), (size_t)p.g2_smem_bytes, s,
                                   p, (const uint8_t*)k.done, k.obs, k.obs_stride, k, h->theta_rows.rows));
        else reset_k<<<h->grid_blocks, GRID_THREADS, p.g2_smem_bytes, s>>>(p, k.done, k.obs, k.obs_stride, k, h->theta_rows.rows);
        if (h->feat_form) {      // (k.obs is NULL: the reset kernel wrote no windows) the new episodes' reset rows
            h->launches++;
            launch_reset_features(h, k.done, s);
        }
    }
    if (h->timing) cudaEventRecord(h->tev[2], s);
    return check_launch(h, "step");
}

int ssd_step(ssd_handle* h, const ssd_step_io* io, void* stream)
{
    if (!h || !io) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    StepIO k;
    int rc = make_step_io(h, io, k);
    if (rc) return rc;
    return launch_step(h, k, (cudaStream_t)stream, nullptr);
}

// One step with HOST buffers (what a CPU-side rollout worker holds): actions_host -> device, the step, rewards / dones ->
// host; returns when the host outputs are valid.  The device -> host copy runs on a library-owned side stream as soon as
// the rewards exist, so for cleanup it overlaps the observe kernel (observations stay in the device batch tensor).
int ssd_step_host(ssd_handle* h, const ssd_step_io* io, const void* actions_host, double* rew_host, uint8_t* done_host, void* stream)
{
    if (!h || !io || !actions_host || !rew_host) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    StepIO k;
    int rc = make_step_io(h, io, k);
    if (rc) return rc;
    if (done_host && !k.done) return fail(h, SSD_EINVAL, "step_host: done_host needs io->done_dev");
    const GridParams& p = h->gp;
    cudaStream_t s = (cudaStream_t)stream;
    if (!h->side) {
        CUDA_TRY(h, cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
        CUDA_TRY(h, cudaEventCreateWithFlags(&h->ev_rew, cudaEventDisableTiming));
        CUDA_TRY(h, cudaEventCreateWithFlags(&h->ev_copied, cudaEventDisableTiming));
    }
    const size_t na = (size_t)p.E * p.n;
    CUDA_TRY(h, cudaMemcpyAsync(const_cast<uint8_t*>(k.actions), actions_host, na, cudaMemcpyHostToDevice, s));
    const HostCopy hc = { rew_host, done_host, -1 };
    rc = launch_step(h, k, s, &hc);
    if (rc) return rc;
    CUDA_TRY(h, cudaStreamSynchronize(s));
    CUDA_TRY(h, cudaEventSynchronize(h->ev_copied));
    return SSD_OK;
}

// ---- pipelined host-buffer step (see include/ssd_b200.h) --------------------------------------------------------
// bytes of one env's actions / done flags on the host paths: uint8 [n] / 1 (gridworlds, feature envs), float32 [n] / n + 1 (selfdrive)
static int64_t host_action_bytes(const ssd_handle* h) { return (int64_t)h->cfg.num_agents * (h->cfg.env_kind == SSD_ENV_SELFDRIVE ? 4 : 1); }
static int64_t host_done_bytes(const ssd_handle* h) { return h->cfg.env_kind == SSD_ENV_SELFDRIVE ? h->cfg.num_agents + 1 : 1; }
static void host_layout(const ssd_handle* h, ssd_host_layout* l)
{
    const int64_t E = h->cfg.num_envs, n = h->cfg.num_agents;
    l->count_offset = 0;
    l->done_offset = 64;
    l->rew_i8_offset = l->done_offset + (E * host_done_bytes(h) + 63) / 64 * 64;
    l->records_offset = l->rew_i8_offset + (E * n + 63) / 64 * 64;
    l->record_bytes = (int32_t)(8 + 8 * n);
    l->record_capacity = (int32_t)E;
    l->total_bytes = l->records_offset + E * l->record_bytes;
}

int ssd_host_result_layout(const ssd_handle* h, ssd_host_layout* out)
{
    if (!h || !out) return SSD_EINVAL;
    host_layout(h, out);
    return SSD_OK;
}

static int async_setup(ssd_handle* h)
{
    if (h->s_out) return SSD_OK;
    host_layout(h, &h->lay);
    for (int i = 0; i < 2; i++) {
        int rc;
        if ((rc = dev_zalloc(h, (size_t)h->cfg.num_envs * (size_t)host_action_bytes(h), &h->slot[i].d_actions))) return rc;
        if ((rc = dev_zalloc(h, (size_t)h->lay.total_bytes, &h->slot[i].d_block))) return rc;
        CUDA_TRY(h, cudaEventCreateWithFlags(&h->slot[i].ev_up, cudaEventDisableTiming));
        CUDA_TRY(h, cudaEventCreateWithFlags(&h->slot[i].ev_rew, cudaEventDisableTiming));
        CUDA_TRY(h, cudaEventCreateWithFlags(&h->slot[i].ev_copied, cudaEventDisableTiming));
        CUDA_TRY(h, cudaEventCreateWithFlags(&h->slot[i].ev_logic, cudaEventDisableTiming));
        h->slot[i].busy = false; h->slot[i].ticket = -1;
    }
    CUDA_TRY(h, cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
    CUDA_TRY(h, cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
    h->next_ticket = 0;
    h->recent_count[0] = h->recent_count[1] = 0;
    return SSD_OK;
}

int ssd_step_host_async(ssd_handle* h, const ssd_step_io* io, const void* actions_host, void* result_host, int64_t* ticket_out,
                        void* stream)
{
    if (!h || !io || !actions_host || !result_host || !ticket_out) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    int rc = async_setup(h);
    if (rc) return rc;
    const int si = (int)(h->next_ticket & 1);
    ssd_handle::Slot& sl = h->slot[si];
    if (sl.busy) return fail(h, SSD_EINVAL, "step_host_async: ticket %lld of this slot has not been waited for", (long long)sl.ticket);
    StepIO k;
    rc = make_step_io(h, io, k, true);
    if (rc) return rc;
    const GridParams& p = h->gp;
    cudaStream_t s = (cudaStream_t)stream;
    // copy-in stream: the slot's action buffer is free once the logic kernel of its previous step has run
    if (sl.ticket >= 0) CUDA_TRY(h, cudaStreamWaitEvent(h->s_in, sl.ev_logic, 0));
    CUDA_TRY(h, cudaMemcpyAsync(sl.d_actions, actions_host, (size_t)p.E * p.n, cudaMemcpyHostToDevice, h->s_in));
    CUDA_TRY(h, cudaEventRecord(sl.ev_up, h->s_in));
    CUDA_TRY(h, cudaStreamWaitEvent(s, sl.ev_up, 0));
    // the slot's result block was copied out (and its record count cleared) before the slot could be resubmitted, but
    // the copy-out stream is not ordered with `s`: make it so
    if (sl.ticket >= 0) CUDA_TRY(h, cudaStreamWaitEvent(s, sl.ev_copied, 0));
    k.actions = sl.d_actions;
    k.c_count = reinterpret_cast<uint32_t*>(sl.d_block + h->lay.count_offset);
    k.c_done = sl.d_block + h->lay.done_offset;
    k.c_rew8 = reinterpret_cast<int8_t*>(sl.d_block + h->lay.rew_i8_offset);
    k.c_rec = sl.d_block + h->lay.records_offset;
    sl.host_block = result_host;
    const HostCopy hc = { nullptr, nullptr, si };
    rc = launch_step(h, k, s, &hc);
    if (rc) return rc;
    sl.ticket = h->next_ticket++;
    sl.busy = true;
    *ticket_out = sl.ticket;
    return SSD_OK;
}

// Front / back halves of the feature-env and selfdrive submissions (one kernel per step): upload the actions into the
// slot on the copy-in stream, order `s` behind the upload and behind the slot's previous copy-out; afterwards mark the
// actions as read, send the result block down on the copy-out stream and hand out the ticket.
static int async_begin(ssd_handle* h, const void* actions_host, void* result_host, cudaStream_t s, int* slot_out)
{
    int rc = async_setup(h);
    if (rc) return rc;
    const int si = (int)(h->next_ticket & 1);
    ssd_handle::Slot& sl = h->slot[si];
    if (sl.busy) return fail(h, SSD_EINVAL, "step_host_async: ticket %lld of this slot has not been waited for", (long long)sl.ticket);
    if (sl.ticket >= 0) CUDA_TRY(h, cudaStreamWaitEvent(h->s_in, sl.ev_logic, 0));
    CUDA_TRY(h, cudaMemcpyAsync(sl.d_actions, actions_host, (size_t)h->cfg.num_envs * (size_t)host_action_bytes(h), cudaMemcpyHostToDevice, h->s_in));
    CUDA_TRY(h, cudaEventRecord(sl.ev_up, h->s_in));
    CUDA_TRY(h, cudaStreamWaitEvent(s, sl.ev_up, 0));
    if (sl.ticket >= 0) CUDA_TRY(h, cudaStreamWaitEvent(s, sl.ev_copied, 0));
    sl.host_block = result_host;
    *slot_out = si;
    return SSD_OK;
}
static int async_end(ssd_handle* h, int si, cudaStream_t s, int64_t* ticket_out)
{
    ssd_handle::Slot& sl = h->slot[si];
    CUDA_TRY(h, cudaEventRecord(sl.ev_logic, s));                       // the slot's actions were read
    const HostCopy hc = { nullptr, nullptr, si };
    const StepIO unused = {};
    int rc = copy_rewards(h, unused, s, &hc);
    if (rc) return rc;
    sl.ticket = h->next_ticket++;
    sl.busy = true;
    *ticket_out = sl.ticket;
    return SSD_OK;
}

int ssd_step_host_wait(ssd_handle* h, int64_t ticket)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    if (!h->s_out || ticket < 0) return fail(h, SSD_EINVAL, "step_host_wait: unknown ticket %lld", (long long)ticket);
    ssd_handle::Slot& sl = h->slot[ticket & 1];
    if (!sl.busy || sl.ticket != ticket) return fail(h, SSD_EINVAL, "step_host_wait: ticket %lld is not in flight", (long long)ticket);
    CUDA_TRY(h, cudaEventSynchronize(sl.ev_copied));
    const uint32_t count = *reinterpret_cast<const volatile uint32_t*>((const uint8_t*)sl.host_block + h->lay.count_offset);
    if (count > (uint32_t)h->lay.record_capacity) return fail(h, SSD_ECUDA, "step_host_wait: corrupt record count %u", count);
    if (count > sl.copied_records) {                      // the predicted prefix was too short: fetch the rest (rare)
        const size_t off = (size_t)h->lay.records_offset + (size_t)sl.copied_records * h->lay.record_bytes;
        CUDA_TRY(h, cudaMemcpyAsync((uint8_t*)sl.host_block + off, sl.d_block + off,
                                    (size_t)(count - sl.copied_records) * h->lay.record_bytes, cudaMemcpyDeviceToHost, h->s_out));
        CUDA_TRY(h, cudaStreamSynchronize(h->s_out));
    }
    h->recent_count[ticket & 1] = count;
    sl.busy = false;
    return SSD_OK;
}

int ssd_host_result_expand(const ssd_handle* h, const void* result_host, double* rew_out)
{
    if (!h || !result_host || !rew_out) return SSD_EINVAL;
    ssd_host_layout l;
    host_layout(h, &l);
    const uint8_t* b = (const uint8_t*)result_host;
    const int64_t E = h->cfg.num_envs, n = h->cfg.num_agents;
    const int8_t* r8 = reinterpret_cast<const int8_t*>(b + l.rew_i8_offset);
    for (int64_t i = 0; i < E * n; i++) rew_out[i] = (double)r8[i];
    const uint32_t count = *reinterpret_cast<const uint32_t*>(b + l.count_offset);
    if (count > (uint32_t)l.record_capacity) return SSD_EINVAL;
    for (uint32_t r = 0; r < count; r++) {
        const uint8_t* rec = b + l.records_offset + (size_t)r * l.record_bytes;
        const int32_t env = *reinterpret_cast<const int32_t*>(rec);
        if (env < 0 || env >= E) return SSD_EINVAL;
        memcpy(rew_out + (size_t)env * n, rec + 8, (size_t)n * sizeof(double));
    }
    return SSD_OK;
}

int ssd_set_episode_stats(ssd_handle* h, double* stats_dev)
{
    if (!h) return SSD_EINVAL;
    REQUIRE_GRID(h);
    h->gp.stats = stats_dev;
    return SSD_OK;
}

static_assert(sizeof(ssd_episode_record) == EPREC_VECS * 16, "ssd_episode_record is written as EPREC_VECS 16-byte vectors");
int ssd_set_episode_log(ssd_handle* h, const ssd_episode_log* log)
{
    if (!h) return SSD_EINVAL;
    EpisodeLog el = { nullptr, nullptr, 0ull };
    if (log) {
        if (log->struct_size < (int32_t)sizeof(ssd_episode_log))
            return fail(h, SSD_EINVAL, "ssd_episode_log.struct_size %d < %d: the caller's declaration of ssd_episode_log is out of date",
                        log->struct_size, (int)sizeof(ssd_episode_log));
        if (log->capacity < 1) return fail(h, SSD_EINVAL, "set_episode_log: capacity %d < 1", log->capacity);
        if (!log->records_dev || (reinterpret_cast<uintptr_t>(log->records_dev) & 15))
            return fail(h, SSD_EINVAL, "set_episode_log: records_dev must be a 16-byte aligned device pointer");
        if (!log->count_dev || (reinterpret_cast<uintptr_t>(log->count_dev) & 7))
            return fail(h, SSD_EINVAL, "set_episode_log: count_dev must be an 8-byte aligned device pointer");
        el.records = reinterpret_cast<uint4*>(log->records_dev);
        el.count = log->count_dev;
        el.capacity = (unsigned long long)log->capacity;
    }
    h->gp.elog = el; h->fp.elog = el; h->cp.elog = el;     // (only the params of the handle's kind are ever launched)
    return SSD_OK;
}

#define SMALL_LAUNCH(kernel, ...)                                                         \
    kernel<<<(h->gp.E + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->gp, __VA_ARGS__)

static SolverParams solver_params(ssd_handle* h);
int ssd_set_contract_params(ssd_handle* h, const double* theta_dev, void* stream)
{
    if (!h || !theta_dev) return SSD_EINVAL;
    ON_DEVICE(h);
    const SolverParams sp = solver_params(h);
    set_theta_kernel<<<(sp.E + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sp, theta_dev);
    return check_launch(h, "set_contract_params");
}

int ssd_negotiate(ssd_handle* h, const uint8_t* mask_dev, const double* proposals_dev, const double* accept_dev, uint8_t* decision_dev,
                  void* stream)
{
    if (!h || !proposals_dev || !accept_dev) return SSD_EINVAL;
    ON_DEVICE(h);
    const SolverParams sp = solver_params(h);            // every env kind: episode / theta addressed by (pointer, stride)
    negotiate_kernel<<<(sp.E + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sp, mask_dev, proposals_dev, accept_dev, decision_dev);
    return check_launch(h, "negotiate");
}

// ---- JointEnv output layouts (two_stage_train.py:476-617) ----------------------------------------
int ssd_global_view(ssd_handle* h, uint8_t* out_dev, void* stream)
{
    if (!h || !out_dev) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    if (reinterpret_cast<uintptr_t>(out_dev) & 3) return fail(h, SSD_EINVAL, "out_dev must be 4-byte aligned");
    const GridParams& p = h->gp;
    global_view_kernel<<<(p.E + VIEW_GROUP - 1) / VIEW_GROUP, VIEW_THREADS, VIEW_GROUP * (p.map_bytes + round_up(p.H * p.W * 3, 4)), (cudaStream_t)stream>>>(p, out_dev, 0);
    return check_launch(h, "global_view");
}

// ---- render path (map_env.py:389-392,460-475) --------------------------------------------------------
int ssd_record_beams(ssd_handle* h, int32_t enable)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    GridParams& p = h->gp;
    if (!enable) { p.beam = nullptr; return SSD_OK; }
    if (!h->d_beam) {
        int rc = dev_zalloc(h, (size_t)p.E * p.map_bytes, &h->d_beam);
        if (rc) return rc;
    }
    p.beam = h->d_beam;
    return SSD_OK;
}

int ssd_render(ssd_handle* h, uint8_t* out_dev, void* stream)
{
    if (!h || !out_dev) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    if (reinterpret_cast<uintptr_t>(out_dev) & 3) return fail(h, SSD_EINVAL, "out_dev must be 4-byte aligned");
    const GridParams& p = h->gp;
    global_view_kernel<<<(p.E + VIEW_GROUP - 1) / VIEW_GROUP, VIEW_THREADS, VIEW_GROUP * (p.map_bytes + round_up(p.H * p.W * 3, 4)), (cudaStream_t)stream>>>(p, out_dev, 1);
    return check_launch(h, "render");
}

int ssd_concat_obs(ssd_handle* h, const uint8_t* obs_dev, int64_t obs_env_stride, uint8_t* out_dev, void* stream)
{
    if (!h || !obs_dev || !out_dev) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    const GridParams& p = h->gp;
    const int64_t dense = (int64_t)p.n * SSD_OBS_BYTES;
    if (obs_env_stride == 0) obs_env_stride = dense;
    if (obs_env_stride < dense) return fail(h, SSD_EINVAL, "obs_env_stride %lld < %lld", (long long)obs_env_stride, (long long)dense);
    if ((reinterpret_cast<uintptr_t>(out_dev) | reinterpret_cast<uintptr_t>(obs_dev)) & 3)
        return fail(h, SSD_EINVAL, "obs_dev and out_dev must be 4-byte aligned");
    concat_obs_kernel<<<(p.E + VIEW_GROUP - 1) / VIEW_GROUP, VIEW_THREADS, 2 * VIEW_GROUP * (int)dense, (cudaStream_t)stream>>>(p, obs_dev, obs_env_stride, out_dev);
    return check_launch(h, "concat_obs");
}

// ---- policy-side consumer (environments/Networks/vision_net.py:150-181) -----------------------------------
int ssd_policy_inputs(ssd_handle* h, const uint8_t* obs_dev, int64_t obs_env_stride, int32_t dtype, void* image_dev, void* contract_dev,
                      void* stream)
{
    if (!h || !obs_dev || !image_dev) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    const GridParams& p = h->gp;
    const int64_t dense = (int64_t)p.n * SSD_OBS_BYTES;
    if (obs_env_stride == 0) obs_env_stride = dense;
    if (obs_env_stride < dense) return fail(h, SSD_EINVAL, "obs_env_stride %lld < %lld", (long long)obs_env_stride, (long long)dense);
    if (p.n * 10 > VIEW_THREADS) return fail(h, SSD_EUNSUPPORTED, "policy_inputs: too many agents");
    const dim3 grid(p.E), block(VIEW_THREADS);
    const size_t smem = (size_t)((dense + 15) / 16 * 16);
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == SSD_POLICY_F32) policy_inputs_kernel<float><<<grid, block, smem, s>>>(p, obs_dev, obs_env_stride, (float*)image_dev, (float*)contract_dev);
    else if (dtype == SSD_POLICY_F16) policy_inputs_kernel<__half><<<grid, block, smem, s>>>(p, obs_dev, obs_env_stride, (__half*)image_dev, (__half*)contract_dev);
    else if (dtype == SSD_POLICY_BF16) policy_inputs_kernel<__nv_bfloat16><<<grid, block, smem, s>>>(p, obs_dev, obs_env_stride, (__nv_bfloat16*)image_dev, (__nv_bfloat16*)contract_dev);
    else return fail(h, SSD_EINVAL, "policy_inputs: dtype must be SSD_POLICY_F32, _F16 or _BF16");
    return check_launch(h, "policy_inputs");
}

int ssd_set_policy_output(ssd_handle* h, const ssd_policy_out* out)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    if (!out) return set_form(h, 0, nullptr, ThetaRows{});
    int rc = check_policy_out(h, out, "ssd_policy_out", "set_policy_output", out->image_dev, "image_dev");
    if (rc) return rc;
    const uintptr_t esize = out->dtype == SSD_POLICY_F32 ? 4 : 2;
    if (reinterpret_cast<uintptr_t>(out->contract_dev) & (esize - 1))
        return fail(h, SSD_EINVAL, "set_policy_output: contract_dev must be aligned to its element size");
    return set_form(h, 1 + out->dtype, out->image_dev, ThetaRows{ out->contract_dev, out->dtype, 10, 0, 5 });
}

int ssd_set_feature_output(ssd_handle* h, const ssd_feature_out* out)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    if (!out) return set_form(h, 0, nullptr, ThetaRows{});
    if (out->struct_size < (int32_t)sizeof(ssd_feature_out))
        return fail(h, SSD_EINVAL, "ssd_feature_out.struct_size %d < %d: the caller's declaration of ssd_feature_out is out of date",
                    out->struct_size, (int)sizeof(ssd_feature_out));
    if (out->dtype != SSD_FEATURE_F64 && out->dtype != SSD_POLICY_F32 && out->dtype != SSD_POLICY_F16 && out->dtype != SSD_POLICY_BF16)
        return fail(h, SSD_EINVAL, "set_feature_output: dtype %d is not SSD_FEATURE_F64, SSD_POLICY_F32, _F16 or _BF16", out->dtype);
    if (!out->obs_dev || (reinterpret_cast<uintptr_t>(out->obs_dev) & 15))
        return fail(h, SSD_EINVAL, "set_feature_output: obs_dev must be a 16-byte aligned device pointer");
    CUDA_TRY(h, cudaFuncSetAttribute((const void*)feature_kernel_fn(h->cfg.env_kind, h->rounds4, out->dtype),
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, h->gp.g2_smem_bytes));
    const bool theta_col = out->dtype != SSD_FEATURE_F64 && h->cfg.contract_kind != SSD_CONTRACT_NONE;
    const int width = h->gp.F + (theta_col ? 2 : 0);
    int rc = set_form(h, 0, out->obs_dev, ThetaRows{ theta_col ? out->obs_dev : nullptr, out->dtype, width, width - 2, 1 });
    if (rc) return rc;
    h->feat_form = 1 + out->dtype;
    return SSD_OK;
}

int ssd_set_flat_policy_output(ssd_handle* h, const ssd_flat_policy_out* out)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    if (h->cfg.env_kind != SSD_ENV_SELFDRIVE && !IS_FEAT(h))
        return fail(h, SSD_EINVAL, "set_flat_policy_output: handle is a gridworld (env_kind %d; see ssd_set_policy_output)", h->cfg.env_kind);
    if (!out) return set_form(h, 0, nullptr, ThetaRows{});
    int rc = check_policy_out(h, out, "ssd_flat_policy_out", "set_flat_policy_output", out->obs_dev, "obs_dev");
    if (rc) return rc;
    const bool contract = h->cfg.contract_kind != SSD_CONTRACT_NONE;       // the rows end in [theta, 0] only under a contract
    const int width = ssd_feature_dim(h) + (contract ? 2 : 0);
    return set_form(h, 1 + out->dtype, out->obs_dev, ThetaRows{ contract ? out->obs_dev : nullptr, out->dtype, width, width - 2, 1 });
}

// ---- NegotiationSolver (two_stage_train.py:619-776) ------------------------------------------------
static SolverParams solver_params(ssd_handle* h)
{
    SolverParams s;
    memset(&s, 0, sizeof(s));
    s.seed = h->cfg.seed; s.first_env_id = h->cfg.first_env_id;
    s.low = h->cfg.theta_low; s.high = h->cfg.theta_high;
    s.E = h->cfg.num_envs; s.n = h->cfg.num_agents;
    s.rows = h->theta_rows;
    if (h->cfg.env_kind == SSD_ENV_SELFDRIVE) {
        s.episode = reinterpret_cast<const uint8_t*>(h->cp.episode); s.episode_stride = 4; s.episode_mask = 0xFFFFFFFFu;
        s.theta = reinterpret_cast<uint8_t*>(h->cp.theta); s.theta_stride = 8;
    } else if (IS_FEAT(h)) {
        s.episode = reinterpret_cast<const uint8_t*>(h->fp.rec + FR_EPISODE); s.episode_stride = 4 * FR_WORDS; s.episode_mask = 0x7FFFFFFFu;
        s.theta = reinterpret_cast<uint8_t*>(h->fp.rec + FR_THETA); s.theta_stride = 4 * FR_WORDS;
    } else {
        const GridParams& p = h->gp;
        s.episode = p.state + RO_EPISODE; s.episode_stride = p.rec_stride; s.episode_mask = 0xFFFFFFFFu;
        s.theta = p.state + RO_THETA; s.theta_stride = p.rec_stride;
    }
    return s;
}

int ssd_solver_sample(ssd_handle* h, int32_t num_samples, double* params_dev, void* stream)
{
    if (!h || !params_dev || num_samples < 0) return SSD_EINVAL;
    ON_DEVICE(h);
    if (h->cfg.contract_kind == SSD_CONTRACT_NONE) return fail(h, SSD_EINVAL, "solver_sample: the handle has no contract");
    const SolverParams s = solver_params(h);
    const long long total = (long long)s.E * (num_samples + 1);
    if (total > 0x7FFFFFFFll) return fail(h, SSD_EINVAL, "solver_sample: E * (1 + num_samples) too large");
    solver_sample_kernel<<<(unsigned)((total + 127) / 128), 128, 0, (cudaStream_t)stream>>>(s, num_samples, params_dev);
    return check_launch(h, "solver_sample");
}

int ssd_solver_choose(ssd_handle* h, int32_t num_samples, int32_t rule, const double* params_dev, const double* vals_dev,
                      double* best_param_dev, int32_t* best_index_dev, void* stream)
{
    if (!h || !params_dev || !vals_dev || num_samples < 0) return SSD_EINVAL;
    ON_DEVICE(h);
    if (rule != SOLVER_RULE_MAX && rule != SOLVER_RULE_MAJORITY) return fail(h, SSD_EINVAL, "solver_choose: unknown decision rule %d", rule);
    if (h->cfg.contract_kind == SSD_CONTRACT_NONE) return fail(h, SSD_EINVAL, "solver_choose: the handle has no contract");
    const SolverParams s = solver_params(h);
    solver_choose_kernel<<<(s.E + 127) / 128, 128, 0, (cudaStream_t)stream>>>(s, num_samples, rule, params_dev, vals_dev, best_param_dev, best_index_dev);
    return check_launch(h, "solver_choose");
}

// ---- the solver queue of a vectorised sampler (ssd_solver.cuh) ----------------------------------------
// the handle's part of a SolverQueue: where the pending test reads each env, the resolved episodes, the scan's scratch
static SolverQueue solver_queue_params(ssd_handle* h)
{
    SolverQueue q;
    memset(&q, 0, sizeof(q));
    q.s = solver_params(h);
    if (h->cfg.env_kind == SSD_ENV_SELFDRIVE) {
        q.t = reinterpret_cast<const uint8_t*>(h->cp.t); q.t_stride = 4;
        q.init = reinterpret_cast<const uint8_t*>(h->cp.meta); q.init_stride = 4;
    } else if (IS_FEAT(h)) {
        q.t = reinterpret_cast<const uint8_t*>(h->fp.rec + FR_T); q.t_stride = 4 * FR_WORDS;
        q.init = reinterpret_cast<const uint8_t*>(h->fp.rec + FR_EPISODE); q.init_stride = 4 * FR_WORDS;
    } else {
        q.t = h->gp.state + RO_T; q.t_stride = h->gp.rec_stride;
        q.init = h->gp.state + RO_FLAGS; q.init_stride = h->gp.rec_stride;
    }
    q.resolved = h->d_resolved;
    q.block_count = h->d_sq_blocks;
    return q;
}

// validates the window (before anything is launched) and fills the rest of the SolverQueue
static int solver_window(ssd_handle* h, const ssd_solver_window* w, const char* what, SolverQueue* q)
{
    if (h->cfg.contract_kind == SSD_CONTRACT_NONE) return fail(h, SSD_EINVAL, "%s: the handle has no contract", what);
    if (!h->solver_on) return fail(h, SSD_EINVAL, "%s: the solver queue is off (ssd_solver_enable)", what);
    if (!w) return fail(h, SSD_EINVAL, "%s: window is NULL", what);
    if (w->struct_size < (int32_t)sizeof(ssd_solver_window))
        return fail(h, SSD_EINVAL, "ssd_solver_window.struct_size %d < %d: the caller's declaration of ssd_solver_window is out of date",
                    w->struct_size, (int)sizeof(ssd_solver_window));
    if (w->num_samples < 0) return fail(h, SSD_EINVAL, "%s: num_samples %d < 0", what, w->num_samples);
    if (w->capacity < 1 || w->capacity > h->cfg.num_envs)
        return fail(h, SSD_EINVAL, "%s: capacity %d is not in [1, %d]", what, w->capacity, h->cfg.num_envs);
    if ((long long)w->capacity * (w->num_samples + 1) * h->cfg.num_agents > 0x7FFFFFFFll)
        return fail(h, SSD_EINVAL, "%s: capacity * (1 + num_samples) * n too large", what);
    const struct { const void* p; uintptr_t align; const char* name; } ptrs[] = {
        { w->env_dev, 4, "env_dev" }, { w->episode_dev, 4, "episode_dev" }, { w->count_dev, 4, "count_dev" },
        { w->params_dev, 8, "params_dev" } };
    for (const auto& x : ptrs)
        if (!x.p || (reinterpret_cast<uintptr_t>(x.p) & (x.align - 1)))
            return fail(h, SSD_EINVAL, "%s: %s must be a %d-byte aligned device pointer", what, x.name, (int)x.align);
    *q = solver_queue_params(h);
    q->C = w->capacity; q->S = w->num_samples;
    q->env = w->env_dev; q->episode = w->episode_dev; q->count = w->count_dev; q->params = w->params_dev;
    return SSD_OK;
}

int ssd_solver_enable(ssd_handle* h, int32_t on)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    if (h->cfg.contract_kind == SSD_CONTRACT_NONE) return fail(h, SSD_EINVAL, "solver_enable: the handle has no contract");
    if (!on) { h->solver_on = false; return SSD_OK; }
    const int E = h->cfg.num_envs;
    int rc;
    if (!h->d_resolved) {
        if ((rc = dev_zalloc(h, (size_t)E, &h->d_resolved))) return rc;
        if ((rc = dev_zalloc(h, (size_t)(E + SQ_BLOCK - 1) / SQ_BLOCK, &h->d_sq_blocks))) return rc;
    }
    CUDA_TRY(h, cudaMemset(h->d_resolved, 0xFF, (size_t)E * sizeof(uint32_t)));     // SQ_NONE
    h->solver_on = true;
    return SSD_OK;
}

int ssd_solver_rows(ssd_handle* h, const ssd_solver_window* win, const void* obs_dev, void* stream)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    SolverQueue q;
    int rc = solver_window(h, win, "solver_rows", &q);
    if (rc) return rc;
    if (!win->rows_dev || (reinterpret_cast<uintptr_t>(win->rows_dev) & 15))
        return fail(h, SSD_EINVAL, "solver_rows: rows_dev must be a 16-byte aligned device pointer");
    // the rows of the handle's observation form: layout, element type (SSD_POLICY_* or SSD_FEATURE_F64 = double), width
    const bool grid = h->cfg.env_kind == SSD_ENV_CLEANUP || h->cfg.env_kind == SSD_ENV_HARVEST;
    int layout = SQ_ROWS_FLAT, dtype, W, reps = 0, F = 0, src_width = 0;
    const void* src = nullptr;
    bool obs_required = false;
    if (grid && !h->feat_form) {                            // image forms: the contract part alone
        layout = SQ_ROWS_CONTRACT;
        if (h->form) { dtype = h->form - 1; W = 10; reps = 5; }
        else { dtype = SSD_FEATURE_F64; W = 2; reps = 1; }
    } else {
        F = ssd_feature_dim(h); W = F + 2;
        if (grid) { dtype = h->feat_form - 1; src = h->pol_rows; src_width = dtype == SSD_FEATURE_F64 ? F : F + 2; }
        else if (h->form) { dtype = h->form - 1; src = h->pol_rows; src_width = F + 2; }
        else { dtype = SSD_FEATURE_F64; src = obs_dev; src_width = F; obs_required = true; }
    }
    if (obs_required && (!obs_dev || (reinterpret_cast<uintptr_t>(obs_dev) & 7)))
        return fail(h, SSD_EINVAL, "solver_rows: obs_dev must be the float64 observation double [E][n][F] (8-byte aligned): the "
                    "handle's observation is passed per call");
    if (!obs_required && obs_dev)
        return fail(h, SSD_EINVAL, "solver_rows: obs_dev must be NULL: the rows are built from the handle's own observation form");
    cudaStream_t s = (cudaStream_t)stream;
    const unsigned nb = (unsigned)((q.s.E + SQ_BLOCK - 1) / SQ_BLOCK);
    solver_count_kernel<<<nb, SQ_BLOCK, 0, s>>>(q);
    if ((rc = check_launch(h, "solver_rows"))) return rc;
    solver_scatter_kernel<<<nb, SQ_BLOCK, 0, s>>>(q);
    if ((rc = check_launch(h, "solver_rows"))) return rc;
    if (dtype == SSD_FEATURE_F64) launch_solver_rows<double>(q, layout, win->rows_dev, W, reps, src, F, src_width, s);
    else if (dtype == SSD_POLICY_F32) launch_solver_rows<float>(q, layout, win->rows_dev, W, reps, src, F, src_width, s);
    else if (dtype == SSD_POLICY_F16) launch_solver_rows<__half>(q, layout, win->rows_dev, W, reps, src, F, src_width, s);
    else launch_solver_rows<__nv_bfloat16>(q, layout, win->rows_dev, W, reps, src, F, src_width, s);
    return check_launch(h, "solver_rows");
}

int ssd_solver_resolve(ssd_handle* h, const ssd_solver_window* win, int32_t rule, const double* vals_dev, double* best_param_dev,
                       int32_t* best_index_dev, uint32_t* stale_dev, void* stream)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    if (rule != SOLVER_RULE_MAX && rule != SOLVER_RULE_MAJORITY) return fail(h, SSD_EINVAL, "solver_resolve: unknown decision rule %d", rule);
    SolverQueue q;
    int rc = solver_window(h, win, "solver_resolve", &q);
    if (rc) return rc;
    if (!vals_dev || (reinterpret_cast<uintptr_t>(vals_dev) & 7))
        return fail(h, SSD_EINVAL, "solver_resolve: vals_dev must be an 8-byte aligned device pointer");
    if ((reinterpret_cast<uintptr_t>(best_param_dev) & 7) || (reinterpret_cast<uintptr_t>(best_index_dev) & 3) ||
        (reinterpret_cast<uintptr_t>(stale_dev) & 3))
        return fail(h, SSD_EINVAL, "solver_resolve: best_param_dev, best_index_dev and stale_dev must be aligned to their elements");
    cudaStream_t s = (cudaStream_t)stream;
    if (stale_dev) CUDA_TRY(h, cudaMemsetAsync(stale_dev, 0, sizeof(uint32_t), s));
    solver_resolve_kernel<<<(q.C + 127) / 128, 128, 0, s>>>(q, rule, vals_dev, best_param_dev, best_index_dev, stale_dev);
    return check_launch(h, "solver_resolve");
}

int ssd_get_state(ssd_handle* h, uint8_t* map_dev, int32_t* pos_dev, int32_t* ori_dev, int32_t* t_dev, double* theta_dev, void* stream)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    SMALL_LAUNCH(get_state_kernel, map_dev, pos_dev, ori_dev, t_dev, theta_dev);
    return check_launch(h, "get_state");
}

int ssd_set_state(ssd_handle* h, const uint8_t* map_dev, const int32_t* pos_dev, const int32_t* ori_dev, const int32_t* t_dev,
                  const double* theta_dev, void* stream)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    SMALL_LAUNCH(set_state_kernel, map_dev, pos_dev, ori_dev, t_dev, theta_dev);
    return check_launch(h, "set_state");
}

int ssd_get_metrics(ssd_handle* h, double* out_dev, void* stream)
{
    if (!h || !out_dev) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    SMALL_LAUNCH(get_metrics_kernel, out_dev);
    return check_launch(h, "get_metrics");
}

int ssd_random_actions(ssd_handle* h, uint32_t step_index, int32_t num_actions, uint8_t* actions_dev, void* stream)
{
    if (!h || !actions_dev || num_actions < 1 || num_actions > 255) return SSD_EINVAL;
    ON_DEVICE(h);
    const bool autoidx = step_index == SSD_STEP_AUTO;
    if (IS_FEAT(h)) {
        feat_random_actions_kernel<<<(h->fp.E + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->fp, step_index, autoidx ? h->d_counter : nullptr,
                                                                                              num_actions, actions_dev);
        return check_launch(h, "random_actions");
    }
    REQUIRE_GRID(h);
    SMALL_LAUNCH(random_actions_kernel, step_index, autoidx ? h->d_counter : nullptr, num_actions, actions_dev);
    return check_launch(h, "random_actions");
}

// ---- feature envs --------------------------------------------------------------------------------------
int ssd_feat_reset(ssd_handle* h, const uint8_t* mask_dev, double* obs_dev, void* stream)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_FEAT(h);
    FeatIO k = {};
    int rc = flat_obs_target(h, "feat_reset", obs_dev, false, &k.obs);
    if (rc) return rc;
    feat_kernel_fn(h->cfg.env_kind == SSD_ENV_CLEANUP_FEATURES, true, h->form)<<<h->grid_blocks, FEAT_THREADS, h->feat_smem,
                                                                                      (cudaStream_t)stream>>>(h->fp, k, mask_dev);
    return check_launch(h, "feat_reset");
}

int ssd_feat_step(ssd_handle* h, const ssd_feat_io* io, void* stream)
{
    if (!h || !io) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_FEAT(h);
    void* obs = nullptr;
    int rc = flat_obs_target(h, "feat_step", io->obs_dev, true, &obs);
    if (rc) return rc;
    if (!io->actions_dev || !io->rew_dev) return fail(h, SSD_EINVAL, "actions_dev, obs_dev and rew_dev are required");
    if (io->info_dev && (reinterpret_cast<uintptr_t>(io->info_dev) & 3)) return fail(h, SSD_EINVAL, "info_dev must be 4-byte aligned");
    FeatIO k = { io->actions_dev, obs, io->rew_dev, io->base_rew_dev, io->transfers_dev, io->info_dev, io->done_dev, io->auto_reset };
    feat_kernel_fn(h->cfg.env_kind == SSD_ENV_CLEANUP_FEATURES, false, h->form)<<<h->grid_blocks, FEAT_THREADS, h->feat_smem,
                                                                                       (cudaStream_t)stream>>>(h->fp, k, nullptr);
    return check_launch(h, "feat_step");
}

int ssd_feat_step_host_async(ssd_handle* h, const ssd_feat_io* io, const void* actions_host, void* result_host, int64_t* ticket_out,
                             void* stream)
{
    if (!h || !io || !actions_host || !result_host || !ticket_out || (!io->obs_dev && !h->form)) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_FEAT(h);
    void* obs = nullptr;
    int rc = flat_obs_target(h, "feat_step_host_async", io->obs_dev, true, &obs);
    if (rc) return rc;
    if (io->info_dev && (reinterpret_cast<uintptr_t>(io->info_dev) & 3)) return fail(h, SSD_EINVAL, "info_dev must be 4-byte aligned");
    int si = 0;
    rc = async_begin(h, actions_host, result_host, (cudaStream_t)stream, &si);
    if (rc) return rc;
    ssd_handle::Slot& sl = h->slot[si];
    FeatIO k = { sl.d_actions, obs, io->rew_dev, io->base_rew_dev, io->transfers_dev, io->info_dev, io->done_dev, io->auto_reset };
    k.c_count = reinterpret_cast<uint32_t*>(sl.d_block + h->lay.count_offset);
    k.c_done = sl.d_block + h->lay.done_offset;
    k.c_rew8 = reinterpret_cast<int8_t*>(sl.d_block + h->lay.rew_i8_offset);
    k.c_rec = sl.d_block + h->lay.records_offset;
    feat_kernel_fn(h->cfg.env_kind == SSD_ENV_CLEANUP_FEATURES, false, h->form)<<<h->grid_blocks, FEAT_THREADS, h->feat_smem,
                                                                                       (cudaStream_t)stream>>>(h->fp, k, nullptr);
    if ((rc = check_launch(h, "feat_step_host_async"))) return rc;
    return async_end(h, si, (cudaStream_t)stream, ticket_out);
}

int ssd_feat_get_state(ssd_handle* h, int32_t* pos_dev, int32_t* ori_dev, uint8_t* cells_dev, double* theta_dev, int32_t* t_dev, void* stream)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_FEAT(h);
    feat_get_state_kernel<<<(h->fp.E + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->fp, pos_dev, ori_dev, cells_dev, theta_dev, t_dev);
    return check_launch(h, "feat_get_state");
}

int ssd_feat_get_metrics(ssd_handle* h, double* out_dev, void* stream)
{
    if (!h || !out_dev) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_FEAT(h);
    feat_get_metrics_kernel<<<(h->fp.E + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->fp, out_dev);
    return check_launch(h, "feat_get_metrics");
}

// ---- selfdrive -------------------------------------------------------------------------------------
int ssd_selfdrive_reset(ssd_handle* h, const uint8_t* mask_dev, double* obs_dev, void* stream)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_CAR(h);
    CarIO k = {};
    int rc = flat_obs_target(h, "selfdrive_reset", obs_dev, false, &k.obs);
    if (rc) return rc;
    car_kernel_fn(true, h->form)<<<h->grid_blocks, CAR_THREADS, h->car_smem, (cudaStream_t)stream>>>(h->cp, k, mask_dev);
    return check_launch(h, "selfdrive_reset");
}

int ssd_selfdrive_step(ssd_handle* h, const ssd_selfdrive_io* io, void* stream)
{
    if (!h || !io) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_CAR(h);
    void* obs = nullptr;
    int rc = flat_obs_target(h, "selfdrive_step", io->obs_dev, true, &obs);
    if (rc) return rc;
    if (!io->actions_dev || !io->rew_dev) return fail(h, SSD_EINVAL, "actions_dev, obs_dev and rew_dev are required");
    if (io->info_dev && (reinterpret_cast<uintptr_t>(io->info_dev) & 31)) return fail(h, SSD_EINVAL, "info_dev must be 32-byte aligned");
    CarIO k = { io->actions_dev, obs, io->rew_dev, io->base_rew_dev, io->transfers_dev, io->info_dev, io->done_dev, io->auto_reset };
    car_kernel_fn(false, h->form)<<<h->grid_blocks, CAR_THREADS, h->car_smem, (cudaStream_t)stream>>>(h->cp, k, nullptr);
    return check_launch(h, "selfdrive_step");
}

int ssd_selfdrive_step_host_async(ssd_handle* h, const ssd_selfdrive_io* io, const void* actions_host, void* result_host,
                                  int64_t* ticket_out, void* stream)
{
    if (!h || !io || !actions_host || !result_host || !ticket_out || (!io->obs_dev && !h->form)) return SSD_EINVAL;
    ON_DEVICE(h);
    if (h->cfg.env_kind != SSD_ENV_SELFDRIVE) return fail(h, SSD_EINVAL, "selfdrive_step_host_async: handle is not a selfdrive env");
    void* obs = nullptr;
    int rc = flat_obs_target(h, "selfdrive_step_host_async", io->obs_dev, true, &obs);
    if (rc) return rc;
    if (io->info_dev && (reinterpret_cast<uintptr_t>(io->info_dev) & 31)) return fail(h, SSD_EINVAL, "info_dev must be 32-byte aligned");
    int si = 0;
    rc = async_begin(h, actions_host, result_host, (cudaStream_t)stream, &si);
    if (rc) return rc;
    ssd_handle::Slot& sl = h->slot[si];
    CarIO k = { reinterpret_cast<const float*>(sl.d_actions), obs, io->rew_dev, io->base_rew_dev, io->transfers_dev, io->info_dev, io->done_dev,
                io->auto_reset };
    k.c_count = reinterpret_cast<uint32_t*>(sl.d_block + h->lay.count_offset);
    k.c_done = sl.d_block + h->lay.done_offset;
    k.c_rew8 = reinterpret_cast<int8_t*>(sl.d_block + h->lay.rew_i8_offset);
    k.c_rec = sl.d_block + h->lay.records_offset;
    car_kernel_fn(false, h->form)<<<h->grid_blocks, CAR_THREADS, h->car_smem, (cudaStream_t)stream>>>(h->cp, k, nullptr);
    if ((rc = check_launch(h, "selfdrive_step_host_async"))) return rc;
    return async_end(h, si, (cudaStream_t)stream, ticket_out);
}

int ssd_selfdrive_get_state(ssd_handle* h, double* pos_dev, double* vel_dev, double* theta_dev, double* transfers_dev,
                            int32_t* t_dev, void* stream)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_CAR(h);
    car_get_state_kernel<<<(h->cp.E + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->cp, pos_dev, vel_dev, theta_dev, transfers_dev, t_dev);
    return check_launch(h, "selfdrive_get_state");
}

int ssd_selfdrive_random_actions(ssd_handle* h, uint32_t step_index, float lo, float hi, float* actions_dev, void* stream)
{
    if (!h || !actions_dev) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_CAR(h);
    const bool autoidx = step_index == SSD_STEP_AUTO;
    car_random_actions_kernel<<<(h->cp.E + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->cp, step_index, autoidx ? h->d_counter : nullptr,
                                                                                         lo, hi, actions_dev);
    return check_launch(h, "selfdrive_random_actions");
}

// ---- checkpoint / restore / copy of env state (ssd_checkpoint.cuh) -------------------------------------------------
int ssd_checkpoint_get_layout(const ssd_handle* h, ssd_checkpoint_layout* out)
{
    if (!h || !out) return SSD_EINVAL;
    out->row_bytes = h->ck.row_bytes;
    out->config_tag = h->config_tag;
    return SSD_OK;
}

static int checkpoint_args(ssd_handle* h, const char* what, const int32_t* env_idx_dev, int32_t count, const void* rows_dev)
{
    if (count < 0) return fail(h, SSD_EINVAL, "%s: count %d < 0", what, count);
    if (!env_idx_dev && count > h->cfg.num_envs)
        return fail(h, SSD_EINVAL, "%s: count %d exceeds the handle's %d envs (no index list)", what, count, h->cfg.num_envs);
    if (count > 0 && !rows_dev) return fail(h, SSD_EINVAL, "%s: rows_dev is NULL", what);
    if (reinterpret_cast<uintptr_t>(rows_dev) & 15) return fail(h, SSD_EINVAL, "%s: rows_dev must be 16-byte aligned", what);
    return SSD_OK;
}

int ssd_checkpoint_save(ssd_handle* h, const int32_t* env_idx_dev, int32_t count, uint8_t* rows_dev, void* stream)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    int rc = checkpoint_args(h, "checkpoint_save", env_idx_dev, count, rows_dev);
    if (rc || count == 0) return rc;
    ck_save_kernel<<<(count + CK_ROWS - 1) / CK_ROWS, CK_THREADS, (size_t)CK_ROWS * h->ck.row_bytes, (cudaStream_t)stream>>>(
        h->ck, env_idx_dev, count, rows_dev);
    return check_launch(h, "checkpoint_save");
}

int ssd_checkpoint_load(ssd_handle* h, uint64_t config_tag, const int32_t* env_idx_dev, int32_t count, const uint8_t* rows_dev,
                        uint8_t* row_ok_dev, void* stream)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    if (config_tag != h->config_tag)
        return fail(h, SSD_EINVAL, "checkpoint_load: config_tag %016llx does not match the handle's %016llx (rows saved under "
                    "another env kind, agent count, map, horizon, contract or reward configuration)",
                    (unsigned long long)config_tag, (unsigned long long)h->config_tag);
    int rc = checkpoint_args(h, "checkpoint_load", env_idx_dev, count, rows_dev);
    if (rc || count == 0) return rc;
    uint8_t* row_ok = row_ok_dev;
    if (h->solver_on && !row_ok) {          // the solver queue needs to know which rows loaded
        if (count > h->sq_ok_cap) {
            if ((rc = dev_zalloc(h, (size_t)count, &h->d_sq_ok))) return rc;
            h->sq_ok_cap = count;
        }
        row_ok = h->d_sq_ok;
    }
    ck_load_kernel<<<(count + CK_ROWS - 1) / CK_ROWS, CK_THREADS, (size_t)CK_ROWS * h->ck.row_bytes, (cudaStream_t)stream>>>(
        h->ck, env_idx_dev, count, rows_dev, row_ok);
    if ((rc = check_launch(h, "checkpoint_load"))) return rc;
    if (h->theta_rows.rows) {
        // theta came with the rows: the policy output's rows that carry it follow
        theta_rows_refresh_kernel<<<(count + 127) / 128, 128, 0, (cudaStream_t)stream>>>(solver_params(h), env_idx_dev, count);
        if ((rc = check_launch(h, "checkpoint_load"))) return rc;
    }
    if (!h->solver_on) return SSD_OK;
    // and so did the contract of their episode: the loaded envs are not pending
    solver_mark_loaded_kernel<<<(count + 127) / 128, 128, 0, (cudaStream_t)stream>>>(solver_queue_params(h), env_idx_dev, count, row_ok);
    return check_launch(h, "checkpoint_load");
}

int ssd_enable_timing(ssd_handle* h, int32_t on)
{
    if (!h) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    if (on && !h->tev[0])
        for (int i = 0; i < 3; i++) CUDA_TRY(h, cudaEventCreate(&h->tev[i]));
    h->timing = on != 0;
    return SSD_OK;
}

int ssd_get_step_times(ssd_handle* h, double* out_ms)
{
    if (!h || !out_ms) return SSD_EINVAL;
    ON_DEVICE(h);
    REQUIRE_GRID(h);
    if (!h->tev[0]) return fail(h, SSD_EINVAL, "ssd_get_step_times: timing was never enabled");
    float a = 0.f, b = 0.f;
    CUDA_TRY(h, cudaEventSynchronize(h->tev[2]));
    CUDA_TRY(h, cudaEventElapsedTime(&a, h->tev[0], h->tev[1]));
    CUDA_TRY(h, cudaEventElapsedTime(&b, h->tev[1], h->tev[2]));
    out_ms[0] = a; out_ms[1] = b;
    return SSD_OK;
}

int ssd_feature_dim(const ssd_handle* h)
{
    if (!h) return 0;
    return h->cfg.env_kind == SSD_ENV_SELFDRIVE ? h->cp.D : (IS_FEAT(h) ? h->fp.F : h->gp.F);
}
int64_t ssd_state_bytes_per_env(const ssd_handle* h)
{
    if (!h) return 0;
    if (IS_FEAT(h)) return (int64_t)(4 * FR_WORDS + h->fp.LS + 28 * h->fp.n + 64);
    return h->cfg.env_kind == SSD_ENV_SELFDRIVE ? (int64_t)(16 * h->cp.n + 44) : (int64_t)h->gp.rec_stride;
}
int64_t ssd_kernel_launches(const ssd_handle* h) { return h ? h->launches : 0; }

}  // extern "C"
