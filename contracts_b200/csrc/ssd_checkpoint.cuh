// ssd_checkpoint.cuh — save / load the complete per-env state of a handle as env-major rows (ssd_checkpoint_save /
// ssd_checkpoint_load, include/ssd_b200.h).  Pure data movement, designed for HBM bandwidth.
//
// A row is the concatenation of
//   * env-major SEGMENTS: a contiguous run of the env's bytes in a state array (the grid record, the feature-env hot
//     record, the feature-env point lists), moved as 16-byte vectors by one warp per row;
//   * [k][E] COLUMNS: element `env` of a struct-of-arrays state array (the feature-env accumulators, every selfdrive
//     array), moved by consecutive threads for consecutive rows so that a contiguous index list gives coalesced accesses.
// A CTA takes CK_ROWS consecutive rows.  They are one contiguous run of the caller's row buffer, so the CTA stages them in
// shared memory and that side of the copy is one coalesced 16-byte-vector pass.  The load validates each staged row
// (warp per row, ck_row_valid) before anything of it is written to the handle's state.
#pragma once
#include "ssd_common.cuh"
#include "ssd_grid.cuh"
#include "ssd_features.cuh"
#include "ssd_selfdrive.cuh"

#define CK_THREADS 256
#define CK_WARPS (CK_THREADS / 32)
#define CK_ROWS 32                  // rows per CTA (<= CK_THREADS: one thread per row writes row_ok)
#define CK_MAX_COLS 40              // feature envs: 8 metric rows + 4 accumulators x 8 agents
#define CK_LAYOUT_VERSION 1u        // hashed into config_tag: bump whenever a row's layout changes

enum { CK_GRID = 0, CK_FEAT = 1, CK_CAR = 2 };

struct CkSeg { uint8_t* base; long long stride; int bytes; int row_off; };   // env bytes at base + env * stride (bytes % 16 == 0)
struct CkCol { uint8_t* base; int elem; int row_off; };                     // element of env at base + env * elem (4 or 8 bytes)

struct CkParams {
    int fam;                        // CK_GRID / CK_FEAT / CK_CAR
    int E, n, row_bytes;
    int zero_fill;                  // the row has padding bytes that no segment or column covers (saved as zeros)
    int nseg, ncol;
    CkSeg seg[2];
    CkCol col[CK_MAX_COLS];
    // validation
    int H, W, horizon, n_apple, n_waste;
    int lists_off, LA, LW;          // feature envs: row offset of the apple list (the waste list follows at lists_off + LA)
    int car_crossed_off, car_meta_off;
};

__device__ __forceinline__ uint32_t ck_valid_word(int npts, int w)
{
    const int left = npts - 32 * w;
    return left >= 32 ? 0xFFFFFFFFu : (left <= 0 ? 0u : ((1u << left) - 1u));
}

// agent word row | col << 8 | ori << 16 (grid record and feature-env record alike)
__device__ __forceinline__ bool ck_agent_bad(const CkParams& p, uint32_t v)
{
    return (int)(v & 255u) >= p.H || (int)((v >> 8) & 255u) >= p.W || (v >> 16) > 3u;
}

// Every field a later kernel uses as an index or loop bound (warp-collective; the result is warp-uniform).
__device__ __forceinline__ bool ck_row_valid(const CkParams& p, const uint8_t* row, uint32_t* scratch, int lane)
{
    const uint32_t* w = reinterpret_cast<const uint32_t*>(row);
    bool bad = false;
    if (p.fam == CK_GRID) {
        int pc = 0;
        if (lane < p.n) bad = ck_agent_bad(p, w[RO_AGENTS / 4 + lane]);
        if (lane >= 8 && lane < 16) bad = bad || (w[RO_AMASK / 4 + lane - 8] & ~ck_valid_word(p.n_apple, lane - 8)) != 0u;
        if (lane >= 16 && lane < 24) {
            const uint32_t m = w[RO_WMASK / 4 + lane - 16];
            bad = bad || (m & ~ck_valid_word(p.n_waste, lane - 16)) != 0u;
            pc = __popc(m);
        }
        pc = __reduce_add_sync(FULL, pc);
        if (lane == 0) {
            const int t = (int)w[RO_T / 4];
            bad = bad || t < 0 || t > p.horizon || (int)w[RO_HCOUNT / 4] != pc;
        }
        return !__any_sync(FULL, bad);
    }
    if (p.fam == CK_CAR) {
        if (lane == 0) {
            const uint32_t nc = *reinterpret_cast<const uint32_t*>(row + p.car_meta_off) & 0xFFu;
            const uint32_t crossed = *reinterpret_cast<const uint32_t*>(row + p.car_crossed_off);
            bad = nc > (uint32_t)p.n;
            if (!bad) {
                for (uint32_t i = 0; i < nc; i++) bad = bad || ((crossed >> (4 * i)) & 15u) >= (uint32_t)p.n;
                if (nc < 8u) bad = bad || (crossed >> (4 * nc)) != 0u;      // appending ORs into the free nibbles
            }
        }
        return !__any_sync(FULL, bad);
    }
    // feature envs: lengths, agents and t first (the lengths bound the list scan below)
    const uint32_t nA = w[FR_NA], nW = w[FR_NW];
    if (lane < p.n) bad = ck_agent_bad(p, w[FR_AGENT + lane]);
    if (lane == 0) bad = bad || nA > (uint32_t)p.n_apple || nW > (uint32_t)p.n_waste || (int)w[FR_T] < 0 || (int)w[FR_T] > p.horizon;
    if (__any_sync(FULL, bad)) return false;
    // every entry names a point, and the entries of a list set exactly the bits of its presence mask, each once
    if (lane < 16) scratch[lane] = 0u;
    __syncwarp();
    const uint8_t* al = row + p.lists_off;
    const uint8_t* wl = al + p.LA;
    for (uint32_t j = lane; j < nA; j += 32) {
        const uint32_t e = al[j];
        if (e >= (uint32_t)p.n_apple) bad = true;
        else atomicOr(scratch + (e >> 5), 1u << (e & 31u));
    }
    for (uint32_t j = lane; j < nW; j += 32) {
        const uint32_t e = wl[j];
        if (e >= (uint32_t)p.n_waste) bad = true;
        else atomicOr(scratch + 8 + (e >> 5), 1u << (e & 31u));
    }
    __syncwarp();
    int pa = 0, pw = 0;
    if (lane < 8) {
        bad = bad || scratch[lane] != w[FR_AM + lane] || scratch[8 + lane] != w[FR_WM + lane];
        pa = __popc(scratch[lane]); pw = __popc(scratch[8 + lane]);
    }
    pa = __reduce_add_sync(FULL, pa);
    pw = __reduce_add_sync(FULL, pw);
    bad = bad || (uint32_t)pa != nA || (uint32_t)pw != nW;
    const bool ok = !__any_sync(FULL, bad);
    __syncwarp();                                        // the scratch words are reused by the warp's next row
    return ok;
}

// local env of row r (-1: outside [0, E))
__device__ __forceinline__ int ck_env(const CkParams& p, const int32_t* idx, int r)
{
    const int e = idx ? idx[r] : r;
    return (e >= 0 && e < p.E) ? e : -1;
}

// rows [r0, r0 + nr): rows_dev + r0 * row_bytes is one contiguous, 16-byte aligned run
__global__ void __launch_bounds__(CK_THREADS) ck_save_kernel(const CkParams p, const int32_t* __restrict__ idx, int count,
                                                             uint8_t* __restrict__ rows)
{
    extern __shared__ __align__(16) uint8_t ck_sm[];
    __shared__ int s_env[CK_ROWS];
    const int r0 = blockIdx.x * CK_ROWS, nr = min(CK_ROWS, count - r0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int stage16 = nr * p.row_bytes / 16;
    uint4* st4 = reinterpret_cast<uint4*>(ck_sm);
    if (threadIdx.x < nr) s_env[threadIdx.x] = ck_env(p, idx, r0 + threadIdx.x);
    if (p.zero_fill)
        for (int i = threadIdx.x; i < stage16; i += CK_THREADS) st4[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    // env-major segments: warp per row
    for (int r = warp; r < nr; r += CK_WARPS) {
        const int env = s_env[r];
        uint8_t* dst = ck_sm + (size_t)r * p.row_bytes;
        for (int s = 0; s < p.nseg; s++) {
            const uint8_t* src = p.seg[s].base + (size_t)max(env, 0) * p.seg[s].stride;
            for (int o = lane * 16; o < p.seg[s].bytes; o += 32 * 16) {
                const uint4 v = env >= 0 ? *reinterpret_cast<const uint4*>(src + o) : make_uint4(0u, 0u, 0u, 0u);
                *reinterpret_cast<uint4*>(dst + p.seg[s].row_off + o) = v;
            }
        }
        if (p.fam == CK_FEAT) {
            // the bytes behind a list's end are leftovers of earlier list contents that no kernel reads: saved as zeros, so
            // that equal states give equal rows
            __syncwarp();
            const uint32_t* rec = reinterpret_cast<const uint32_t*>(dst);
            const int nA = (int)min(rec[FR_NA], (uint32_t)p.LA), nW = (int)min(rec[FR_NW], (uint32_t)p.LW);
            uint8_t* al = dst + p.lists_off;
            for (int j = nA + lane; j < p.LA; j += 32) al[j] = 0;
            for (int j = nW + lane; j < p.LW; j += 32) al[p.LA + j] = 0;
        }
    }
    // [k][E] columns: consecutive threads, consecutive rows
    for (int i = threadIdx.x; i < nr * p.ncol; i += CK_THREADS) {
        const int c = i / nr, r = i - c * nr;
        const int env = s_env[r];
        const CkCol col = p.col[c];
        uint8_t* dst = ck_sm + (size_t)r * p.row_bytes + col.row_off;
        if (col.elem == 8)
            *reinterpret_cast<unsigned long long*>(dst) = env >= 0 ? reinterpret_cast<const unsigned long long*>(col.base)[env] : 0ull;
        else
            *reinterpret_cast<uint32_t*>(dst) = env >= 0 ? reinterpret_cast<const uint32_t*>(col.base)[env] : 0u;
    }
    __syncthreads();
    uint4* out = reinterpret_cast<uint4*>(rows + (size_t)r0 * p.row_bytes);
    for (int i = threadIdx.x; i < stage16; i += CK_THREADS) out[i] = st4[i];
}

__global__ void __launch_bounds__(CK_THREADS) ck_load_kernel(const CkParams p, const int32_t* __restrict__ idx, int count,
                                                             const uint8_t* __restrict__ rows, uint8_t* __restrict__ row_ok)
{
    extern __shared__ __align__(16) uint8_t ck_sm[];
    __shared__ int s_env[CK_ROWS];
    __shared__ uint32_t s_scratch[CK_WARPS][16];
    const int r0 = blockIdx.x * CK_ROWS, nr = min(CK_ROWS, count - r0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int stage16 = nr * p.row_bytes / 16;
    uint4* st4 = reinterpret_cast<uint4*>(ck_sm);
    const uint4* in = reinterpret_cast<const uint4*>(rows + (size_t)r0 * p.row_bytes);
    for (int i = threadIdx.x; i < stage16; i += CK_THREADS) st4[i] = in[i];
    if (threadIdx.x < nr) s_env[threadIdx.x] = ck_env(p, idx, r0 + threadIdx.x);
    __syncthreads();
    // validate, then the env-major segments: warp per row.  A rejected row writes nothing (s_env = -1 from here on).
    for (int r = warp; r < nr; r += CK_WARPS) {
        const uint8_t* src = ck_sm + (size_t)r * p.row_bytes;
        const int env = s_env[r];
        const bool ok = env >= 0 && ck_row_valid(p, src, s_scratch[warp], lane);
        __syncwarp();
        if (lane == 0 && !ok) s_env[r] = -1;
        if (!ok) continue;
        for (int s = 0; s < p.nseg; s++) {
            uint8_t* dst = p.seg[s].base + (size_t)env * p.seg[s].stride;
            for (int o = lane * 16; o < p.seg[s].bytes; o += 32 * 16)
                *reinterpret_cast<uint4*>(dst + o) = *reinterpret_cast<const uint4*>(src + p.seg[s].row_off + o);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nr * p.ncol; i += CK_THREADS) {
        const int c = i / nr, r = i - c * nr;
        const int env = s_env[r];
        if (env < 0) continue;
        const CkCol col = p.col[c];
        const uint8_t* src = ck_sm + (size_t)r * p.row_bytes + col.row_off;
        if (col.elem == 8) reinterpret_cast<unsigned long long*>(col.base)[env] = *reinterpret_cast<const unsigned long long*>(src);
        else reinterpret_cast<uint32_t*>(col.base)[env] = *reinterpret_cast<const uint32_t*>(src);
    }
    if (row_ok && threadIdx.x < nr) row_ok[r0 + threadIdx.x] = s_env[threadIdx.x] >= 0 ? 1 : 0;
}
