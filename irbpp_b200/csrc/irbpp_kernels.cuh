// irbpp_kernels.cuh -- the packing-environment step as two kernels for sm_100a.
//
//   irbpp_scan_kernel        one CTA (128 threads) per bin
//     A  apply the chosen candidate: decode (binPhy.py:234-236), prejudge (:238-245), drop height of that
//        pose, placement test (Interface.py:365-369 semantics), heightmap update (space.py:213 closed
//        form), reward / episode bookkeeping (binPhy.py:299-327, monitor.py:58-75), item queue
//        (IRcreator.py:6-24), auto-reset on failure (shmem_vec_env.py:140-144); float32 copy of the
//        heightmap + next_item_vec into the observation (binPhy.py:196-203); state write-back
//     B  scan every (rotation, X, Y) pose for the next item: drop height + feasibility
//        (space.py:98-129), one warp per rotation, lanes = poses; level quantisation with NumPy
//        floor_divide semantics (cvTools.py:78-79); one 16x16 bitmap per (rotation, level) by warp
//        ballots -> global scratch (L2 resident).  Tables that are constant on square blocks of cells
//        (voxel shapes) are scanned from block maxima of the heightmap (TileEntry lists)
//   irbpp_candidates_kernel  one CTA per 4 bins (up to four rotations) or 8 bins (from R = 8), one warp per bin
//     C  candidate extraction (cvTools.py:61-103): the (bin, rotation, level) images of the CTA are
//        ordered by a cost key; every (image, start pixel) pair is one lane's task, dealt in that order
//        so that the lanes of a warp carry contours of similar length: border following, then (after
//        re-dealing the contours by length) approxPolyDP + convex filter (irbpp_contour.cuh), results
//        OR-ed into a 256-bit set per (bin, rotation) in shared memory (np.unique == sorted set)
//     D  select / pad (binPhy.py:205-225): one warp per bin ranks the set bits and writes the
//        candidate rows of the observation (float32, envs.py:151,163 cast) and the packed candidate
//        table the next step decodes its action from
// (paths relative to the reference root)
//
// Why two kernels: phase C is one serial task per lane with ~40 tasks per bin; inside a one-bin CTA it
// ran at ~3 active lanes per instruction and left the other warps waiting at a barrier (profiles/).
// Splitting lets phase C pack tasks of several bins into full warps and lets phase B run with 12 KB of
// shared memory per CTA.  The hand-over (float64 drop heights, masks, level bitmaps: ~9 KB per bin) is
// written and re-read within microseconds and stays in the 126 MB L2.
//
// Arithmetic is IEEE float64 exactly as NumPy performs it (compile with -fmad=false); masks are
// folded into the tables as +/-inf sentinels at load time, which changes no comparison result.
#pragma once
#include <stdint.h>
#include <math.h>
#include "irbpp_contour.cuh"
#include "irbpp_math.cuh"
#include "irbpp_heuristic.cuh"
#include "irbpp_tma.cuh"

namespace irbpp {

constexpr int HX = 32, HY = 32;          // heightmap cells (rangeX_C, rangeY_C)
constexpr int AX = 16, AY = 16;          // action grid (rangeX_A, rangeY_A)
constexpr int STEP = 2;                  // stepSize = resolutionAct / resolutionH
constexpr int NPOSE = AX * AY;           // 256 poses per rotation
constexpr int CTA_THREADS = 128;
constexpr int CTA_WARPS = CTA_THREADS / 32;
// CTA shapes of the candidates kernel (one warp per bin): 4 bins per CTA up to four rotations, 8 from WIDE_MIN_R rotations on.
// Measured (profiles/README.md, round 2 sweep): BlockOut R = 4  0.109 ms with 4 bins / 0.126 with 8 (512 CTAs of 62 KB no longer
// fit one wave); irregular R = 8  0.370 / 0.355; R = 24  2.91 / 2.28 -- with many rotations a CTA's fixed phases amortise over
// more images and the task deal balances over 256 lanes.  Fewer than 4 bins, or more warps than bins, lost everywhere.
#ifndef IRBPP_ENVS_PER_CTA
#define IRBPP_ENVS_PER_CTA 4
#endif
#ifndef IRBPP_ENVS_PER_CTA_WIDE
#define IRBPP_ENVS_PER_CTA_WIDE 8
#endif
#ifndef IRBPP_WIDE_MIN_R
#define IRBPP_WIDE_MIN_R 8
#endif
constexpr int ENVS_PER_CTA_NARROW = IRBPP_ENVS_PER_CTA;
constexpr int ENVS_PER_CTA_WIDE = IRBPP_ENVS_PER_CTA_WIDE;
__host__ __device__ inline int envs_per_cta_for(int R) { return R >= IRBPP_WIDE_MIN_R ? ENVS_PER_CTA_WIDE : ENVS_PER_CTA_NARROW; }
constexpr int MAX_LEVELS = 64;           // level-image slots per (bin, rotation) in the scratch
#ifndef IRBPP_TASKS_PER_LANE
#define IRBPP_TASKS_PER_LANE 3
#endif
constexpr int TASKS_PER_LANE = IRBPP_TASKS_PER_LANE;        // micro-tasks a lane takes per batch of the candidates kernel (one follow / sort / approximate cycle)
constexpr int TASK_TAB = 384;            // start pixels of a round listed explicitly (the rest are found by search)
constexpr int FAST_CAP = 64;             // contour points on the fast path (32 was measured slower: every overflow redo stalls a warp)
constexpr int BIG_CAP = 1024;            // contour points on the overflow path
constexpr int LEVEL_OFFSET = 32;         // levels in [-32, 31] -> presence bit (level + 32)
constexpr int MAX_QUEUE = 16;            // buffer_size limit
constexpr int MAX_ROT = 32;
constexpr double POSZ_INVALID = 1e3;     // space.py:101,126

enum Mode : int {
    MODE_RESET = 0,        // reset selected envs, emit observation
    MODE_STEP = 1,         // phase A then observation (online: B-D for queue[0]; buffered: order obs)
    MODE_CANDIDATES = 2,   // get_action_candidates(order): B-D for queue[order]
    MODE_ALL_OBS = 3,      // get_all_possible_observation: one pipeline pass per queue slot
    MODE_DEBUG_SCAN = 4,   // B-D for a caller-supplied item, no state change
    MODE_DEBUG_HULLS = 5,  // C-D on caller-supplied posZValid / mask (levels kernel instead of scan)
};

struct ShapeRot {          // one (shape, rotation) entry, device resident
    int32_t w, h;          // window in heightmap cells (rangeX_OH, rangeY_OH; space.py:105)
    int32_t nX, nY;        // number of X / Y positions scanned: A - ceil(ext/resA) + 1 (space.py:115-116)
    uint32_t okx, oky;     // bit lx set <=> prejudge passes in x / y for that lx (binPhy.py:240-241)
    int32_t any_zero;      // maskB has a zero cell -> the window max includes a 0 term
    int32_t tile;          // 4 / 2: the bottom table is constant on tile x tile blocks (see TileEntry); 1: cell list
    double ez;             // round(extent_z, 6)   (space.py:104,120)
    int64_t off;           // offset of Bs / Ts of this entry in the pools (doubles)
    int32_t tile_off;      // first TileEntry of this (shape, rotation)
    int32_t ntiles;
};

// Bottom tables of voxel shapes (BlockOut) are constant on square blocks of heightmap cells.  Rounding is
// monotone, so max over a block of fl(hm - b) == fl(max over the block of hm - b): the scan can take the
// block maxima M of the heightmap once per bin and then visit one entry per BLOCK instead of one per
// cell -- bit-identical, 16x fewer window operations for 4x4 blocks.  Detected per shape at load time;
// tables without that structure use the per-cell loop.
// One entry of a rotation's scan list: either a block of a block-structured table (offset into the
// block-maxima array M, indexed like the action grid) or one unmasked cell of an arbitrary table (offset
// into the column-parity heightmap planes).  Masked cells / blocks have no entry.
struct alignas(16) TileEntry {     // 16 bytes: one LDS.128 per entry
    int32_t off;           // BYTE offset added to the pose's base address: 8 * (block du*16 + dv), 8 * cell hm_index(i, j)
    int32_t pad;
    double b;              // bottom height of the block / cell
};

// Scalar state of one bin, 128 bytes so that one warp loads / stores it with one coalesced access.
struct EnvState {
    int32_t cursor;            // position in the item-id sequence (persists across episodes)
    int32_t cur_item;          // item the current candidate table refers to (binPhy.py: next_item_ID)
    int32_t order_act;         // binPhy.py: orderAction
    int32_t packed;            // items packed in this episode (item_idx)
    int32_t ep_len;            // steps in this episode
    int32_t mask_any;          // sum(naiveMask) != 0 of the last scan (prejudge, binPhy.py:243)
    double vol_sum;            // packed volume (get_ratio, binPhy.py:149-153)
    double ep_rew;             // sum of episode rewards (monitor.py:60)
    int32_t queue[MAX_QUEUE];  // item FIFO (IRcreator.py:6-24)
    int32_t next_seq;          // the sequence entry the next draw returns (fetched one draw ahead: off the step's critical path)
    int32_t seq_pos;           // cursor modulo the sequence length, kept incrementally
    int32_t pad[4];
};
static_assert(sizeof(EnvState) == 128, "EnvState must be 128 bytes");

// The per-bin results of a step, one array of N per field, in the field order of irbpp_step_result.
struct StepResults {
    float* reward; uint8_t* done; uint8_t* valid; uint8_t* error;
    int32_t* counter; int32_t* ep_len; double* ratio; double* ep_reward;
};

// The arrays of N bins in one block: ratio | ep_reward | reward | counter | ep_len | done | valid | error, 8-byte fields
// first so that every array stays aligned.  irbpp_b200/_lib.py RESULT_FIELDS states the same layout.
constexpr size_t RESULT_BYTES_PER_BIN = 8 + 8 + 4 + 4 + 4 + 1 + 1 + 1;
inline StepResults carve_results(void* block, size_t n) {
    char* b = static_cast<char*>(block);
    StepResults r;
    r.ratio = reinterpret_cast<double*>(b);     b += n * 8;
    r.ep_reward = reinterpret_cast<double*>(b); b += n * 8;
    r.reward = reinterpret_cast<float*>(b);     b += n * 4;
    r.counter = reinterpret_cast<int32_t*>(b);  b += n * 4;
    r.ep_len = reinterpret_cast<int32_t*>(b);   b += n * 4;
    r.done = reinterpret_cast<uint8_t*>(b);     b += n;
    r.valid = reinterpret_cast<uint8_t*>(b);    b += n;
    r.error = reinterpret_cast<uint8_t*>(b);
    return r;
}

struct Params {
    // configuration
    int32_t N, R, sel, K;                // K = buffer_size (1 = online)
    int32_t loc_len, order_len, obs_stride;
    int32_t legacy;
    double binz, resZ, binvol, resA;
    // shapes
    int32_t S;
    int32_t maxwh;                       // largest scan list of the library (entries of a warp's staging buffer)
    const ShapeRot* srot;                // [S*R]
    const double* Bs;                    // bottom tables, +inf where maskB == 0
    const double* Ts;                    // top tables, -inf where maskT == 0
    const double* vol;                   // [S]
    const double* reward_tab;            // [S] (vol / binvol) * 10
    const TileEntry* tiles;              // block form of the bottom tables (tile > 1 entries only)
    // sequences
    const int32_t* seq; int32_t L;       // L == 0: ids drawn from the counter-based generator below instead
    uint64_t rng_seed;
    // per-env state
    double* hm;                          // [N][2][32][16] column-parity planes
    uint16_t* cand;                      // [N][cand_stride] rot<<8 | x<<4 | y  (rows padded to 16 bytes: bulk-copied)
    int32_t cand_stride;                 // uint16 entries per row, sel rounded up to a multiple of 8
    EnvState* state;                     // [N]
    // scan -> candidates hand-over (global scratch, L2 resident)
    double* posz;                        // [N][R][256] drop heights (posZmap)
    uint32_t* maskbits;                  // [N][R][8]   feasibility bits (naiveMask)
    uint32_t* bitmaps;                   // [N][R][MAX_LEVELS][8] level images
    int32_t* nlevels;                    // [N][R]
    // inputs of this call
    const int64_t* actions;              // MODE_STEP / MODE_CANDIDATES
    const uint8_t* which;                // MODE_RESET (NULL = all)
    const int32_t* dbg_items;            // MODE_DEBUG_SCAN
    int32_t ws_bytes;                    // per-warp scratch of the candidates kernel (ws_bytes_for(R))
    uint16_t* dlist;                     // [units][2][R*256] phase D lists for R > LISTS_SMEM_MAX_R, else NULL
    uint32_t* ready;                     // [units] hand-over flags: the scan CTA of a unit stores `epoch` when its scratch is written (NULL: grid-wide wait)
    uint32_t epoch;                      // value of this launch (never 0)
    int32_t pose_actions;                // MODE_STEP: actions are flat poses (rot*256 + lx*16 + ly), not candidate rows
    int32_t heur_method, heur_dir;       // heuristic kernel: Heuristic, dirIdx 0..3 (space.py:162-166)
    int32_t* heur_pose;                  // [N][3] rot, lx, ly
    int64_t* heur_index;                 // [N] row of that pose in the candidate table, -1 if absent
    int32_t env_lo, env_hi;              // bins [env_lo, env_hi) handled by this launch (the full range [0, N))
    // outputs
    float* obs;                          // [N][obs_stride] (+ slot offset in MODE_ALL_OBS)
    StepResults res;                     // the device result block
    double* dbg_cand; int32_t* dbg_nhull;
    StepResults res_host;                // host-mapped mirror of this step's results (zero-copy stores; NULL on the device-resident path)
    unsigned long long* phase_cycles;    // [8] summed SM cycles per phase (thread 0 of every CTA), or NULL
    int32_t mode;
};

// A bin's step result, stored to the device block and to the host mirror when there is one.
__device__ __forceinline__ void store_result(const Params& P, int env, float reward, uint8_t done, uint8_t valid,
                                             int32_t counter, int32_t ep_len, double ratio, double ep_reward) {
    auto put = [&](const StepResults& r) {
        r.reward[env] = reward; r.done[env] = done; r.valid[env] = valid;
        r.counter[env] = counter; r.ep_len[env] = ep_len; r.ratio[env] = ratio; r.ep_reward[env] = ep_reward;
    };
    put(P.res);
    if (P.res_host.reward) put(P.res_host);
}

__device__ __forceinline__ void store_error(const Params& P, int env, uint8_t code) {
    P.res.error[env] = code;
    if (P.res_host.error) P.res_host.error[env] = code;
}

// Cell (x, y) of a bin's heightmap: plane y & 1 holds the columns of that parity.
__host__ __device__ __forceinline__ int hm_index(int x, int y) { return ((y & 1) * HX + x) * (HY / 2) + (y >> 1); }

// Counter-based item generator (stand-in for RandomItemCreator, IRcreator.py:26-33, when no explicit sequences
// are loaded): id = mix(seed, env, draw counter) mod S -- i.i.d. uniform ids, no period, no memory.
__host__ __device__ __forceinline__ uint32_t item_rng(uint64_t seed, uint32_t env, uint32_t counter) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ull * (((uint64_t)env << 32) | counter) + 0x9E3779B97F4A7C15ull;   // splitmix64
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (uint32_t)(z >> 32);
}

// generate_item (IRcreator.py:17-24): the id at the bin's cursor.  With explicit sequences the entry was fetched
// by the previous draw (EnvState::next_seq) and this draw fetches the one after it.
// `next` is the caller's register copy of EnvState::next_seq: the load issued here is consumed by the NEXT draw
// (normally in the next step; the caller stores it back with the state), so nothing waits for it.
__device__ __forceinline__ int draw_item(const Params& P, int env, EnvState& st, int& next) {
    if (P.L == 0) {
        const int id = (int)(item_rng(P.rng_seed, (uint32_t)env, (uint32_t)st.cursor) % (uint32_t)P.S);
        st.cursor += 1;
        return id;
    }
    const int id = next;
    int pos = st.seq_pos + 1;
    if (pos >= P.L) pos = 0;
    st.seq_pos = pos;
    st.cursor += 1;
    next = P.seq[(int64_t)env * P.L + pos];
    return id;
}

__host__ __device__ __forceinline__ bool mode_emits_loc(int mode, int K) {
    return !((mode == MODE_STEP || mode == MODE_RESET) && K > 1);
}

// ---- level bitmaps of one rotation -------------------------------------------------------------------
// lv[pass] = level of pose pass*32+lane (or -1).  One 16x16 bitmap (8 words, two rows each) per level
// present, by warp ballots, written to the scratch; returns the number of levels.
__device__ __forceinline__ int emit_level_bitmaps(uint32_t* bm_g, int lane, const int (&lv)[8], uint64_t present) {
    present &= ~(1ull << (LEVEL_OFFSET - 1));        // level -1 is skipped (cvTools.py:84)
    int k = 0;
    while (present) {
        const int b = __ffsll((long long)present) - 1;
        present &= present - 1;
        const int L = b - LEVEL_OFFSET;
        uint32_t mine = 0;
#pragma unroll
        for (int pass = 0; pass < 8; ++pass) {
            const uint32_t bits = __ballot_sync(0xffffffffu, lv[pass] == L);
            if (lane == pass) mine = bits;
        }
        if (lane < 8) bm_g[k * 8 + lane] = mine;
        ++k;
    }
    return k;
}

__device__ __forceinline__ int level_of(const Params& P, double posz, double inv, uint32_t& pres_lo,
                                        uint32_t& pres_hi, int& err) {
    int L = (int)floor_divide_exact(posz, P.resZ, inv);        // cvTools.py:78
    if (L < -LEVEL_OFFSET || L >= LEVEL_OFFSET) { err = 1; return -1; }
    if (L != -1) {
        const int b = L + LEVEL_OFFSET;
        if (b < 32) pres_lo |= 1u << b; else pres_hi |= 1u << (b - 32);
    }
    return L;
}

// ---- phase B: one warp scans one rotation -------------------------------------------------------------
// Writes posz[r][256], maskbits[r][8], the level bitmaps and their count (space.py:98-129,
// cvTools.py:78-85).  Returns true if any pose is feasible.
// `arr` is the array the entry offsets refer to: the block maxima M (pose base = X*16 + Y) for block
// tables, the heightmap planes (pose base = 2X*16 + Y) for cell lists.  The entry list is staged in this
// warp's shared-memory buffer (all lanes read the same entry: a broadcast); each lane carries two poses,
// (X, Y) and (X + 8, Y), so one entry serves two window positions.
__device__ __forceinline__ bool scan_rotation(const Params& P, const double* arr, int stride_x, TileEntry* es,
                                              int env, int item, int r, int lane, int& err) {
    const ShapeRot* sr = P.srot + (int64_t)item * P.R + r;
    const int nX = sr->nX, nY = sr->nY, nt = sr->ntiles;
    const double ez = sr->ez;
    const double init = sr->any_zero ? 0.0 : -INFINITY;
    {
        const TileEntry* __restrict__ te = P.tiles + sr->tile_off;
        __syncwarp();                                   // previous rotation's readers are done
        for (int k = lane; k < nt; k += 32) es[k] = te[k];
        __syncwarp();
    }
    const double inv = 1.0 / P.resZ;
    double* posz_g = P.posz + ((int64_t)env * P.R + r) * NPOSE;
    uint32_t* mask_g = P.maskbits + ((int64_t)env * P.R + r) * 8;
    int lv[8];
    uint32_t pres_lo = 0, pres_hi = 0, any = 0;
    const int Y = lane & 15;
#pragma unroll
    for (int pass = 0; pass < 4; ++pass) {
        const int pA = pass * 32 + lane;
        const int X = pA >> 4;
        const bool validA = (X < nX) && (Y < nY);
        const bool validB = (X + 8 < nX) && (Y < nY);
        double accA = POSZ_INVALID, accB = POSZ_INVALID;
        bool feasA = false, feasB = false;
        if (validA) {
            accA = init; accB = init;
            const double* a0 = arr + X * stride_x + Y;
            const double* b0 = validB ? a0 + 8 * stride_x : a0;                  // pose (X + 8, Y)
#pragma unroll 4
            for (int k = 0; k < nt; ++k) {
                const TileEntry e = es[k];
                const double u = *reinterpret_cast<const double*>(reinterpret_cast<const char*>(a0) + e.off) - e.b;
                const double v = *reinterpret_cast<const double*>(reinterpret_cast<const char*>(b0) + e.off) - e.b;
                accA = (u > accA) ? u : accA;
                accB = (v > accB) ? v : accB;
            }
            feasA = round6_le0(accA + ez - P.binz);
            if (validB) feasB = round6_le0(accB + ez - P.binz); else accB = POSZ_INVALID;
        }
        posz_g[pA] = accA;
        posz_g[pA + 128] = accB;
        const uint32_t mbA = __ballot_sync(0xffffffffu, feasA);
        const uint32_t mbB = __ballot_sync(0xffffffffu, feasB);
        if (lane == 0) { mask_g[pass] = mbA; mask_g[pass + 4] = mbB; }
        any |= mbA | mbB;
        lv[pass] = feasA ? level_of(P, accA, inv, pres_lo, pres_hi, err) : -1;
        lv[pass + 4] = feasB ? level_of(P, accB, inv, pres_lo, pres_hi, err) : -1;
    }
    pres_lo = __reduce_or_sync(0xffffffffu, pres_lo);
    pres_hi = __reduce_or_sync(0xffffffffu, pres_hi);
    const int nl = emit_level_bitmaps(P.bitmaps + ((int64_t)env * P.R + r) * MAX_LEVELS * 8, lane, lv,
                                      ((uint64_t)pres_hi << 32) | pres_lo);
    if (lane == 0) P.nlevels[(int64_t)env * P.R + r] = nl;
    return any != 0;
}

// ---- phase B for arbitrary tables: dense pose packing ------------------------------------------------------
// scan_rotation maps the 16 x 16 action grid onto the lanes as it is, so a rotation whose scanned range is
// nX x nY leaves (256 - nX nY) / 256 of the lane slots idle while they wait for the entry loop -- half of them
// for the irregular library -- and an arbitrary table's entry loop (one entry per unmasked cell, ~60, up to 246)
// is where the scan of general shapes spends its time.  Here only the nX * nY scanned poses are dealt to the
// lanes (pose v -> X = v / nY, Y = v mod nY), four per lane, so one staged entry serves 128 window positions
// and four independent accumulators hide the latency of the max chain.  Results go to posz as before and, as
// one level code per pose, to a 256-byte map in shared memory from which a second, fixed-layout pass takes the
// feasibility bits and the level bitmaps by warp ballots (emit_level_bitmaps).
__device__ __forceinline__ bool scan_rotation_dense(const Params& P, const double* arr, int stride_x, TileEntry* es,
                                                    uint8_t* lv_s /* [256], this warp's */, int env, int item, int r,
                                                    int lane, int& err) {
    const ShapeRot* sr = P.srot + (int64_t)item * P.R + r;
    const int nX = sr->nX, nY = sr->nY, nt = sr->ntiles;
    const int V = nX * nY;
    const double ez = sr->ez;
    const double init = sr->any_zero ? 0.0 : -INFINITY;
    {
        const TileEntry* __restrict__ te = P.tiles + sr->tile_off;
        __syncwarp();                                   // previous rotation's readers are done
        for (int k = lane; k < nt; k += 32) es[k] = te[k];
        reinterpret_cast<uint32_t*>(lv_s)[lane] = 0u;
        reinterpret_cast<uint32_t*>(lv_s)[lane + 32] = 0u;
        __syncwarp();
    }
    const double inv = 1.0 / P.resZ;
    double* posz_g = P.posz + ((int64_t)env * P.R + r) * NPOSE;
    const uint32_t magic = 65536u / (uint32_t)(nY > 0 ? nY : 1) + 1u;      // v / nY == (v * magic) >> 16 for v < 256, nY <= 16
    // PPL poses per lane: chunks of 128 poses with four accumulators per lane, then what is left (nX * nY is
    // rarely a multiple of 128) with two or one, so the tail does not cost a full four-pose pass
    auto chunk = [&](int c0, auto ppl_tag) {
        constexpr int PPL = decltype(ppl_tag)::value;
        int cell[PPL];
        const char* base[PPL];
        bool valid[PPL];
        double acc[PPL];
#pragma unroll
        for (int k = 0; k < PPL; ++k) {
            const int v = c0 + k * 32 + lane;
            valid[k] = v < V;
            const int X = valid[k] ? (int)(((uint32_t)v * magic) >> 16) : 0;
            const int Y = valid[k] ? v - X * nY : 0;
            cell[k] = X * 16 + Y;
            base[k] = reinterpret_cast<const char*>(arr + X * stride_x + Y);
            acc[k] = init;
        }
#pragma unroll 2
        for (int e = 0; e < nt; ++e) {
            const TileEntry en = es[e];
#pragma unroll
            for (int k = 0; k < PPL; ++k) {
                const double u = *reinterpret_cast<const double*>(base[k] + en.off) - en.b;      // entry offsets are in bytes
                acc[k] = (u > acc[k]) ? u : acc[k];
            }
        }
#pragma unroll
        for (int k = 0; k < PPL; ++k) {
            if (valid[k]) {
                const bool feas = round6_le0(acc[k] + ez - P.binz);
                int code = 0;
                if (feas) {
                    const int L = (int)floor_divide_exact(acc[k], P.resZ, inv);        // cvTools.py:78
                    if (L < -LEVEL_OFFSET || L >= LEVEL_OFFSET) { err = 1; code = LEVEL_OFFSET; /* level -1: skipped */ }
                    else code = L + LEVEL_OFFSET + 1;                                    // 1 .. 64
                }
                posz_g[cell[k]] = acc[k];
                lv_s[cell[k]] = (uint8_t)code;
            }
        }
    };
    {
        int c0 = 0;
        for (; V - c0 > 64; c0 += 128) chunk(c0, std::integral_constant<int, 4>());
        if (V - c0 > 32) chunk(c0, std::integral_constant<int, 2>());
        else if (V - c0 > 0) chunk(c0, std::integral_constant<int, 1>());
    }
    __syncwarp();
    // fixed-layout pass: feasibility bits, level presence, bitmaps; poses outside the scanned range keep 1e3 / 0
    uint32_t* mask_g = P.maskbits + ((int64_t)env * P.R + r) * 8;
    int lv[8];
    uint32_t pres_lo = 0, pres_hi = 0, any = 0;
#pragma unroll
    for (int pass = 0; pass < 8; ++pass) {
        const int pA = pass * 32 + lane;
        const int code = lv_s[pA];
        if ((pA >> 4) >= nX || (pA & 15) >= nY) posz_g[pA] = POSZ_INVALID;
        const uint32_t mb = __ballot_sync(0xffffffffu, code != 0);
        if (lane == 0) mask_g[pass] = mb;
        any |= mb;
        const int L = code - (LEVEL_OFFSET + 1);
        lv[pass] = code ? L : -1;
        if (code && L != -1) { const int b = L + LEVEL_OFFSET; if (b < 32) pres_lo |= 1u << b; else pres_hi |= 1u << (b - 32); }
    }
    pres_lo = __reduce_or_sync(0xffffffffu, pres_lo);
    pres_hi = __reduce_or_sync(0xffffffffu, pres_hi);
    const int nl = emit_level_bitmaps(P.bitmaps + ((int64_t)env * P.R + r) * MAX_LEVELS * 8, lane, lv,
                                      ((uint64_t)pres_hi << 32) | pres_lo);
    if (lane == 0) P.nlevels[(int64_t)env * P.R + r] = nl;
    return any != 0;
}

// ---- scan -> candidates hand-over flags -------------------------------------------------------------------
// The candidates grid is launched programmatically (PDL) and becomes resident while the scan grid's last wave
// drains (3.46 waves on the bench workload: for ~13 us about half the SM slots have no scan CTA).  Waiting there
// for the WHOLE scan grid (griddepcontrol.wait) wastes that time for every bin of an earlier wave, so a scan CTA
// publishes a per-unit flag (release) once its part of the scratch is written and a candidates CTA starts as soon
// as the flags of ITS bins carry this launch's epoch (acquire).  No deadlock: the scan CTAs trigger the dependent
// launch at their start, so a candidates CTA exists only when every scan CTA is resident; and a poll that runs out
// falls back to the grid-wide wait.
#ifdef IRBPP_HOST_EMULATION
static inline void ready_publish(uint32_t* f, uint32_t v) { __atomic_store_n(f, v, __ATOMIC_RELEASE); }
static inline uint32_t ready_peek(const uint32_t* f) { return __atomic_load_n(f, __ATOMIC_ACQUIRE); }
static inline void grid_dependency_wait() {}
static inline void backoff() {}
#else
__device__ __forceinline__ void ready_publish(uint32_t* f, uint32_t v) { asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(f), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ready_peek(const uint32_t* f) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
    return v;
}
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void backoff() { __nanosleep(100); }
#endif
constexpr int READY_POLLS = 1 << 16;       // ~10 ms of polling before the fallback

// ---- scan kernel ------------------------------------------------------------------------------------------
#ifndef IRBPP_SCAN_MIN_CTAS
#define IRBPP_SCAN_MIN_CTAS 8
#endif
__global__ void __launch_bounds__(CTA_THREADS, IRBPP_SCAN_MIN_CTAS) irbpp_scan_kernel(const Params P) {
    __shared__ __align__(128) double hm_s[HX * HY];
    extern __shared__ __align__(16) TileEntry estage[];  // CTA_WARPS x P.maxwh: scan list of each warp's rotation
    __shared__ __align__(16) EnvState st_s;              // this bin's scalar state (loaded / stored by warp 0)
    __shared__ double M_s[NPOSE];                        // block maxima of the heightmap (block form of phase B)
    __shared__ double P2_s[NPOSE];                       // 2x2 block maxima
    __shared__ double z_sh;
    __shared__ int ok_sh, rot_sh, lx_sh, ly_sh, item_sh, err_sh, any_sh;
    __shared__ __align__(8) mbarrier_t mbar;             // completion of the bulk copies of this bin's inputs
    __shared__ __align__(16) ShapeRot srot_s[MAX_ROT];   // (56 bytes each) table headers of the item the action places (all rotations), prefetched
    __shared__ long long a_sh;                           // the bin's action
    __shared__ __align__(16) uint8_t lvmap_s[CTA_WARPS * NPOSE];   // per warp: level code of every pose of its rotation (dense scan)
    const int mode = P.mode;
    // One CTA per bin; get_all_possible_observation (MODE_ALL_OBS) runs one CTA per (bin, buffer slot) in a single
    // launch: `vb` indexes the hand-over scratch, the slot picks the item and the place in the observation.
    const int vb = P.env_lo + blockIdx.x;
    const int slot = (mode == MODE_ALL_OBS) ? vb % P.K : 0;
    const int env = (mode == MODE_ALL_OBS) ? vb / P.K : vb;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    asm volatile("griddepcontrol.launch_dependents;");      // the candidates grid may be scheduled as this one drains (PDL)
    if (mode == MODE_RESET && P.which && !P.which[env]) {
        if (P.ready && tid == 0) ready_publish(P.ready + vb, P.epoch);      // nothing to hand over, nobody shall wait
        return;
    }
    long long t_prev = P.phase_cycles ? clock64() : 0;
    auto phase_mark = [&](int idx) {
        if (P.phase_cycles && tid == 0) {
            const long long now = clock64();
            atomicAdd(P.phase_cycles + idx, (unsigned long long)(now - t_prev));
            t_prev = now;
        }
    };

    // ---- load heightmap (column-parity planes, 8 KB), candidate table and the bin's scalar state ----
    // All of these are first-touch DRAM reads (the agent's forward pass sits between two steps).  The 8 KB
    // heightmap and the bin's packed candidate table (1 KB) are brought in by the copy engine: one elected
    // thread arms an mbarrier and issues two 1-D bulk copies (cp.async.bulk), nothing is staged through
    // registers, and the action is decoded from the shared-memory copy of the table -- the chain
    // action -> candidate row no longer costs a second DRAM round trip.
    double* hm_g = P.hm + (int64_t)env * (HX * HY);
    uint16_t* cand_s = reinterpret_cast<uint16_t*>(estage + CTA_WARPS * P.maxwh);     // [cand_stride], behind the staging lists
    const bool need_cand = (mode == MODE_STEP) && !P.pose_actions;
    int64_t a_pf = 0;
    double rew_pf = 0.0, vol_pf = 0.0;      // thread 0: reward and volume of the item being placed (fetched while the copies land)
    if (tid == 0) {
        mbar_init(&mbar, 1);
        if (mode != MODE_RESET) {
            const uint32_t cbytes = need_cand ? (uint32_t)P.cand_stride * 2u : 0u;
            mbar_expect_tx(&mbar, (uint32_t)(HX * HY * sizeof(double)) + cbytes);
            bulk_g2s(hm_s, hm_g, (uint32_t)(HX * HY * sizeof(double)), &mbar);
            if (need_cand) bulk_g2s(cand_s, P.cand + (int64_t)env * P.cand_stride, cbytes, &mbar);
        }
    }
    if (warp == 0) {
        const uint32_t stw = reinterpret_cast<const uint32_t*>(P.state + env)[lane];
        if (mode == MODE_STEP) a_pf = P.actions[env];
        reinterpret_cast<uint32_t*>(&st_s)[lane] = stw;
        if (mode == MODE_STEP && lane == 0) a_sh = a_pf;
    }
    if (mode == MODE_RESET) {
        double2* dst = reinterpret_cast<double2*>(hm_s);
        for (int i = tid; i < HX * HY / 2; i += CTA_THREADS) dst[i] = make_double2(0.0, 0.0);
    }
    if (tid == 0) { err_sh = 0; any_sh = 0; }
    __syncthreads();                       // mbarrier initialised, state in shared memory
    if (mode == MODE_STEP) {
        // while the bulk copies land: the table headers of the item to be placed, all rotations (48 bytes each), so
        // that decoding the action does not start another round trip to L2
        static_assert(sizeof(ShapeRot) % 8 == 0, "headers are copied as 8-byte words");
        constexpr int HW = (int)(sizeof(ShapeRot) / 8);
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(P.srot + (int64_t)st_s.cur_item * P.R);
        for (int i = tid; i < P.R * HW; i += CTA_THREADS) reinterpret_cast<unsigned long long*>(srot_s)[i] = src[i];
        if (tid == 0) { rew_pf = P.reward_tab[st_s.cur_item]; vol_pf = P.vol[st_s.cur_item]; }   // thread 0's bookkeeping inputs
    }
    if (mode != MODE_RESET) mbar_wait(&mbar, 0);
    if (mode == MODE_STEP) __syncthreads();        // headers visible to every thread

    int32_t* queue_g = st_s.queue;
    int next_seq = st_s.next_seq;          // thread 0's register copy; written back with the state
    auto draw = [&]() { return draw_item(P, env, st_s, next_seq); };
    // zero the bin's heightmap in global memory (reset / auto-reset); the shared copy is zeroed by the caller
    auto zero_hm_global = [&]() {
        double2* dst = reinterpret_cast<double2*>(hm_g);
        for (int i = tid; i < HX * HY / 2; i += CTA_THREADS) dst[i] = make_double2(0.0, 0.0);
    };
    bool st_dirty = false;

    // ---- phase A: bookkeeping / apply action ----
    if (mode == MODE_RESET) {
        if (tid == 0) {
            const int nfill = P.K > 1 ? P.K : 1;
            for (int q = 0; q < nfill; ++q) queue_g[q] = draw();
            st_s.packed = 0; st_s.ep_len = 0; st_s.vol_sum = 0.0; st_s.ep_rew = 0.0;
            st_s.order_act = 0;
            item_sh = queue_g[0];
        }
        zero_hm_global();
        st_dirty = true;
        __syncthreads();
    } else if (mode == MODE_STEP) {
        // every thread decodes the action: the whole CTA then fetches the placed rotation's top table (what the
        // heightmap update needs) while warp 0 computes the drop height of that single pose from the bottom table --
        // the two table reads overlap instead of following each other
        const int item = st_s.cur_item;
        int rot = 0, lx = 0, ly = 0;
        bool ok = true;
        {
            const int64_t a = a_sh;
            if (a < 0 || a >= (P.pose_actions ? P.R * NPOSE : P.sel)) { ok = false; if (tid == 0) err_sh = 2; }
            else {
                const uint32_t c = P.pose_actions ? (uint32_t)a : (uint32_t)cand_s[a];
                rot = c >> 8; lx = (c >> 4) & 15; ly = c & 15;
                if (rot >= P.R) { rot = 0; ok = false; if (tid == 0) err_sh = 2; }
            }
        }
        const ShapeRot& sr = srot_s[rot];
        const int w = sr.w, h = sr.h;
        const double* __restrict__ T = P.Ts + sr.off;
        double tp0 = -INFINITY, tp1 = -INFINITY;               // this thread's first two cells of the top table
        if (tid < w * h) tp0 = T[tid];
        if (tid + CTA_THREADS < w * h) tp1 = T[tid + CTA_THREADS];
        if (warp == 0) {
            // prejudge (binPhy.py:238-245)
            if (!((sr.okx >> lx) & 1u) || !((sr.oky >> ly) & 1u)) ok = false;
            if (!st_s.mask_any) ok = false;
            double z = POSZ_INVALID;     // posZmap keeps 1e3 outside the scanned range (space.py:101)
            if (lx < sr.nX && ly < sr.nY) {
                const double* __restrict__ B = P.Bs + sr.off;
                double acc = sr.any_zero ? 0.0 : -INFINITY;
                for (int c = lane; c < w * h; c += 32) {
                    const int i = c / h, j = c - i * h;
                    const double v = hm_s[hm_index(STEP * lx + i, STEP * ly + j)] - B[c];
                    acc = (v > acc) ? v : acc;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double t = __shfl_xor_sync(0xffffffffu, acc, o);
                    acc = (t > acc) ? t : acc;
                }
                z = acc;
            }
            // Interface.simulateHeight (Interface.py:365-369): AABB top above the bin -> failure
            if (ok && !round6_le0(z + sr.ez - P.binz)) ok = false;
            if (lane == 0) { z_sh = z; ok_sh = ok; }
        }
        __syncthreads();
        ok = ok_sh != 0;
        if (ok) {
            // heightmap update: hm[win] = max(hm[win], (T + z) * maskT)   (space.py:213)
            const double z = z_sh;
            const int x0 = STEP * lx, y0 = STEP * ly;
            // only the cells the item raises are written back (in shared and in global memory): a placement
            // touches at most w x h cells, the other 8 KB of the bin's heightmap stay as they are in HBM
            for (int c = tid; c < w * h; c += CTA_THREADS) {
                const int i = c / h, j = c - i * h;
                const double t = (c == tid) ? tp0 : ((c == tid + CTA_THREADS) ? tp1 : T[c]);
                const double v = t + z;
                const int idx = hm_index(x0 + i, y0 + j);
                if (v > hm_s[idx]) { hm_s[idx] = v; hm_g[idx] = v; }
            }
        } else {
            for (int i = tid; i < HX * HY; i += CTA_THREADS) hm_s[i] = 0.0;    // auto-reset
            zero_hm_global();
        }
        if (tid == 0) {
            const int nfill = P.K > 1 ? P.K : 1;
            if (ok) {
                const double rew = rew_pf;
                store_result(P, env, (float)rew, 0, 1, -1, 0, -1.0, 0.0);
                st_s.packed += 1; st_s.ep_len += 1;
                st_s.vol_sum += vol_pf;
                st_s.ep_rew += rew;
                // item_creator.update_item_queue(orderAction); generate_item()  (binPhy.py:324-325)
                const int oa = st_s.order_act;
                for (int q = oa; q + 1 < nfill; ++q) queue_g[q] = queue_g[q + 1];
                queue_g[nfill - 1] = draw();
            } else {
                store_result(P, env, 0.0f, 1, 1, st_s.packed, st_s.ep_len + 1, st_s.vol_sum / P.binvol, st_s.ep_rew + 0.0);
                st_s.packed = 0; st_s.ep_len = 0; st_s.vol_sum = 0.0; st_s.ep_rew = 0.0;
                st_s.order_act = 0;
                for (int q = 0; q < nfill; ++q) queue_g[q] = draw();   // reset(): clear + preview
            }
            item_sh = queue_g[0];
        }
        st_dirty = true;
        __syncthreads();
    } else if (mode == MODE_CANDIDATES) {
        if (tid == 0) {
            int64_t oa = P.actions[env];
            if (oa < 0 || oa >= P.K) { err_sh = 3; oa = 0; }
            st_s.order_act = (int)oa;
            item_sh = queue_g[oa];
        }
        st_dirty = true;
        __syncthreads();
    } else if (mode == MODE_ALL_OBS) {
        if (tid == 0) item_sh = queue_g[slot];
        __syncthreads();
    } else {   // MODE_DEBUG_SCAN
        if (tid == 0) item_sh = P.dbg_items[env];
        __syncthreads();
    }
    phase_mark(0);   // load + phase A

    const bool emit_loc = mode_emits_loc(mode, P.K);
    float* obs_g = P.obs + (int64_t)env * P.obs_stride + slot * P.loc_len;
    const int item = item_sh;
    const int ncand = P.sel * 5;

    // the heightmap is final for this call: float32 copy into the observation, state write-back
    {
        const int hm_obs_off = emit_loc ? ncand + 9 : P.K;
        for (int i = tid; i < HX * HY; i += CTA_THREADS)
            obs_g[hm_obs_off + i] = (float)hm_s[hm_index(i >> 5, i & 31)];
    }
    if (!emit_loc) {
        // order observation: [next k item ids | heightmap]  (binPhy.py:229-230)
        for (int i = tid; i < P.K; i += CTA_THREADS) obs_g[i] = (float)queue_g[i];
        if (tid == 0) { store_error(P, env, (uint8_t)err_sh); st_s.next_seq = next_seq; }
        if (st_dirty && warp == 0) {
            __syncwarp();
            reinterpret_cast<uint32_t*>(P.state + env)[lane] = reinterpret_cast<const uint32_t*>(&st_s)[lane];
        }
        return;
    }
    if (tid < 9) obs_g[ncand + tid] = (tid == 0) ? (float)item : 0.0f;      // next_item_vec (binPhy.py:191)

    // ---- phase B ----
    {
        int err = 0;
        bool any = false;
        const int tile = P.srot[(int64_t)item * P.R].tile;      // same for every rotation of a shape
        if (tile > 1) {
            // block maxima of the heightmap, one entry per action-grid offset.  max is exact, so the
            // 4x4 maximum is taken as the maximum of four 2x2 maxima (8 loads per entry instead of 16).
            for (int e = tid; e < NPOSE; e += CTA_THREADS) {
                const double* p0 = hm_s + (2 * (e >> 4)) * (HY / 2) + (e & 15);     // plane of even y, row x = 2a
                const double* p1 = p0 + HX * (HY / 2);                              // plane of odd y
                const double m0 = (p0[0] > p0[HY / 2]) ? p0[0] : p0[HY / 2];
                const double m1 = (p1[0] > p1[HY / 2]) ? p1[0] : p1[HY / 2];
                P2_s[e] = (m0 > m1) ? m0 : m1;
            }
            __syncthreads();
            if (tile == 4) {
                for (int e = tid; e < NPOSE; e += CTA_THREADS) {
                    double m = -INFINITY;
                    if ((e >> 4) < AX - 1 && (e & 15) < AY - 1) {
                        const double m0 = (P2_s[e] > P2_s[e + 1]) ? P2_s[e] : P2_s[e + 1];
                        const double m1 = (P2_s[e + 16] > P2_s[e + 17]) ? P2_s[e + 16] : P2_s[e + 17];
                        m = (m0 > m1) ? m0 : m1;
                    }
                    M_s[e] = m;
                }
                __syncthreads();
            }
            const double* Marr = (tile == 4) ? M_s : P2_s;
            for (int r = warp; r < P.R; r += CTA_WARPS)
                any |= scan_rotation(P, Marr, 16, estage + warp * P.maxwh, vb, item, r, lane, err);
        } else {
            for (int r = warp; r < P.R; r += CTA_WARPS)
                any |= scan_rotation_dense(P, hm_s, STEP * (HY / 2), estage + warp * P.maxwh, lvmap_s + warp * NPOSE, vb, item, r, lane, err);
        }
        if (lane == 0 && any) any_sh = 1;
        if (__any_sync(0xffffffffu, err) && lane == 0) err_sh = 4;
    }
    __syncthreads();
    if (tid == 0) {
        // (several CTAs per bin in MODE_ALL_OBS: only error codes are written; the candidates kernel may overwrite with its own code)
        if (mode != MODE_ALL_OBS || err_sh) store_error(P, env, (uint8_t)err_sh);
        const bool write_state = (mode == MODE_STEP || mode == MODE_RESET || mode == MODE_CANDIDATES ||
                                  (mode == MODE_ALL_OBS && slot == P.K - 1));
        if (write_state) { st_s.cur_item = item; st_s.mask_any = any_sh; }
        st_s.next_seq = next_seq;
    }
    {
        const bool write_state = (mode == MODE_STEP || mode == MODE_RESET || mode == MODE_CANDIDATES ||
                                  (mode == MODE_ALL_OBS && slot == P.K - 1));
        if (st_dirty || write_state) {
            __syncthreads();
            if (warp == 0) reinterpret_cast<uint32_t*>(P.state + env)[lane] = reinterpret_cast<const uint32_t*>(&st_s)[lane];
        }
    }
    if (P.ready) {
        // hand-over: all writes of the CTA (scratch, observation, state) happen-before thread 0's release store through
        // the block barrier -- a release is cumulative over what its thread has synchronised with -- so one fence per
        // CTA (the MEMBAR.GPU inside st.release) is enough
        __syncthreads();
        if (tid == 0) ready_publish(P.ready + vb, P.epoch);
    }
    phase_mark(1);   // observation heightmap, write-back, scan, level bitmaps
}


// ---- levels kernel (MODE_DEBUG_HULLS): level bitmaps from caller-supplied posZValid / mask ------------------
__global__ void __launch_bounds__(CTA_THREADS) irbpp_levels_kernel(const Params P) {
    __shared__ int err_sh;
    const int env = P.env_lo + blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double inv = 1.0 / P.resZ;
    if (threadIdx.x == 0) err_sh = 0;
    __syncthreads();
    int err = 0;
    for (int r = warp; r < P.R; r += CTA_WARPS) {
        const double* posz_g = P.posz + ((int64_t)env * P.R + r) * NPOSE;
        const uint32_t* mask_g = P.maskbits + ((int64_t)env * P.R + r) * 8;
        int lv[8];
        uint32_t pres_lo = 0, pres_hi = 0;
#pragma unroll
        for (int pass = 0; pass < 8; ++pass) {
            const bool feas = (mask_g[pass] >> lane) & 1u;
            lv[pass] = feas ? level_of(P, posz_g[pass * 32 + lane], inv, pres_lo, pres_hi, err) : -1;
        }
        pres_lo = __reduce_or_sync(0xffffffffu, pres_lo);
        pres_hi = __reduce_or_sync(0xffffffffu, pres_hi);
        const int nl = emit_level_bitmaps(P.bitmaps + ((int64_t)env * P.R + r) * MAX_LEVELS * 8, lane, lv,
                                          ((uint64_t)pres_hi << 32) | pres_lo);
        if (lane == 0) P.nlevels[(int64_t)env * P.R + r] = nl;
    }
    if (err) err_sh = 4;
    __syncthreads();
    if (threadIdx.x == 0) store_error(P, env, (uint8_t)err_sh);
}

// ---- heuristic kernel (space.py:162-227) ---------------------------------------------------------------------
// One CTA per bin over the scan scratch of the bin's current item: every thread scores the poses
// e = tid, tid + 128, ... (flat (rot, lx, ly) order), then a lexicographic (score, e) minimum gives
// np.argmin's first-minimum pose.  Also looks the pose up in the bin's candidate table.
__global__ void __launch_bounds__(CTA_THREADS) irbpp_heuristic_kernel(const Params P) {
    __shared__ __align__(16) double hm_s[HX * HY];
    __shared__ double best_sh[CTA_WARPS];
    __shared__ int beste_sh[CTA_WARPS];
    __shared__ int idx_sh;
    const int env = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int item = P.state[env].cur_item;
    const int method = P.heur_method;
    if (method == HEUR_HM) {
        const double2* src = reinterpret_cast<const double2*>(P.hm + (int64_t)env * (HX * HY));
        double2* dst = reinterpret_cast<double2*>(hm_s);
        for (int i = tid; i < HX * HY / 2; i += CTA_THREADS) dst[i] = src[i];
    }
    if (tid == 0) idx_sh = 0x7fffffff;
    __syncthreads();
    auto hm_at = [&](int x, int y) { return hm_s[hm_index(x, y)]; };
    double best = INFINITY;
    int beste = 0x7fffffff;
    for (int e = tid; e < P.R * NPOSE; e += CTA_THREADS) {
        const int r = e >> 8, p = e & 255;
        const bool feas = (P.maskbits[((int64_t)env * P.R + r) * 8 + (p >> 5)] >> (p & 31)) & 1u;
        double s = HEUR_INVALID;
        if (feas) {
            const ShapeRot* sr = P.srot + (int64_t)item * P.R + r;
            const double z = P.posz[((int64_t)env * P.R + r) * NPOSE + p];
            s = heuristic_score(method, P.heur_dir, p >> 4, p & 15, z, P.resA, AX, AY, STEP, hm_at,
                                P.Ts + sr->off, sr->w, sr->h);
        }
        if (s < best) { best = s; beste = e; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double s2 = __shfl_xor_sync(0xffffffffu, best, o);
        const int e2 = __shfl_xor_sync(0xffffffffu, beste, o);
        if (s2 < best || (s2 == best && e2 < beste)) { best = s2; beste = e2; }
    }
    if (lane == 0) { best_sh[warp] = best; beste_sh[warp] = beste; }
    __syncthreads();
    best = best_sh[0]; beste = beste_sh[0];
#pragma unroll
    for (int k = 1; k < CTA_WARPS; ++k) {
        const double s2 = best_sh[k]; const int e2 = beste_sh[k];
        if (s2 < best || (s2 == best && e2 < beste)) { best = s2; beste = e2; }
    }
    const uint16_t* cand_g = P.cand + (int64_t)env * P.cand_stride;
    int first = 0x7fffffff;
    for (int i = tid; i < P.sel; i += CTA_THREADS)
        if ((int)cand_g[i] == beste) { first = i; break; }
    if (first != 0x7fffffff) atomicMin(&idx_sh, first);
    __syncthreads();
    if (tid == 0) {
        P.heur_pose[env * 3 + 0] = beste >> 8;
        P.heur_pose[env * 3 + 1] = (beste >> 4) & 15;
        P.heur_pose[env * 3 + 2] = beste & 15;
        P.heur_index[env] = (idx_sh == 0x7fffffff) ? -1 : idx_sh;
    }
}

// ---- candidates kernel ----------------------------------------------------------------------------------
// One CTA per ENVS_PER_CTA bins, one warp per bin in phase D.  In phase C every (bin, rotation, level)
// image of the CTA is one lane's task; the tasks are ordered by a cost key (number of border pixels) so
// that the lanes of a warp carry images of similar size -- the lanes run in lock step and a warp costs
// what its heaviest lane costs (the floor-level image of each rotation is an order of magnitude
// heavier than the small plateaus above it).
// Per-warp scratch of the candidates kernel, sized at run time (Params::ws_bytes, >= WS_MIN_BYTES): the first
// FAST_CAP * 32 bytes are the lane-strided contour points of phase C (also the 1024-point overflow
// buffers); in phase D the whole block holds the candidate list and its bucket-sorted index list, so its
// size grows with the rotation count (a bin can have up to R * 256 candidates).
constexpr int WS_MIN_BYTES = 4096;
static_assert(WS_MIN_BYTES >= 2 * BIG_CAP && WS_MIN_BYTES >= FAST_CAP * 32, "overflow buffers must fit the lane scratch");
constexpr int RANK_BUCKETS = 256;                        // height buckets of the phase-D truncation ranking (per warp: bases + cursors)
static_assert(RANK_BUCKETS % 32 == 0 && 32 * ROWS_WORDS >= 2 * RANK_BUCKETS, "phase D's rank histograms reuse the image slots (one warp's share each)");
// Phase D's candidate list + bucket-sorted entry list (2 x uint16 per candidate): up to R = 4 the warp scratch holds them for
// every pose of the bin (4 KB).  Beyond that a worst-case sized scratch would decide the residency (8 KB per warp at R = 8:
// 4 CTAs per SM in two waves, 12.7 warps active; 24 KB at R = 24: 2 CTAs), so the scratch stays at 4 KB, a bin whose
// candidates fit it (Ktot <= 1024, the usual case at R = 8) keeps its lists there and only a larger one spills to a global
// scratch (Params::dlist, L2 resident).  Measured: irregular R = 8  0.390 -> 0.370 ms per step, R = 24 unchanged.
#ifndef IRBPP_LISTS_SMEM_MAX_R
#define IRBPP_LISTS_SMEM_MAX_R 4
#endif
constexpr int LISTS_SMEM_MAX_R = IRBPP_LISTS_SMEM_MAX_R;
__host__ __device__ inline bool lists_in_smem(int R) { return R <= LISTS_SMEM_MAX_R; }
__host__ __device__ inline int ws_bytes_for(int R) {
    const int need = lists_in_smem(R) ? R * NPOSE * 4 : 0;     // uint16 list + uint16 sorted list for every pose
    return ((need > WS_MIN_BYTES ? need : WS_MIN_BYTES) + 15) & ~15;
}

template <int EPC>
struct CandSmem {
    static constexpr int ENVS_PER_CTA = EPC, CAND_WARPS = EPC, CAND_THREADS = 32 * EPC;
    uint32_t slots[CAND_THREADS * ROWS_WORDS];            // level images of this round in padded row form (one per thread)
    uint16_t task_tab[TASK_TAB];                          // micro-task m < TASK_TAB: slot << 8 | x << 4 | y of its start pixel
    int32_t pre[ENVS_PER_CTA * MAX_ROT + 1];              // prefix of level counts over (bin, rotation)
    int32_t cand_off[CAND_THREADS + 1];                   // prefix of start-candidate counts over the images, in cost order
    uint16_t slot_of[CAND_THREADS];                       // image slot at each position of the cost order
    uint16_t order2[CAND_THREADS * TASKS_PER_LANE];       // contour owner (task slot j * CAND_THREADS + thread) by decreasing contour length
    uint16_t q_of[CAND_THREADS * TASKS_PER_LANE];         // (bin, rotation) pair of a task slot's contour
    uint8_t n_of[CAND_THREADS * TASKS_PER_LANE];          // points of a task slot's contour (0: nothing to approximate)
    int32_t hist[64], hbase[64];
    uint16_t pair_of[CAND_THREADS];                       // (bin, rotation) pair of image t
    int32_t warp_tot[CAND_WARPS];
    int32_t error[ENVS_PER_CTA];
};

template <int EPC>
__global__ void __launch_bounds__(32 * EPC) irbpp_candidates_kernel(const Params P) {
    constexpr int ENVS_PER_CTA = EPC, CAND_WARPS = EPC, CAND_THREADS = 32 * EPC;     // one warp per bin
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CandSmem<EPC>& S = *reinterpret_cast<CandSmem<EPC>*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int env0 = P.env_lo + blockIdx.x * ENVS_PER_CTA;
    const int nenv = min(ENVS_PER_CTA, P.env_hi - env0);
    if (P.ready) {                                          // start when the scans of THIS CTA's bins are done (see ready_publish)
        if (tid < nenv) {
            const uint32_t* f = P.ready + env0 + tid;
            int polls = 0;
            while (ready_peek(f) != P.epoch) {
                if (++polls > READY_POLLS) { grid_dependency_wait(); break; }
                backoff();
            }
        }
        __syncthreads();
    } else {
        grid_dependency_wait();                             // PDL: scan grid complete, its scratch writes visible
    }
    const int R = P.R;
    const int npairs = nenv * R;
    long long t_prev = P.phase_cycles ? clock64() : 0;
    auto phase_mark = [&](int idx) {
        if (P.phase_cycles && tid == 0) {
            const long long now = clock64();
            atomicAdd(P.phase_cycles + idx, (unsigned long long)(now - t_prev));
            t_prev = now;
        }
    };
#ifdef IRBPP_PROBE_TRACE
    // profiling build only: per-CTA timeline (globaltimer, ns) in P.phase_cycles[8 + blockIdx.x * 8 + slot]
    auto trace = [&](int slot, unsigned long long v = ~0ull) {
        if (P.phase_cycles && tid == 0) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
            P.phase_cycles[8 + (size_t)blockIdx.x * 8 + slot] = (v == ~0ull) ? t : v;
        }
    };
    trace(0);
#else
    auto trace = [&](int, unsigned long long = 0ull) {};
#endif
    auto env_live = [&](int e) { return !(P.mode == MODE_RESET && P.which && !P.which[e]); };
    // the "bins" of this kernel are (bin, buffer slot) pairs in MODE_ALL_OBS (see the scan kernel): real bin, slot and
    // the place of a pair's rows in the observation
    const bool all_obs = (P.mode == MODE_ALL_OBS);
    auto real_env = [&](int e) { return all_obs ? e / P.K : e; };
    auto slot_of_e = [&](int e) { return all_obs ? e % P.K : 0; };
    auto obs_offset = [&](int e) { return (int64_t)real_env(e) * P.obs_stride + slot_of_e(e) * P.loc_len; };
    // Zero the candidate rows [first, sel) of one bin's observation (one warp): scalar stores up to a 16-byte
    // boundary, float4 after it.
    auto zero_obs_rows = [&](int e, int first) {
        float* z0 = P.obs + obs_offset(e) + first * 5;
        const int count = (P.sel - first) * 5;
        int head = (int)((16u - ((uint32_t)(uintptr_t)z0 & 15u)) & 15u) >> 2;
        head = head < count ? head : count;
        const int nvec = (count - head) >> 2;
        if (lane < head) z0[lane] = 0.0f;
        float4* zv = reinterpret_cast<float4*>(z0 + head);
        for (int i = lane; i < nvec; i += 32) zv[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        for (int i = head + 4 * nvec + lane; i < count; i += 32) z0[i] = 0.0f;
    };

    // dynamic tail: CAND_WARPS blocks of P.ws_bytes, then the 256-bit candidate sets per (bin, rotation)
    uint32_t* candbits = reinterpret_cast<uint32_t*>(smem_raw + ((sizeof(CandSmem<EPC>) + 15) & ~(size_t)15) + (size_t)CAND_WARPS * P.ws_bytes);
    for (int i = tid; i < ENVS_PER_CTA * R * 8; i += CAND_THREADS) candbits[i] = 0u;
    if (tid < ENVS_PER_CTA) S.error[tid] = 0;
    if (warp == 0) {   // prefix of the level counts over the (bin, rotation) pairs, 32 pairs per step
        int carry = 0;
        for (int b = 0; b < npairs; b += 32) {
            const int q = b + lane;
            int c = 0;
            if (q < npairs && env_live(env0 + q / R)) c = P.nlevels[(int64_t)env0 * R + q];
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int tt = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += tt; }
            if (q < npairs) S.pre[q + 1] = carry + incl;
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) S.pre[0] = 0;
    }
    __syncthreads();
    const int nimg = S.pre[npairs];
    trace(1);
    unsigned char* ws_base = smem_raw + ((sizeof(CandSmem<EPC>) + 15) & ~(size_t)15);     // CAND_WARPS blocks of P.ws_bytes
    uint8_t* W_pts = ws_base + (size_t)warp * P.ws_bytes;

    // ---- phase C: rounds of CAND_THREADS level images; inside a round one (image, start pixel) per lane ----
    for (int base = 0; base < nimg; base += CAND_THREADS) {
        const int nround = min(CAND_THREADS, nimg - base);
        // 1. thread t loads image t, counts its start candidates (background at W, NW, N, NE) and a cost key
        //    (foreground/background transitions ~ border length)
        int cnt = 0, bucket = 63, my_off = 0;
        uint32_t sm[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};   // start-pixel masks of this thread's image, two 16-bit rows per word
        if (tid < 64) S.hist[tid] = 0;
        __syncthreads();
        if (tid < nround) {
            const int t = base + tid;
            int lo = 0, hi = npairs;                        // pre[lo] <= t < pre[hi]
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (S.pre[mid] <= t) lo = mid; else hi = mid; }
            const uint4* src = reinterpret_cast<const uint4*>(
                P.bitmaps + (((int64_t)env0 * R + lo) * MAX_LEVELS + (t - S.pre[lo])) * 8);
            const uint4 a = src[0], b = src[1];
            uint32_t* rows = S.slots + tid * ROWS_WORDS;
            S.pair_of[tid] = (uint16_t)lo;
            const uint32_t wv[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
            rows[0] = 0u; rows[17] = 0u;
#pragma unroll
            for (int k = 0; k < 8; ++k) { rows[1 + 2 * k] = (wv[k] & 0xFFFFu) << 1; rows[2 + 2 * k] = (wv[k] >> 16) << 1; }
            uint32_t up = 0;
            int key = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t r0 = wv[k] & 0xFFFFu, r1 = wv[k] >> 16;
                sm[k] = start_mask(r0, up) | (start_mask(r1, r0) << 16);
                cnt += __popc(sm[k]);
                key += __popc(r0 ^ (r0 << 1)) + __popc(r1 ^ (r1 << 1)) + __popc(r0 ^ up) + __popc(r1 ^ r0);
                up = r1;
            }
            bucket = 63 - min(63, key >> 2);                // bucket 0 = longest borders
            my_off = atomicAdd(&S.hist[bucket], 1);
        }
        __syncthreads();
        if (warp == 0) {   // exclusive prefix over the 64 buckets
            const int h0 = S.hist[lane], h1 = S.hist[32 + lane];
            int i0 = h0, i1 = h1;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t0 = __shfl_up_sync(0xffffffffu, i0, o), t1 = __shfl_up_sync(0xffffffffu, i1, o);
                if (lane >= o) { i0 += t0; i1 += t1; }
            }
            const int tot0 = __shfl_sync(0xffffffffu, i0, 31);
            S.hbase[lane] = i0 - h0;
            S.hbase[32 + lane] = tot0 + i1 - h1;
        }
        __syncthreads();
        // position in cost order -> (slot, count); cand_off[] temporarily holds the counts
        int my_pos = 0;
        if (tid < nround) {
            my_pos = S.hbase[bucket] + my_off;
            S.slot_of[my_pos] = (uint16_t)tid;
            S.cand_off[my_pos + 1] = cnt;
        }
        for (int i = nround + tid; i < CAND_THREADS; i += CAND_THREADS) S.cand_off[i + 1] = 0;
        __syncthreads();
        {   // CTA-wide inclusive prefix of the counts in cost order
            const int c = S.cand_off[tid + 1];
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int tt = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += tt; }
            if (lane == 31) S.warp_tot[warp] = incl;
            __syncthreads();
            int wbase = 0;
            for (int w2 = 0; w2 < warp; ++w2) wbase += S.warp_tot[w2];
            S.cand_off[tid + 1] = wbase + incl;
            if (tid == 0) S.cand_off[0] = 0;
        }
        __syncthreads();
        const int ntask = S.cand_off[CAND_THREADS];
        // every image lists its start pixels (raster order) at its offset of the task table, so that a
        // micro-task lane finds its pixel with one load
        if (tid < nround && cnt > 0) {
            int off = S.cand_off[my_pos];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                uint32_t c = sm[k];
                while (c && off < TASK_TAB) {
                    const int b = __ffs((int)c) - 1;           // bit b: column b & 15 of row 2k + (b >> 4)
                    c &= c - 1;
                    S.task_tab[off++] = (uint16_t)((tid << 8) | ((b & 15) << 4) | (2 * k + (b >> 4)));
                }
            }
        }
        __syncthreads();
        if (base == 0) trace(2);
#ifdef IRBPP_PROBE_FINE
        phase_mark(4);   // prologue, image loads, cost sort, start-pixel prefix
#else
        if (P.phase_cycles && tid == 0) { atomicAdd(P.phase_cycles + 4, (unsigned long long)nround); atomicAdd(P.phase_cycles + 5, (unsigned long long)ntask); atomicAdd(P.phase_cycles + 6, 1ull); }
#endif

        // 2. micro-tasks: one (image, start pixel) pair each, TASKS_PER_LANE per lane and batch.  The tasks are in cost
        //    order, so task slot 0 of the lanes holds the 128 most expensive ones (64-point scratch), slots 1 and 2 the
        //    cheap rest (32-point scratch): one follow / sort / approximate cycle with its five block barriers serves
        //    up to 384 tasks -- a 4-bin CTA of the bench workload has ~170 (profiles/: per-CTA timelines showed the
        //    second and third cycle of the one-task-per-lane form costing 7.5 us of a 43 us CTA, 30 us in the worst)
        constexpr int TPL = TASKS_PER_LANE;
        constexpr int BATCH = CAND_THREADS * TPL;
        static_assert(FAST_CAP * 32 + (TPL - 1) * 32 * 32 <= WS_MIN_BYTES, "the task slots' point buffers share the warp scratch");
        // points per contour in task slots 1, 2: what the warp scratch holds beside slot 0's 64-point buffers -- 32 at
        // R <= 4 (4 KB per warp), 64 from R = 8 on (the scratch grows with R for phase D's lists), where long contours
        // in the cheaper slots are not rare and every overflow is a serial redo
        const int cap12 = min(FAST_CAP, (P.ws_bytes - FAST_CAP * 32) / ((TPL > 1 ? TPL - 1 : 1) * 32));
        auto slot_scratch = [&](int owner) {               // point buffer of task slot `owner` (j * CAND_THREADS + thread)
            const int jj = owner / CAND_THREADS, th = owner - jj * CAND_THREADS;
            return ws_base + (size_t)(th >> 5) * P.ws_bytes + (jj == 0 ? 0 : FAST_CAP * 32 + (jj - 1) * cap12 * 32) + (th & 31);
        };
        for (int mb = 0; mb < ntask; mb += BATCH) {
            int tk[TPL];                                    // slot << 8 | x << 4 | y of my tasks, -1: none
            int npts_j[TPL];
            uint32_t ovf_bits = 0;
#pragma unroll
            for (int jt = 0; jt < TPL; ++jt) {
                const int m = mb + jt * CAND_THREADS + tid;
                const bool has = m < ntask;
                int slot = 0, x = 0, y = 0;
                if (has && m < TASK_TAB) {
                    const int t = S.task_tab[m];
                    slot = t >> 8; x = (t >> 4) & 15; y = t & 15;
                } else if (has) {                               // beyond the table: search the prefix and the image
                    int lo = 0, hi = CAND_THREADS;              // cand_off[lo] <= m < cand_off[hi]
                    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (S.cand_off[mid] <= m) lo = mid; else hi = mid; }
                    slot = S.slot_of[lo];
                    int k = m - S.cand_off[lo];
                    const uint32_t* ri = S.slots + slot * ROWS_WORDS;
                    for (y = 0; y < 16; ++y) {
                        const uint32_t c = start_candidates_rows(ri, y);
                        const int pc = __popc(c);
                        if (k < pc) { x = (int)__fns(c, 0u, k + 1); break; }
                        k -= pc;
                    }
                }
                tk[jt] = has ? ((slot << 8) | (x << 4) | y) : -1;
                // (a) the lane follows the border; the points stay in the task slot's scratch
                int n = -2, area2 = 1;
                if (has) {
                    StridedScratch<32, FAST_CAP> sc;
                    sc.b = slot_scratch(jt * CAND_THREADS + tid);
                    sc.kept = 0;
                    n = follow_outer_rows(sc, S.slots + slot * ROWS_WORDS, x, y, area2, jt == 0 ? FAST_CAP : cap12);
                }
                const bool keep = has && n != -2 && area2 <= 0;        // a raster-first start of an outer border
                if (keep && n < 0) ovf_bits |= 1u << jt;
                npts_j[jt] = (keep && n > 0) ? n : 0;
            }
            // (b) the contours of the CTA are re-dealt in decreasing length, so that the approximation loops
            //     of a warp have similar trip counts and abandoned / hole paths drop out
            if (tid < 64) S.hist[tid] = 0;
            __syncthreads();
            if (base == 0 && mb == 0) trace(3);
#ifdef IRBPP_PROBE_FINE
            phase_mark(5);   // find start pixel + follow (incl. waiting for the slowest warp)
#endif
            int boff[TPL];
#pragma unroll
            for (int jt = 0; jt < TPL; ++jt) {
                boff[jt] = atomicAdd(&S.hist[63 - min(63, npts_j[jt])], 1);
                S.n_of[jt * CAND_THREADS + tid] = (uint8_t)npts_j[jt];
                S.q_of[jt * CAND_THREADS + tid] = (uint16_t)(tk[jt] >= 0 ? S.pair_of[tk[jt] >> 8] : 0);
            }
            __syncthreads();
            if (warp == 0) {   // exclusive prefix over the 64 buckets
                const int h0 = S.hist[lane], h1 = S.hist[32 + lane];
                int i0 = h0, i1 = h1;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t0 = __shfl_up_sync(0xffffffffu, i0, o), t1 = __shfl_up_sync(0xffffffffu, i1, o);
                    if (lane >= o) { i0 += t0; i1 += t1; }
                }
                const int tot0 = __shfl_sync(0xffffffffu, i0, 31);
                S.hbase[lane] = i0 - h0;
                S.hbase[32 + lane] = tot0 + i1 - h1;
            }
            __syncthreads();
#pragma unroll
            for (int jt = 0; jt < TPL; ++jt)
                S.order2[S.hbase[63 - min(63, npts_j[jt])] + boff[jt]] = (uint16_t)(jt * CAND_THREADS + tid);
            __syncthreads();
#ifdef IRBPP_PROBE_FINE
            phase_mark(6);   // length sort
#endif
            // (c) lane i approximates the contours of rank i, 128 + i, 256 + i (points live in their owners' scratch)
#pragma unroll 1
            for (int jt = 0; jt < TPL; ++jt) {
                const int owner = S.order2[jt * CAND_THREADS + tid];
                const int on = S.n_of[owner];
                if (on > 0) {
                    StridedScratch<32, FAST_CAP> sc;
                    sc.b = slot_scratch(owner);
                    sc.kept = 0;
                    uint32_t* cb = candbits + (int)S.q_of[owner] * 8;
                    approx_and_emit(sc, on, P.legacy != 0,
                                    [&](int ex, int ey) { const int b = ex * 16 + ey; atomicOr(cb + (b >> 5), 1u << (b & 31)); });
                }
            }
            __syncthreads();           // scratch of every lane is free again
            if (base == 0 && mb == 0) { trace(4); int mx = 0; for (int i = 0; i < BATCH; ++i) mx = max(mx, (int)S.n_of[i]); trace(7, ((unsigned long long)ntask << 8) | (unsigned long long)mx); }
#ifdef IRBPP_PROBE_FINE
            phase_mark(7);   // approxPolyDP + emit
#endif
            // rare: a contour longer than its slot's buffer; the lanes concerned redo it one at a time with
            // 1024-point buffers laid over the (now idle) scratch of this warp
#pragma unroll 1
            for (int jt = 0; jt < TPL; ++jt) {
                uint32_t ovf = __ballot_sync(0xffffffffu, (ovf_bits >> jt) & 1u);
                while (ovf) {
                    const int src_lane = __ffs((int)ovf) - 1;
                    ovf &= ovf - 1;
                    if (lane == src_lane) {
#ifndef IRBPP_PROBE_FINE
                        if (P.phase_cycles) atomicAdd(P.phase_cycles + 7, 1ull);     // overflow redo counter
#endif
                        FlatScratch<BIG_CAP> bs;
                        bs.b = W_pts;
                        const int slot = tk[jt] >> 8, q = S.pair_of[slot];
                        uint32_t* cb = candbits + q * 8;
                        if (!process_start_candidate(bs, S.slots + slot * ROWS_WORDS, (tk[jt] >> 4) & 15, tk[jt] & 15, P.legacy != 0,
                                [&](int ex, int ey) { const int b = ex * 16 + ey; atomicOr(cb + (b >> 5), 1u << (b & 31)); }))
                            atomicMax(&S.error[q / R], 6);
                    }
                    __syncwarp();
                }
            }
            __syncthreads();
        }
        __syncthreads();
    }
    __syncthreads();
    trace(5);
    phase_mark(2);   // contour tasks
    // the scan grid has long completed; waiting for it formally keeps the stream-order guarantee of a dependent launch
    // (this grid does not complete before its prerequisite) without delaying the start
    if (P.ready && tid == 0) grid_dependency_wait();

    // ---- phase D: warp w serves bin env0 + w ----
    if (warp >= nenv) return;
    const int env = env0 + warp;
    if (!env_live(env)) return;
    const int dev_err = S.error[warp];
    // ---- phase D ----
    const int sel = P.sel;
    const uint32_t* cbits = candbits + warp * R * 8;
    const uint32_t* mask_g = P.maskbits + (int64_t)env * R * 8;
    const double* posz_g = P.posz + (int64_t)env * R * NPOSE;
    const int renv = real_env(env);
    float* obs_g = P.obs + obs_offset(env);
    const bool write_state = (P.mode == MODE_STEP || P.mode == MODE_RESET || P.mode == MODE_CANDIDATES ||
                              (all_obs && slot_of_e(env) == P.K - 1));
    uint16_t* cand_g = write_state ? P.cand + (int64_t)renv * P.cand_stride : nullptr;
    double* dbg_cand = P.dbg_cand ? P.dbg_cand + (int64_t)env * sel * 5 : nullptr;

    // candidate counts per rotation (lane r), exclusive prefix, total
    int cnt = 0;
    if (lane < R) { for (int qd = 0; qd < 8; ++qd) cnt += __popc(cbits[lane * 8 + qd]); }
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int tt = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += tt; }
    const int excl = incl - cnt;
    const int Ktot = __shfl_sync(0xffffffffu, incl, 31);
    uint32_t anym = 0;
    for (int qd = lane; qd < R * 8; qd += 32) anym |= mask_g[qd];
    anym = __reduce_or_sync(0xffffffffu, anym);

    auto put_row = [&](int row, int rot, int x, int y, double H, double V) {
        float* d = obs_g + row * 5;
        d[0] = (float)rot; d[1] = (float)x; d[2] = (float)y; d[3] = (float)H; d[4] = (float)V;
        if (cand_g) cand_g[row] = (uint16_t)((rot << 8) | (x << 4) | y);
        if (dbg_cand) { double* qd = dbg_cand + row * 5; qd[0] = rot; qd[1] = x; qd[2] = y; qd[3] = H; qd[4] = V; }
    };
    auto zero_rows = [&](int first) {
        zero_obs_rows(env, first);
        if (cand_g) for (int i = first + lane; i < sel; i += 32) cand_g[i] = 0;
        if (dbg_cand) for (int i = first * 5 + lane; i < sel * 5; i += 32) dbg_cand[i] = 0.0;
    };
    auto height_of = [&](int cell, bool& m) -> double {     // posZValid at a flat pose index
        m = (mask_g[cell >> 5] >> (cell & 31)) & 1u;
        return m ? posz_g[cell] : POSZ_INVALID;
    };

    if (Ktot == 0) {
        // no hull candidate at all (binPhy.py:217-225): the `sel` smallest posZValid, stable order
        const int total = R * NPOSE;
        if (!anym) {
            const int nrow = total < sel ? total : sel;
            for (int i = lane; i < nrow; i += 32) put_row(i, i >> 8, (i >> 4) & 15, i & 15, P.binz, 0.0);
            zero_rows(nrow);
        } else {
            for (int i = lane; i < total; i += 32) {
                bool mi; const double vi = height_of(i, mi);
                int rank = 0;
                for (int j = 0; j < total; ++j) {
                    bool mj; const double vj = height_of(j, mj);
                    rank += (vj < vi) || (vj == vi && j < i);
                }
                if (rank < sel) put_row(rank, i >> 8, (i >> 4) & 15, i & 15, P.binz, mi ? 1.0 : 0.0);
            }
            zero_rows(total < sel ? total : sel);
        }
    } else {
        // rows in rotation order, then (col, row) ascending == bit order of the per-rotation sets.
        // Pass 1 compacts the set bits into a list (no memory loads); pass 2 gives every lane one
        // candidate, so the height gathers of 32 candidates are in flight together.
        // candidate list + bucket-sorted index list: the (now idle) lane scratch, or the pair's slice of the global scratch
        // (a bin whose candidates fit the warp scratch keeps its lists there even when the global scratch exists)
        const bool spill = P.dlist && Ktot > P.ws_bytes / 4;
        const int LIST_CAP = spill ? R * NPOSE : P.ws_bytes / 4;      // >= Ktot
        uint16_t* list = spill ? P.dlist + (int64_t)env * 2 * (R * NPOSE) : reinterpret_cast<uint16_t*>(W_pts);
        auto cell_of = [](int e) { const int b = e & 255; return (e >> 8) * NPOSE + (b & 15) * 16 + (b >> 4); };
        {
            for (int r = 0; r < R; ++r) {
                const uint32_t* cb = cbits + r * 8;
                int ord0 = __shfl_sync(0xffffffffu, excl, r);
#pragma unroll
                for (int qd = 0; qd < 8; ++qd) {
                    const uint32_t wbits = cb[qd];
                    if ((wbits >> lane) & 1u)
                        list[ord0 + __popc(wbits & ((1u << lane) - 1u))] = (uint16_t)((r << 8) | (qd * 32 + lane));
                    ord0 += __popc(wbits);
                }
            }
            __syncwarp();
            if (Ktot <= sel) {
                for (int i = lane; i < Ktot; i += 32) {
                    const int e = list[i];
                    const int b = e & 255;
                    bool m; const double H = height_of(cell_of(e), m);
                    put_row(i, e >> 8, b & 15, b >> 4, H, m ? 1.0 : 0.0);
                }
            } else {
                // More candidates than rows: keep the `sel` lowest heights, ties by original order (stable
                // argsort; binPhy.py:209-212).  Exact ranks without a full sort: the feasible candidates are
                // bucketed by a monotone map of their height (256 buckets over [min, max] of this bin), a
                // candidate's rank = (candidates in lower buckets) + (its rank inside its own bucket), so it is
                // compared only with its bucket; the infeasible ones all carry POSZ_INVALID, i.e. they follow the
                // feasible ones in list order, which a running ballot count gives directly.  List entries grow
                // with the list index, so "earlier in the list" is a comparison of the entries themselves.
                uint16_t* sorted = list + LIST_CAP;                  // second half of the scratch: entries grouped by bucket
                int32_t* hist = reinterpret_cast<int32_t*>(S.slots) + warp * (2 * RANK_BUCKETS);   // image slots are idle now
                double hmin = POSZ_INVALID, hmax = -POSZ_INVALID;
                int nvalid = 0;
                for (int i = lane; i < Ktot; i += 32) {
                    bool m; const double H = height_of(cell_of(list[i]), m);
                    if (m) { hmin = fmin(hmin, H); hmax = fmax(hmax, H); ++nvalid; }
                }
#pragma unroll
                for (int o = 16; o; o >>= 1) {
                    hmin = fmin(hmin, __shfl_xor_sync(0xffffffffu, hmin, o));
                    hmax = fmax(hmax, __shfl_xor_sync(0xffffffffu, hmax, o));
                    nvalid += __shfl_xor_sync(0xffffffffu, nvalid, o);
                }
                const double scale = hmax > hmin ? (double)RANK_BUCKETS / (hmax - hmin) : 0.0;
                auto bucket_of = [&](double H) { const int v = (int)((H - hmin) * scale); return v > RANK_BUCKETS - 1 ? RANK_BUCKETS - 1 : v; };
                for (int b = lane; b < RANK_BUCKETS; b += 32) hist[b] = 0;
                __syncwarp();
                for (int i = lane; i < Ktot; i += 32) {
                    bool m; const double H = height_of(cell_of(list[i]), m);
                    if (m) atomicAdd(&hist[bucket_of(H)], 1);
                }
                __syncwarp();
                {   // exclusive prefix over the buckets: lane l owns buckets [l * BPL, (l + 1) * BPL)
                    constexpr int BPL = RANK_BUCKETS / 32;
                    int c[BPL], tot = 0;
#pragma unroll
                    for (int q = 0; q < BPL; ++q) { c[q] = hist[lane * BPL + q]; tot += c[q]; }
                    int inc = tot;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) { const int t0 = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t0; }
                    int base = inc - tot;
                    __syncwarp();
#pragma unroll
                    for (int q = 0; q < BPL; ++q) {
                        hist[lane * BPL + q] = base;                          // bucket bases
                        hist[RANK_BUCKETS + lane * BPL + q] = base;           // fill cursors
                        base += c[q];
                    }
                }
                __syncwarp();
                for (int i = lane; i < Ktot; i += 32) {
                    const int e = list[i];
                    bool m; const double H = height_of(cell_of(e), m);
                    if (m) sorted[atomicAdd(&hist[RANK_BUCKETS + bucket_of(H)], 1)] = (uint16_t)e;
                }
                __syncwarp();
                int inv_before = 0;                                  // infeasible candidates in earlier trips
                for (int i0 = 0; i0 < Ktot; i0 += 32) {
                    const int i = i0 + lane;
                    const int e = i < Ktot ? list[i] : 0;
                    const int b = e & 255;
                    bool m = false; double H = 0.0;
                    if (i < Ktot) H = height_of(cell_of(e), m);
                    const uint32_t inv = __ballot_sync(0xffffffffu, i < Ktot && !m);
                    if (i < Ktot && m) {
                        const int bk = bucket_of(H);
                        const int lo = hist[bk], hi = hist[RANK_BUCKETS + bk];   // this bucket's segment of `sorted`
                        if (lo < sel) {                                  // else everything in it ranks beyond the table
                            int rank = lo;
                            for (int t = lo; t < hi; ++t) {
                                const int e2 = sorted[t];
                                const double H2 = posz_g[cell_of(e2)];
                                rank += (H2 < H) || (H2 == H && e2 < e);
                            }
                            if (rank < sel) put_row(rank, e >> 8, b & 15, b >> 4, H, 1.0);
                        }
                    } else if (i < Ktot) {
                        const int rank = nvalid + inv_before + __popc(inv & ((1u << lane) - 1u));
                        if (rank < sel) put_row(rank, e >> 8, b & 15, b >> 4, H, 0.0);
                    }
                    inv_before += __popc(inv);
                }
            }
        }
        if (Ktot < sel) zero_rows(Ktot);
    }
    if (lane == 0) {
        if (dev_err) store_error(P, renv, (uint8_t)dev_err);
        if (P.dbg_nhull) P.dbg_nhull[env] = Ktot;
    }
    if (warp == 0) trace(6);
    phase_mark(3);   // select / pad, candidate rows of the observation
}

}  // namespace irbpp
