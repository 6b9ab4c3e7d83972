// irbpp.cu -- C-ABI (include/irbpp.h) host side: state ownership, table preprocessing, launches.
//
// No CPU fallback lives here: every entry point that computes anything launches the CUDA kernels of
// irbpp_kernels.cuh (irbpp_scan_kernel -> irbpp_candidates_kernel).
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <cmath>
#include <string>
#include <vector>

#include "../../include/irbpp.h"
#include "irbpp_kernels.cuh"
#include "irbpp_pointnet.cuh"
#include "irbpp_pack.cuh"
#include "irbpp_replay.cuh"

using namespace irbpp;

static thread_local std::string g_create_error;     // error of the calling thread's last failed irbpp_create

struct irbpp_env {
    irbpp_config cfg;
    Params P;                      // device pointers + configuration (mode/inputs filled per launch)
    int cand_smem = 0, scan_smem = 0;
    uint32_t* ready_dev = nullptr;       // scan -> candidates hand-over flags (one per unit)
    uint32_t epoch = 0;                  // launch counter behind the flags
    int epc = ENVS_PER_CTA_NARROW;       // bins per CTA of the candidates kernel (envs_per_cta_for(R))
    std::string err;
    bool shapes_loaded = false, sequences_set = false, was_reset = false, waiting_step = false;
    bool scan_current = false;        // the scan scratch holds the drop heights of every bin's cur_item
    int32_t* heur_pose_dev = nullptr; int64_t* heur_index_dev = nullptr;
    bool results_on_host = false;           // the pending step wrote its results straight to the host mirror
    cudaStream_t pending_stream = nullptr;
    int64_t launches = 0;
    // device allocations
    std::vector<void*> dev_allocs;
    void* results_dev = nullptr;            // the device result block (carve_results)
    void* results_host[2] = {nullptr, nullptr};   // pinned mirrors; the current step's is results_host[res_turn]: the blocks
                                                  // alternate, so the views of step k stay valid until step k + 2 is launched
    StepResults results_mapped[2] = {};     // device views of results_host[]
    int res_turn = 0;
    size_t results_bytes = 0;
    int64_t* actions_dev = nullptr;
    int64_t* actions_pinned = nullptr;      // [2][N] pinned staging: step actions, order actions
    uint8_t* which_dev = nullptr;
    // shape pools
    ShapeRot* srot_dev = nullptr; double* Bs_dev = nullptr; double* Ts_dev = nullptr;
    double* vol_dev = nullptr; double* rew_dev = nullptr; int32_t* seq_dev = nullptr;
    TileEntry* tiles_dev = nullptr;
    unsigned long long* phase_dev = nullptr;
};

// Every entry point runs on its handle's device and leaves the calling thread's current device as it found it: the
// host framework (torch) tracks the current device itself, and a library that changes it behind its back makes the
// caller's next `tensor.cuda()` land on another GPU (seen in a two-device test before this guard existed).
struct DeviceGuard {
    int prev = -1, cur = -1;
    explicit DeviceGuard(int dev) : cur(dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() { if (prev >= 0 && prev != cur) cudaSetDevice(prev); }
};

// device that owns a device pointer (the handle-free entry points run where their buffers live)
static int device_of(const void* p) {
#ifdef IRBPP_HOST_EMULATION
    (void)p; return 0;
#else
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeDevice) return at.device;
    cudaGetLastError();
    int d = 0; cudaGetDevice(&d); return d;
#endif
}

static int fail(irbpp_env* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define CUDA_TRY(h, expr)                                                                         \
    do {                                                                                          \
        cudaError_t e_ = (expr);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return fail(h, IRBPP_ECUDA, "%s failed: %s", #expr, cudaGetErrorString(e_));          \
    } while (0)

template <class T>
static cudaError_t dev_alloc(irbpp_env* h, T** p, size_t count, bool zero = true) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 16);
    if (e != cudaSuccess) return e;
    if (zero) { e = cudaMemset(q, 0, count * sizeof(T) + 16); if (e != cudaSuccess) return e; }
    h->dev_allocs.push_back(q);
    *p = reinterpret_cast<T*>(q);
    return cudaSuccess;
}


static void free_dev(irbpp_env* h, void* p) {
    if (!p) return;
    auto it = std::find(h->dev_allocs.begin(), h->dev_allocs.end(), p);
    if (it != h->dev_allocs.end()) h->dev_allocs.erase(it);
    cudaFree(p);
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-function, PER-DEVICE attribute: the largest value any
// handle needed is tracked per device ordinal and only ever raised (several handles may coexist on a device,
// and one process may hold handles on several devices).  which: 0 / 3 candidates kernel (narrow / wide CTA), 1 scan kernel, 2 shape encoder.
static cudaError_t raise_dynamic_smem(int device, int which, int bytes) {
    static int raised[64][4];
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    if (device < 0 || device >= 64) return cudaErrorInvalidDevice;
    if (bytes <= raised[device][which]) return cudaSuccess;
    cudaError_t e = which == 0
        ? cudaFuncSetAttribute(irbpp_candidates_kernel<ENVS_PER_CTA_NARROW>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)
        : which == 3
        ? cudaFuncSetAttribute(irbpp_candidates_kernel<ENVS_PER_CTA_WIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)
        : (which == 1 ? cudaFuncSetAttribute(irbpp_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)
                      : cudaFuncSetAttribute(irbpp_shape_encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    if (e == cudaSuccess) raised[device][which] = bytes;
    return e;
}

extern "C" {

int irbpp_abi_version(void) { return IRBPP_ABI_VERSION; }

const char* irbpp_last_error(irbpp_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int irbpp_create(const irbpp_config* cfg, irbpp_handle* out) {
    if (!cfg || !out) return fail(nullptr, IRBPP_EINVAL, "null argument");
    *out = nullptr;
    if (cfg->num_envs <= 0) return fail(nullptr, IRBPP_EINVAL, "num_envs must be positive");
    if (cfg->num_rotations < 1 || cfg->num_rotations > 32)
        return fail(nullptr, IRBPP_EINVAL, "num_rotations must be in [1, 32]");
    if (cfg->buffer_size < 1 || cfg->buffer_size > MAX_QUEUE)
        return fail(nullptr, IRBPP_EINVAL, "buffer_size must be in [1, %d]", MAX_QUEUE);
    if (cfg->selected_action < 1 || cfg->selected_action > 4096)
        return fail(nullptr, IRBPP_EINVAL, "selected_action must be in [1, 4096]");
    // grid sizes exactly as Space.__init__ computes them (space.py:19-24)
    const double stepf = cfg->resolution_act / cfg->resolution_h;
    const int step = (int)stepf;
    const int hx = (int)ceil(cfg->bin_dimension[0] / cfg->resolution_h), hy = (int)ceil(cfg->bin_dimension[1] / cfg->resolution_h);
    const int ax = (int)ceil(cfg->bin_dimension[0] / cfg->resolution_act), ay = (int)ceil(cfg->bin_dimension[1] / cfg->resolution_act);
    if ((double)step != stepf || step != STEP || hx != HX || hy != HY || ax != AX || ay != AY)
        return fail(nullptr, IRBPP_EINVAL,
                    "unsupported grid: heightmap %dx%d, actions %dx%d, step %g (this build: %dx%d, %dx%d, %d)",
                    hx, hy, ax, ay, stepf, HX, HY, AX, AY, STEP);
    if (cfg->selected_action > cfg->num_rotations * NPOSE)
        return fail(nullptr, IRBPP_EINVAL, "selected_action exceeds the number of poses (reference fallback "
                                           "binPhy.py:217-225 would return a short table)");
    if (!(cfg->resolution_z > 0) || ceil(cfg->bin_dimension[2] / cfg->resolution_z) + 1 >= LEVEL_OFFSET)
        return fail(nullptr, IRBPP_EINVAL, "bin height / resolution_z must stay below %d levels", LEVEL_OFFSET - 1);

    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, IRBPP_ECUDA, "no CUDA device (%s); this library has no CPU path",
                    e == cudaSuccess ? "count 0" : cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, IRBPP_EINVAL, "bad device ordinal %d", cfg->device);
    DeviceGuard guard(cfg->device);
    {
        int now = -1;
        if (cudaGetDevice(&now) != cudaSuccess || now != cfg->device) return fail(nullptr, IRBPP_ECUDA, "cudaSetDevice(%d) failed", cfg->device);
    }

    irbpp_env* h = new irbpp_env();
    h->cfg = *cfg;
    Params& P = h->P;
    memset(&P, 0, sizeof(P));
    const int N = cfg->num_envs;
    P.N = N; P.R = cfg->num_rotations; P.sel = cfg->selected_action; P.K = cfg->buffer_size;
    P.loc_len = P.sel * 5 + 9 + HX * HY;
    P.order_len = P.K + HX * HY;
    P.obs_stride = (P.K > 1) ? P.order_len : P.loc_len;
    P.legacy = cfg->approx_legacy;
    P.binz = cfg->bin_dimension[2];
    P.resZ = cfg->resolution_z;
    P.resA = cfg->resolution_act;
    P.binvol = (cfg->bin_dimension[0] * cfg->bin_dimension[1]) * cfg->bin_dimension[2];   // np.prod
    P.ws_bytes = ws_bytes_for(P.R);
    h->epc = envs_per_cta_for(P.R);                  // bins (= warps) per CTA of the candidates kernel
    {
        const size_t fixed = h->epc == ENVS_PER_CTA_WIDE ? sizeof(CandSmem<ENVS_PER_CTA_WIDE>) : sizeof(CandSmem<ENVS_PER_CTA_NARROW>);
        h->cand_smem = (int)((fixed + 15) & ~(size_t)15) + h->epc * P.ws_bytes + h->epc * P.R * 8 * 4;
    }

#define TRY_ALLOC(expr)                                                                          \
    do { cudaError_t e2_ = (expr); if (e2_ != cudaSuccess) {                                      \
        fail(nullptr, IRBPP_ECUDA, "%s: %s", #expr, cudaGetErrorString(e2_)); irbpp_destroy(h); return IRBPP_ECUDA; } } while (0)
    TRY_ALLOC(dev_alloc(h, &P.hm, (size_t)N * HX * HY));
    P.cand_stride = (P.sel + 7) & ~7;                 // rows of whole 16-byte units: the scan kernel bulk-copies them
    TRY_ALLOC(dev_alloc(h, &P.cand, (size_t)N * P.cand_stride));
    TRY_ALLOC(dev_alloc(h, &P.state, (size_t)N));
    TRY_ALLOC(dev_alloc(h, &h->actions_dev, N)); TRY_ALLOC(dev_alloc(h, &h->which_dev, N));
    // scan -> candidates hand-over scratch
    // (buffered: one slice per (bin, buffer slot) pair, get_all_possible_observation scans all of them at once)
    const size_t units = (size_t)N * (size_t)P.K;
    TRY_ALLOC(dev_alloc(h, &P.posz, units * P.R * NPOSE));
    TRY_ALLOC(dev_alloc(h, &P.maskbits, units * P.R * 8));
    TRY_ALLOC(dev_alloc(h, &P.bitmaps, units * P.R * MAX_LEVELS * 8));
    TRY_ALLOC(dev_alloc(h, &P.nlevels, units * P.R));
    if (!lists_in_smem(P.R)) TRY_ALLOC(dev_alloc(h, &P.dlist, units * 2 * P.R * NPOSE));
    TRY_ALLOC(dev_alloc(h, &h->ready_dev, units));        // zeroed: no launch has epoch 0
    h->results_bytes = (size_t)N * RESULT_BYTES_PER_BIN;
    TRY_ALLOC(cudaMalloc(&h->results_dev, h->results_bytes + 64));
    TRY_ALLOC(cudaMemset(h->results_dev, 0, h->results_bytes + 64));
    P.res = carve_results(h->results_dev, N);
    for (int t = 0; t < 2; ++t) {
        void* mapped = nullptr;
        TRY_ALLOC(cudaHostAlloc(&h->results_host[t], h->results_bytes + 64, cudaHostAllocMapped));
        TRY_ALLOC(cudaHostGetDevicePointer(&mapped, h->results_host[t], 0));
        memset(h->results_host[t], 0, h->results_bytes + 64);
        h->results_mapped[t] = carve_results(mapped, N);
    }
    TRY_ALLOC(cudaHostAlloc((void**)&h->actions_pinned, 2 * (size_t)N * sizeof(int64_t), cudaHostAllocMapped));
    TRY_ALLOC(raise_dynamic_smem(cfg->device, h->epc == ENVS_PER_CTA_WIDE ? 3 : 0, h->cand_smem));
#undef TRY_ALLOC
    *out = h;
    return IRBPP_OK;
}

int irbpp_destroy(irbpp_handle h) {
    if (!h) return IRBPP_OK;
    DeviceGuard guard(h->cfg.device);
    cudaDeviceSynchronize();
    for (void* p : h->dev_allocs) cudaFree(p);
    if (h->results_dev) cudaFree(h->results_dev);
    for (int t = 0; t < 2; ++t) if (h->results_host[t]) cudaFreeHost(h->results_host[t]);
    if (h->actions_pinned) cudaFreeHost(h->actions_pinned);
    delete h;
    return IRBPP_OK;
}

int irbpp_obs_len(irbpp_handle h, int32_t* obs_len, int32_t* loc_obs_len, int32_t* order_obs_len) {
    if (!h) return IRBPP_EINVAL;
    if (obs_len) *obs_len = h->P.obs_stride;
    if (loc_obs_len) *loc_obs_len = h->P.loc_len;
    if (order_obs_len) *order_obs_len = h->P.order_len;
    return IRBPP_OK;
}

int irbpp_load_shapes(irbpp_handle h, int32_t S, int32_t R, const int32_t* dims, const double* ext,
                      const double* vol, const double* maps, const int64_t* offsets, int64_t maps_len) {
    if (!h || !dims || !ext || !vol || !maps || !offsets) return fail(h, IRBPP_EINVAL, "null argument");
    if (R != h->P.R) return fail(h, IRBPP_EINVAL, "library has %d rotations, env configured for %d", R, h->P.R);
    if (S <= 0) return fail(h, IRBPP_EINVAL, "empty shape library");
    const irbpp_config& c = h->cfg;
    std::vector<ShapeRot> srot((size_t)S * R);
    std::vector<double> Bs, Ts;
    std::vector<TileEntry> tiles;
    std::vector<double> rew(S);
    int maxwh = 1, max_entries = 1;
    for (int s = 0; s < S; ++s) {
        rew[s] = (vol[s] / h->P.binvol) * 10;                        // binPhy.py:155-156,321-322
        for (int r = 0; r < R; ++r) {
            const int32_t* d = dims + ((size_t)s * R + r) * 4;
            const double* e = ext + ((size_t)s * R + r) * 3;
            const int w = d[0], hh = d[1], wA = d[2], hA = d[3];
            if (w <= 0 || hh <= 0 || w > HX || hh > HY || wA <= 0 || hA <= 0)
                return fail(h, IRBPP_EINVAL, "shape %d rot %d: bad window %dx%d / %dx%d", s, r, w, hh, wA, hA);
            // the reference's window slice would run off the heightmap (NumPy broadcast error, space.py:118)
            if (w > STEP * wA || hh > STEP * hA)
                return fail(h, IRBPP_EINVAL, "shape %d rot %d: window %dx%d exceeds action footprint %dx%d "
                            "(the reference fails on this table)", s, r, w, hh, wA, hA);
            const int64_t off = offsets[(size_t)s * R + r];
            const int64_t n = (int64_t)w * hh;
            if ((int)n > maxwh) maxwh = (int)n;
            if (off < 0 || off + 4 * n > maps_len) return fail(h, IRBPP_EINVAL, "shape %d rot %d: table out of range", s, r);
            ShapeRot& q = srot[(size_t)s * R + r];
            q.w = w; q.h = hh;
            q.nX = AX - wA + 1; q.nY = AY - hA + 1;                  // range(rangeX_A - rangeX_OA + 1)
            if (q.nX < 0) q.nX = 0; if (q.nY < 0) q.nY = 0;
            q.ez = np_round6(e[2]);
            // prejudge (binPhy.py:236,240-241): round(round(l*resA, 6) + extent - bin, 6) > 0 fails
            q.okx = 0; q.oky = 0;
            for (int l = 0; l < AX; ++l) {
                const double tx = np_round6((double)l * c.resolution_act);
                if (!(np_round6(tx + e[0] - c.bin_dimension[0]) > 0)) q.okx |= 1u << l;
            }
            for (int l = 0; l < AY; ++l) {
                const double ty = np_round6((double)l * c.resolution_act);
                if (!(np_round6(ty + e[1] - c.bin_dimension[1]) > 0)) q.oky |= 1u << l;
            }
            q.off = (int64_t)Bs.size();
            const double* T = maps + off; const double* B = T + n; const double* mT = B + n; const double* mB = mT + n;
            int any_zero = 0;
            for (int64_t i = 0; i < n; ++i) {
                if ((mB[i] != 0.0 && mB[i] != 1.0) || (mT[i] != 0.0 && mT[i] != 1.0))
                    return fail(h, IRBPP_EINVAL, "shape %d rot %d: masks must be 0/1", s, r);
                if (!isfinite(B[i]) || !isfinite(T[i])) return fail(h, IRBPP_EINVAL, "shape %d rot %d: non-finite height", s, r);
                if (mB[i] == 0.0) any_zero = 1;
                Bs.push_back(mB[i] != 0.0 ? B[i] : INFINITY);
                Ts.push_back(mT[i] != 0.0 ? T[i] : -INFINITY);
            }
            q.any_zero = any_zero;
            q.tile = 1; q.tile_off = 0; q.ntiles = 0;
        }
        // block structure of the bottom tables of shape s (all rotations must agree on the block size)
        for (int t = 4; t >= 2; t >>= 1) {
            bool ok = true;
            std::vector<std::vector<TileEntry>> found(R);
            for (int r = 0; r < R && ok; ++r) {
                const ShapeRot& q = srot[(size_t)s * R + r];
                const double* Bq = Bs.data() + q.off;            // +inf where masked
                for (int bi = 0; bi * t < q.w && ok; ++bi)
                    for (int bj = 0; bj * t < q.h && ok; ++bj) {
                        const int i1 = std::min(bi * t + t, q.w), j1 = std::min(bj * t + t, q.h);
                        bool any_open = false, any_masked = false, same = true;
                        double b0 = 0.0; bool have = false;
                        for (int i = bi * t; i < i1; ++i)
                            for (int j = bj * t; j < j1; ++j) {
                                const double b = Bq[(size_t)i * q.h + j];
                                if (std::isinf(b)) any_masked = true;
                                else { any_open = true; if (!have) { b0 = b; have = true; } else if (b != b0) same = false; }
                            }
                        if (!any_open) continue;                  // fully masked block contributes nothing
                        if (any_masked || !same || i1 - bi * t != t || j1 - bj * t != t) { ok = false; break; }
                        TileEntry e; e.off = 8 * ((bi * t / 2) * 16 + (bj * t / 2)); e.pad = 0; e.b = b0;
                        found[r].push_back(e);
                    }
            }
            if (ok) {
                for (int r = 0; r < R; ++r) {
                    ShapeRot& q = srot[(size_t)s * R + r];
                    q.tile = t; q.tile_off = (int32_t)tiles.size(); q.ntiles = (int32_t)found[r].size();
                    tiles.insert(tiles.end(), found[r].begin(), found[r].end());
                }
                break;
            }
        }
        if (srot[(size_t)s * R].tile == 1) {
            // no block structure: one entry per unmasked cell, offset into the column-parity planes
            for (int r = 0; r < R; ++r) {
                ShapeRot& q = srot[(size_t)s * R + r];
                const double* Bq = Bs.data() + q.off;
                q.tile_off = (int32_t)tiles.size();
                for (int i = 0; i < q.w; ++i)
                    for (int j = 0; j < q.h; ++j) {
                        const double b = Bq[(size_t)i * q.h + j];
                        if (std::isinf(b)) continue;
                        TileEntry e; e.off = 8 * hm_index(i, j); e.pad = 0; e.b = b;
                        tiles.push_back(e);
                    }
                q.ntiles = (int32_t)tiles.size() - q.tile_off;
            }
        }
        for (int r = 0; r < R; ++r) max_entries = std::max(max_entries, (int)srot[(size_t)s * R + r].ntiles);
    }
    DeviceGuard guard(c.device);
    CUDA_TRY(h, cudaDeviceSynchronize());
    for (void* old : {(void*)h->srot_dev, (void*)h->Bs_dev, (void*)h->Ts_dev, (void*)h->vol_dev, (void*)h->rew_dev, (void*)h->tiles_dev})
        free_dev(h, old);                                                 // a reload replaces the previous pools
    CUDA_TRY(h, dev_alloc(h, &h->srot_dev, srot.size(), false));
    CUDA_TRY(h, dev_alloc(h, &h->Bs_dev, Bs.size() + 1, false));
    CUDA_TRY(h, dev_alloc(h, &h->Ts_dev, Ts.size() + 1, false));
    CUDA_TRY(h, dev_alloc(h, &h->vol_dev, (size_t)S, false));
    CUDA_TRY(h, dev_alloc(h, &h->rew_dev, (size_t)S, false));
    CUDA_TRY(h, dev_alloc(h, &h->tiles_dev, tiles.size() + 1, false));
    if (!tiles.empty()) CUDA_TRY(h, cudaMemcpy(h->tiles_dev, tiles.data(), tiles.size() * sizeof(TileEntry), cudaMemcpyHostToDevice));
    h->P.tiles = h->tiles_dev;
    CUDA_TRY(h, cudaMemcpy(h->srot_dev, srot.data(), srot.size() * sizeof(ShapeRot), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->Bs_dev, Bs.data(), Bs.size() * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->Ts_dev, Ts.data(), Ts.size() * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->vol_dev, vol, (size_t)S * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->rew_dev, rew.data(), (size_t)S * 8, cudaMemcpyHostToDevice));
    h->P.S = S; h->P.srot = h->srot_dev; h->P.Bs = h->Bs_dev; h->P.Ts = h->Ts_dev;
    h->P.vol = h->vol_dev; h->P.reward_tab = h->rew_dev;
    (void)maxwh;
    h->P.maxwh = max_entries;
    // per-warp staging lists, then the bin's candidate table row (bulk-copied by the scan kernel)
    h->scan_smem = CTA_WARPS * h->P.maxwh * (int)sizeof(TileEntry) + ((h->P.cand_stride * 2 + 15) & ~15);
    CUDA_TRY(h, raise_dynamic_smem(c.device, 1, h->scan_smem));
    h->shapes_loaded = true;
    return IRBPP_OK;
}

// fresh per-bin state: cursors restart, every bin's first sequence entry is staged for its first draw
static int restart_items(irbpp_env* h, const int32_t* ids, int32_t length) {
    std::vector<EnvState> st((size_t)h->P.N);
    memset(st.data(), 0, st.size() * sizeof(EnvState));
    if (ids) for (int e = 0; e < h->P.N; ++e) st[e].next_seq = ids[(size_t)e * length];
    CUDA_TRY(h, cudaDeviceSynchronize());
    CUDA_TRY(h, cudaMemcpy(h->P.state, st.data(), st.size() * sizeof(EnvState), cudaMemcpyHostToDevice));
    h->was_reset = false;
    h->scan_current = false;
    return IRBPP_OK;
}

int irbpp_set_sequences(irbpp_handle h, const int32_t* ids, int32_t length) {
    if (!h || !ids || length <= 0) return fail(h, IRBPP_EINVAL, "bad sequences");
    if (!h->shapes_loaded) return fail(h, IRBPP_ESTATE, "load shapes before sequences");
    const size_t n = (size_t)h->P.N * length;
    for (size_t i = 0; i < n; ++i)
        if (ids[i] < 0 || ids[i] >= h->P.S) return fail(h, IRBPP_EINVAL, "item id %d out of range at %zu", ids[i], i);
    DeviceGuard guard(h->cfg.device);
    CUDA_TRY(h, cudaDeviceSynchronize());
    free_dev(h, h->seq_dev); h->seq_dev = nullptr;                       // a reload replaces the previous pool
    CUDA_TRY(h, dev_alloc(h, &h->seq_dev, n, false));
    CUDA_TRY(h, cudaMemcpy(h->seq_dev, ids, n * 4, cudaMemcpyHostToDevice));
    int rc = restart_items(h, ids, length); if (rc) return rc;
    h->P.seq = h->seq_dev; h->P.L = length;
    h->sequences_set = true;
    return IRBPP_OK;
}

int irbpp_set_item_rng(irbpp_handle h, uint64_t seed) {
    if (!h) return IRBPP_EINVAL;
    if (!h->shapes_loaded) return fail(h, IRBPP_ESTATE, "load shapes before the item generator");
    DeviceGuard guard(h->cfg.device);
    int rc = restart_items(h, nullptr, 0); if (rc) return rc;
    h->P.seq = nullptr; h->P.L = 0; h->P.rng_seed = seed;
    h->sequences_set = true;
    return IRBPP_OK;
}

// One pass of the pipeline: scan kernel (or the levels kernel for caller-supplied maps), then the
// candidates kernel when the observation carries candidate rows.  (Running bin ranges on separate
// streams so that one range's candidates kernel overlaps the next range's scan kernel was measured:
// no gain -- the scan kernel owns the whole register file, the two cannot co-reside.)
// IRBPP_HANDOVER=grid restores the grid-wide wait (measurement switch)
static bool flags_enabled() {
    static const bool on = [] { const char* e = getenv("IRBPP_HANDOVER"); return !(e && strcmp(e, "grid") == 0); }();
    return on;
}

static int launch(irbpp_env* h, Params& P, cudaStream_t s) {
    // the units of a launch: bins, or (bin, buffer slot) pairs for get_all_possible_observation
    const int units = (P.mode == MODE_ALL_OBS) ? P.N * P.K : P.N;
    P.env_lo = 0;
    P.env_hi = units;
    // per-unit hand-over flags instead of the grid-wide dependency wait.  Not for caller-supplied maps (the levels kernel
    // sets none) and not for the fused all-slot pass (the k scan CTAs of a bin share its state and candidate table, which
    // the candidates CTA of the last slot rewrites: that one must wait for all of them)
    P.ready = (P.mode == MODE_DEBUG_HULLS || P.mode == MODE_ALL_OBS || !flags_enabled()) ? nullptr : h->ready_dev;
    if (++h->epoch == 0) h->epoch = 1;
    P.epoch = h->epoch;
    if (P.mode == MODE_DEBUG_HULLS) irbpp_levels_kernel<<<P.N, CTA_THREADS, 0, s>>>(P);
    else irbpp_scan_kernel<<<units, CTA_THREADS, h->scan_smem, s>>>(P);
    h->launches += 1;
    if (mode_emits_loc(P.mode, P.K)) {
        // programmatic dependent launch: the candidates grid is scheduled while the scan grid's last
        // wave drains and waits at griddepcontrol.wait for the scan's completion
        cudaLaunchConfig_t lc = {};
        lc.gridDim = dim3((units + h->epc - 1) / h->epc); lc.blockDim = dim3(32 * h->epc);
        lc.dynamicSmemBytes = (size_t)h->cand_smem; lc.stream = s;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = (P.mode == MODE_DEBUG_HULLS) ? 0 : 1;
        lc.attrs = at; lc.numAttrs = 1;
        if (h->epc == ENVS_PER_CTA_WIDE) cudaLaunchKernelEx(&lc, irbpp_candidates_kernel<ENVS_PER_CTA_WIDE>, P);
        else cudaLaunchKernelEx(&lc, irbpp_candidates_kernel<ENVS_PER_CTA_NARROW>, P);
        h->launches += 1;
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(h, IRBPP_ECUDA, "kernel launch: %s", cudaGetErrorString(e));
    // buffered step / reset change the heightmap without a scan; the debug modes scan foreign inputs
    // (get_all_possible_observation leaves its scans indexed by (bin, slot): not what the heuristic kernel reads)
    h->scan_current = (P.mode == MODE_CANDIDATES || ((P.mode == MODE_STEP || P.mode == MODE_RESET) && P.K == 1));
    return IRBPP_OK;
}

static int ready(irbpp_env* h) {
    if (!h) return IRBPP_EINVAL;
    if (!h->shapes_loaded || !h->sequences_set) return fail(h, IRBPP_ESTATE, "shapes / sequences not loaded");
    return IRBPP_OK;
}

int irbpp_reset(irbpp_handle h, const uint8_t* which, float* obs_out, void* stream) {
    int rc = ready(h); if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    if (!obs_out) return fail(h, IRBPP_EINVAL, "obs_out is null");
    cudaStream_t s = (cudaStream_t)stream;
    if (h->waiting_step) {         // "Called reset() while waiting for the step to complete" (shmem_vec_env.py:61-63)
        cudaStreamSynchronize(h->pending_stream);
        h->waiting_step = false;
    }
    Params P = h->P;
    P.mode = MODE_RESET; P.obs = obs_out; P.which = nullptr;
    if (which) {
        CUDA_TRY(h, cudaMemcpyAsync(h->which_dev, which, (size_t)P.N, cudaMemcpyHostToDevice, s));
        P.which = h->which_dev;
    }
    rc = launch(h, P, s); if (rc) return rc;
    h->was_reset = true;
    return IRBPP_OK;
}

static int step_async_impl(irbpp_env* h, const int64_t* actions, int32_t on_device, float* obs_out, void* stream,
                           int pose_actions) {
    int rc = ready(h); if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    if (!actions || !obs_out) return fail(h, IRBPP_EINVAL, "null argument");
    if (!h->was_reset) return fail(h, IRBPP_ESTATE, "step before reset");
    if (h->waiting_step) return fail(h, IRBPP_ESTATE, "already running an async step");   // vec_env.py:7-16
    cudaStream_t s = (cudaStream_t)stream;
    Params P = h->P;
    P.mode = MODE_STEP; P.obs = obs_out; P.pose_actions = pose_actions;
    h->results_on_host = !on_device;
    if (on_device) {
        P.actions = actions;
        rc = launch(h, P, s); if (rc) return rc;
    } else {
        // host actions: pinned staging + one H2D copy (measured 12 us faster end to end than letting the kernel read
        // them over PCIe); results: every bin's thread 0 also stores them into this step's pinned host block
        memcpy(h->actions_pinned, actions, (size_t)P.N * sizeof(int64_t));
        P.actions = h->actions_dev;
        h->res_turn ^= 1;                                   // this step's host block (the previous step's stays readable)
        P.res_host = h->results_mapped[h->res_turn];
        // (One CUDA graph per step -- H2D copy + both kernels, instantiated per observation buffer -- was measured:
        // submit 12.8 -> 8.8 us, but the step's wait grew by as much, e2e 0.162 vs 0.155 ms; dropped.)
        CUDA_TRY(h, cudaMemcpyAsync(h->actions_dev, h->actions_pinned, (size_t)P.N * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        rc = launch(h, P, s); if (rc) return rc;
    }
    h->waiting_step = true; h->pending_stream = s;
    return IRBPP_OK;
}

int irbpp_step_async(irbpp_handle h, const int64_t* actions, int32_t on_device, float* obs_out, void* stream) {
    return step_async_impl(h, actions, on_device, obs_out, stream, 0);
}

int irbpp_step_poses_async(irbpp_handle h, const int64_t* poses, int32_t on_device, float* obs_out, void* stream) {
    return step_async_impl(h, poses, on_device, obs_out, stream, 1);
}

static void export_results(const StepResults& r, irbpp_step_result* out) {
    out->reward = r.reward; out->done = r.done; out->valid = r.valid; out->error = r.error;
    out->counter = r.counter; out->ep_len = r.ep_len; out->ratio = r.ratio; out->ep_reward = r.ep_reward;
}

int irbpp_step_wait(irbpp_handle h, irbpp_step_result* out) {
    int rc = ready(h); if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    if (!h->waiting_step) return fail(h, IRBPP_ESTATE, "not running an async step");   // vec_env.py:18-26
    cudaStream_t s = h->pending_stream;
    h->waiting_step = false;
    void* block = h->results_host[h->res_turn];
    if (out && !h->results_on_host)            // a device-resident step waited for with the host call: fetch the block
        CUDA_TRY(h, cudaMemcpyAsync(block, h->results_dev, h->results_bytes, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(h, cudaStreamSynchronize(s));
    if (out) {
        export_results(carve_results(block, h->P.N), out);
        for (int i = 0; i < h->P.N; ++i)
            if (out->error[i]) return fail(h, IRBPP_EDEVICE, "env %d reported device error code %d", i, (int)out->error[i]);
    }
    return IRBPP_OK;
}

int irbpp_step_wait_device(irbpp_handle h, irbpp_device_result* out) {
    int rc = ready(h); if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    if (!h->waiting_step) return fail(h, IRBPP_ESTATE, "not running an async step");
    h->waiting_step = false;
    if (out) export_results(h->P.res, out);
    return IRBPP_OK;
}

int irbpp_device_results(irbpp_handle h, irbpp_device_result* out) {
    if (!h || !out) return IRBPP_EINVAL;
    export_results(h->P.res, out);
    return IRBPP_OK;
}

int irbpp_get_action_candidates(irbpp_handle h, const int64_t* order_actions, int32_t on_device,
                                float* loc_obs_out, void* stream) {
    int rc = ready(h); if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    if (!order_actions || !loc_obs_out) return fail(h, IRBPP_EINVAL, "null argument");
    if (h->P.K <= 1) return fail(h, IRBPP_ESTATE, "get_action_candidates needs buffer_size > 1");
    if (!h->was_reset) return fail(h, IRBPP_ESTATE, "get_action_candidates before reset");
    cudaStream_t s = (cudaStream_t)stream;
    Params P = h->P;
    P.mode = MODE_CANDIDATES; P.obs = loc_obs_out; P.obs_stride = P.loc_len;
    if (on_device) P.actions = order_actions;
    else {
        // staged copy (not zero-copy): the caller may enqueue the following step before this kernel ran
        memcpy(h->actions_pinned + P.N, order_actions, (size_t)P.N * sizeof(int64_t));
        CUDA_TRY(h, cudaMemcpyAsync(h->actions_dev, h->actions_pinned + P.N, (size_t)P.N * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        P.actions = h->actions_dev;
    }
    return launch(h, P, s);
}

int irbpp_get_all_possible_observation(irbpp_handle h, float* out, void* stream) {
    int rc = ready(h); if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    if (!out) return fail(h, IRBPP_EINVAL, "null argument");
    if (h->P.K <= 1) return fail(h, IRBPP_ESTATE, "get_all_possible_observation needs buffer_size > 1");
    if (!h->was_reset) return fail(h, IRBPP_ESTATE, "called before reset");
    Params P = h->P;
    // every (bin, buffered item) pair is one unit of ONE scan launch and ONE candidates launch (binPhy.py:175-179
    // loops over the k items): the K scans of a bin share its heightmap through L2 and the candidate extraction packs
    // the contour tasks of all pairs densely
    P.mode = MODE_ALL_OBS; P.obs = out; P.obs_stride = P.K * P.loc_len;
    return launch(h, P, (cudaStream_t)stream);
}

int irbpp_heuristic_actions(irbpp_handle h, int32_t method, int32_t dir_idx, int32_t* poses_out, int64_t* index_out,
                            int32_t on_device, void* stream) {
    int rc = ready(h); if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    if (method < 0 || method >= HEUR_COUNT) return fail(h, IRBPP_EINVAL, "unknown heuristic %d", method);
    if (dir_idx < 0 || dir_idx > 3) return fail(h, IRBPP_EINVAL, "dir_idx %d not in 0..3", dir_idx);   // space.py:167
    if (!h->was_reset || !h->scan_current)
        return fail(h, IRBPP_ESTATE, "no current scan (call after reset / step, or after get_action_candidates when buffer_size > 1)");
    if (h->waiting_step) return fail(h, IRBPP_ESTATE, "a step is pending");
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = h->P.N;
    if (!h->heur_pose_dev) {
        CUDA_TRY(h, dev_alloc(h, &h->heur_pose_dev, N * 3));
        CUDA_TRY(h, dev_alloc(h, &h->heur_index_dev, N));
    }
    Params P = h->P;
    P.heur_method = method; P.heur_dir = dir_idx;
    P.heur_pose = (on_device && poses_out) ? poses_out : h->heur_pose_dev;
    P.heur_index = (on_device && index_out) ? index_out : h->heur_index_dev;
    irbpp_heuristic_kernel<<<P.N, CTA_THREADS, 0, s>>>(P);
    h->launches += 1;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(h, IRBPP_ECUDA, "kernel launch: %s", cudaGetErrorString(e));
    if (!on_device) {
        if (poses_out) CUDA_TRY(h, cudaMemcpyAsync(poses_out, h->heur_pose_dev, N * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        if (index_out) CUDA_TRY(h, cudaMemcpyAsync(index_out, h->heur_index_dev, N * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(h, cudaStreamSynchronize(s));
    }
    return IRBPP_OK;
}

int irbpp_debug_state(irbpp_handle h, double* heightmap, int32_t* queue, int32_t* cursor, int32_t* packed_count) {
    int rc = ready(h); if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    CUDA_TRY(h, cudaDeviceSynchronize());
    const int N = h->P.N;
    if (heightmap) {
        std::vector<double> raw((size_t)N * HX * HY);
        CUDA_TRY(h, cudaMemcpy(raw.data(), h->P.hm, raw.size() * 8, cudaMemcpyDeviceToHost));
        for (int e = 0; e < N; ++e)
            for (int x = 0; x < HX; ++x)
                for (int y = 0; y < HY; ++y)
                    heightmap[((size_t)e * HX + x) * HY + y] = raw[(size_t)e * HX * HY + hm_index(x, y)];
    }
    if (queue || cursor || packed_count) {
        std::vector<EnvState> st((size_t)N);
        CUDA_TRY(h, cudaMemcpy(st.data(), h->P.state, st.size() * sizeof(EnvState), cudaMemcpyDeviceToHost));
        const int k = h->P.K > 1 ? h->P.K : 1;
        for (int e = 0; e < N; ++e) {
            if (queue) for (int i = 0; i < k; ++i) queue[(size_t)e * k + i] = st[e].queue[i];
            if (cursor) cursor[e] = st[e].cursor;
            if (packed_count) packed_count[e] = st[e].packed;
        }
    }
    return IRBPP_OK;
}

int irbpp_debug_set_heightmap(irbpp_handle h, const double* heightmap) {
    int rc = ready(h); if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    if (!heightmap) return fail(h, IRBPP_EINVAL, "null argument");
    const int N = h->P.N;
    std::vector<double> raw((size_t)N * HX * HY);
    for (int e = 0; e < N; ++e)
        for (int x = 0; x < HX; ++x)
            for (int y = 0; y < HY; ++y)
                raw[(size_t)e * HX * HY + hm_index(x, y)] = heightmap[((size_t)e * HX + x) * HY + y];
    CUDA_TRY(h, cudaDeviceSynchronize());
    CUDA_TRY(h, cudaMemcpy(h->P.hm, raw.data(), raw.size() * 8, cudaMemcpyHostToDevice));
    return IRBPP_OK;
}

static int debug_run(irbpp_env* h, Params& P, double* posZmap, double* posZValid, double* naiveMask,
                     double* cand, int32_t* num_hull) {
    const size_t N = P.N, nm = N * P.R * NPOSE, nc = N * P.sel * 5;
    double* d_cd = nullptr; int32_t* d_nh = nullptr; float* d_obs = nullptr;
    auto cleanup = [&]() { cudaFree(d_cd); cudaFree(d_nh); cudaFree(d_obs); };
#define DBG_TRY(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) { cleanup(); return fail(h, IRBPP_ECUDA, "%s: %s", #expr, cudaGetErrorString(e_)); } } while (0)
    DBG_TRY(cudaMalloc(&d_cd, nc * 8)); DBG_TRY(cudaMalloc(&d_nh, N * 4));
    DBG_TRY(cudaMalloc(&d_obs, N * (size_t)P.loc_len * 4));
    P.dbg_cand = d_cd; P.dbg_nhull = d_nh; P.obs = d_obs; P.obs_stride = P.loc_len;
    int rc = launch(h, P, nullptr);
    if (rc) { cleanup(); return rc; }
    DBG_TRY(cudaDeviceSynchronize());
    if (posZmap || posZValid || naiveMask) {       // float64 views straight from the hand-over scratch
        std::vector<double> pz(nm);
        std::vector<uint32_t> mb(N * P.R * 8);
        DBG_TRY(cudaMemcpy(pz.data(), P.posz, nm * 8, cudaMemcpyDeviceToHost));
        DBG_TRY(cudaMemcpy(mb.data(), P.maskbits, mb.size() * 4, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < nm; ++i) {
            const bool m = (mb[i >> 5] >> (i & 31)) & 1u;
            if (posZmap) posZmap[i] = pz[i];
            if (posZValid) posZValid[i] = m ? pz[i] : POSZ_INVALID;
            if (naiveMask) naiveMask[i] = m ? 1.0 : 0.0;
        }
    }
    if (cand) DBG_TRY(cudaMemcpy(cand, d_cd, nc * 8, cudaMemcpyDeviceToHost));
    if (num_hull) DBG_TRY(cudaMemcpy(num_hull, d_nh, N * 4, cudaMemcpyDeviceToHost));
    std::vector<uint8_t> errs(N);
    DBG_TRY(cudaMemcpy(errs.data(), P.res.error, N, cudaMemcpyDeviceToHost));
    cleanup();
#undef DBG_TRY
    for (size_t i = 0; i < N; ++i) if (errs[i]) return fail(h, IRBPP_EDEVICE, "env %zu reported device error code %d", i, (int)errs[i]);
    return IRBPP_OK;
}

int irbpp_debug_scan(irbpp_handle h, const int32_t* item_ids, double* posZmap, double* posZValid,
                     double* naiveMask, double* cand, int32_t* num_hull) {
    int rc = ready(h); if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    if (!item_ids) return fail(h, IRBPP_EINVAL, "null argument");
    for (int i = 0; i < h->P.N; ++i)
        if (item_ids[i] < 0 || item_ids[i] >= h->P.S) return fail(h, IRBPP_EINVAL, "item id out of range");
    int32_t* d_items = nullptr;
    CUDA_TRY(h, cudaMalloc(&d_items, (size_t)h->P.N * 4));
    CUDA_TRY(h, cudaMemcpy(d_items, item_ids, (size_t)h->P.N * 4, cudaMemcpyHostToDevice));
    Params P = h->P;
    P.mode = MODE_DEBUG_SCAN; P.dbg_items = d_items;
    rc = debug_run(h, P, posZmap, posZValid, naiveMask, cand, num_hull);
    cudaFree(d_items);
    return rc;
}

int irbpp_debug_hulls(irbpp_handle h, const double* posZValid, const double* mask, double* cand, int32_t* num_hull) {
    int rc = ready(h); if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    if (!posZValid || !mask) return fail(h, IRBPP_EINVAL, "null argument");
    const size_t nm = (size_t)h->P.N * h->P.R * NPOSE;
    std::vector<uint32_t> mb((size_t)h->P.N * h->P.R * 8, 0u);
    for (size_t i = 0; i < nm; ++i) if (mask[i] != 0.0) mb[i >> 5] |= 1u << (i & 31);
    CUDA_TRY(h, cudaDeviceSynchronize());
    CUDA_TRY(h, cudaMemcpy(h->P.posz, posZValid, nm * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->P.maskbits, mb.data(), mb.size() * 4, cudaMemcpyHostToDevice));
    Params P = h->P;
    P.mode = MODE_DEBUG_HULLS;
    return debug_run(h, P, nullptr, nullptr, nullptr, cand, num_hull);
}

int64_t irbpp_launch_count(irbpp_handle h) { return h ? h->launches : 0; }

// ---- compact form of the location observation for the rollout gather (csrc/irbpp_pack.cuh) --------------------
int irbpp_packed_obs_bytes(int32_t selected_action) { return selected_action > 0 ? packed_words(selected_action) * 4 : -1; }

int irbpp_pack_observations(const float* obs, int64_t obs_stride, int32_t selected_action, int32_t n, void* packed, void* stream) {
    if (!obs || !packed || n <= 0 || selected_action <= 0 || obs_stride < selected_action * 5 + 9 + 1024)
        return fail(nullptr, IRBPP_EINVAL, "bad pack arguments");
    DeviceGuard guard(device_of(obs));
    irbpp_pack_obs_kernel<<<n, 128, 0, (cudaStream_t)stream>>>(obs, obs_stride, selected_action, reinterpret_cast<uint32_t*>(packed), n);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(nullptr, IRBPP_ECUDA, "kernel launch: %s", cudaGetErrorString(e));
    return IRBPP_OK;
}

int irbpp_unpack_observations(const void* packed, int32_t selected_action, int32_t n, float* obs, int64_t obs_stride, void* stream) {
    if (!obs || !packed || n <= 0 || selected_action <= 0 || obs_stride < selected_action * 5 + 9 + 1024)
        return fail(nullptr, IRBPP_EINVAL, "bad unpack arguments");
    DeviceGuard guard(device_of(obs));
    irbpp_unpack_obs_kernel<<<n, 128, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint32_t*>(packed), selected_action, obs, obs_stride, n);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(nullptr, IRBPP_ECUDA, "kernel launch: %s", cudaGetErrorString(e));
    return IRBPP_OK;
}

// ---- point clouds of the next items (SURVEY.md 8(f)3; csrc/irbpp_pointnet.cuh) ----------------------------------
static int pn_common(PointNetParams& Q, const float* shape_array, int32_t S, int32_t P, const float* obs, int64_t obs_stride,
                     int32_t item_col, const int32_t* ids, int32_t B, uint64_t seed, uint64_t counter, int32_t n_points) {
    if (!shape_array || S <= 0 || P <= 0 || B <= 0 || n_points <= 0) return fail(nullptr, IRBPP_EINVAL, "bad point-cloud arguments");
    if (!obs && !ids) return fail(nullptr, IRBPP_EINVAL, "either the observations or explicit item ids are needed");
    if (obs && !ids && (obs_stride <= 0 || item_col < 0 || item_col >= obs_stride)) return fail(nullptr, IRBPP_EINVAL, "bad item column");
    memset(&Q, 0, sizeof(Q));
    Q.shape_array = shape_array; Q.S = S; Q.P = P; Q.n_points = n_points; Q.seed = seed; Q.counter = counter;
    Q.obs = obs; Q.obs_stride = obs_stride; Q.item_col = item_col; Q.ids = ids; Q.B = B;
    return IRBPP_OK;
}

int irbpp_sample_point_clouds(const float* shape_array, int32_t S, int32_t P, const float* obs, int64_t obs_stride,
                              int32_t item_col, const int32_t* ids, int32_t B, uint64_t seed, uint64_t counter,
                              int32_t n_points, float* out, int32_t* indices_out, void* stream) {
    PointNetParams Q;
    int rc = pn_common(Q, shape_array, S, P, obs, obs_stride, item_col, ids, B, seed, counter, n_points); if (rc) return rc;
    if (!out) return fail(nullptr, IRBPP_EINVAL, "null output");
    Q.out = out; Q.indices_out = indices_out;
    DeviceGuard guard(device_of(shape_array));
    const int64_t n = (int64_t)B * n_points;
    const int blocks = (int)std::min<int64_t>((n + 255) / 256, 148 * 16);
    irbpp_cloud_gather_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(Q);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(nullptr, IRBPP_ECUDA, "kernel launch: %s", cudaGetErrorString(e));
    return IRBPP_OK;
}

int irbpp_shape_features(const float* shape_array, int32_t S, int32_t P, const float* obs, int64_t obs_stride,
                         int32_t item_col, const int32_t* ids, int32_t B, uint64_t seed, uint64_t counter,
                         int32_t n_points, const float* W1, const float* b1, const float* W2, const float* b2,
                         float negative_slope, int32_t* scratch_keys, float* out, void* stream) {
    PointNetParams Q;
    int rc = pn_common(Q, shape_array, S, P, obs, obs_stride, item_col, ids, B, seed, counter, n_points); if (rc) return rc;
    if (!W1 || !b1 || !W2 || !b2 || !scratch_keys || !out) return fail(nullptr, IRBPP_EINVAL, "null argument");
    Q.W1 = W1; Q.b1 = b1; Q.W2 = W2; Q.b2 = b2; Q.slope = negative_slope; Q.feat_keys = scratch_keys; Q.out = out;
    const int dev = device_of(shape_array);
    DeviceGuard guard(dev);
    cudaError_t e = raise_dynamic_smem(dev, 2, PN_SMEM_BYTES);
    if (e != cudaSuccess) return fail(nullptr, IRBPP_ECUDA, "shape encoder set-up: %s", cudaGetErrorString(e));
    cudaStream_t s = (cudaStream_t)stream;
    irbpp_pn_init_kernel<<<(S * PN_H + 255) / 256, 256, 0, s>>>(scratch_keys, S * PN_H);
    const int tiles = (n_points + PN_TILE - 1) / PN_TILE;
    irbpp_shape_encode_kernel<<<S * tiles, PN_THREADS, PN_SMEM_BYTES, s>>>(Q);
    const int64_t n = (int64_t)B * PN_H;
    irbpp_feature_gather_kernel<<<(int)std::min<int64_t>((n + 255) / 256, 148 * 16), 256, 0, s>>>(Q);
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail(nullptr, IRBPP_ECUDA, "kernel launch: %s", cudaGetErrorString(e));
    return IRBPP_OK;
}

// ---- prioritized n-step replay banks (SURVEY.md 8(f)2; csrc/irbpp_replay.cuh) ---------------------------------------
static int replay_check(const irbpp_replay_banks* b) {
    if (!b || b->num_banks <= 0 || b->capacity <= 0 || b->obs_len <= 0 || b->row_stride < b->obs_len || (b->row_stride & 3))
        return fail(nullptr, IRBPP_EINVAL, "bad replay bank descriptor");
    if (!b->tree || !b->states || !b->actions || !b->rewards || !b->nonterminals || !b->index || !b->full ||
        !b->max_priority || !b->timestep || (reinterpret_cast<uintptr_t>(b->states) & 15))
        return fail(nullptr, IRBPP_EINVAL, "replay bank: null or misaligned buffer");
    return IRBPP_OK;
}

static int launch_status(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(nullptr, IRBPP_ECUDA, "%s launch: %s", what, cudaGetErrorString(e));
    return IRBPP_OK;
}

int irbpp_replay_append(const irbpp_replay_banks* banks, const float* state, int64_t state_stride, const int64_t* action,
                        const float* reward, const uint8_t* done, const uint8_t* valid, float reward_clip, void* stream) {
    int rc = replay_check(banks); if (rc) return rc;
    if (!state || !action || !reward || !done || state_stride < banks->obs_len)
        return fail(nullptr, IRBPP_EINVAL, "bad replay append arguments");
    DeviceGuard guard(device_of(banks->tree));
    irbpp_replay_append_kernel<<<banks->num_banks, REPLAY_APPEND_THREADS, 0, (cudaStream_t)stream>>>(
        *banks, state, state_stride, action, reward, done, valid, reward_clip);
    return launch_status("replay append");
}

int irbpp_replay_sample(const irbpp_replay_banks* banks, const irbpp_replay_sample_args* a, void* stream) {
    int rc = replay_check(banks); if (rc) return rc;
    if (!a || a->batch <= 0 || a->multi_step < 0 || a->multi_step > IRBPP_REPLAY_MAX_STEPS || a->max_attempts <= 0 ||
        !a->banks || !a->tree_index || !a->states || !a->actions || !a->returns || !a->next_states || !a->nonterminals ||
        !a->weights || !a->error)
        return fail(nullptr, IRBPP_EINVAL, "bad replay sample arguments");
    const int N = banks->num_banks;
    const bool choose = N > a->batch;                       // agent.py:69 would give 0 draws per memory
    const int m = choose ? a->batch : N, per = choose ? 1 : a->batch / N;
    ReplaySampleParams S;
    memset(&S, 0, sizeof(S));
    S.per = per; S.n = a->multi_step;
    for (int k = 0; k < a->multi_step; ++k) S.scale[k] = a->n_step_scaling[k];
    S.neg_beta = (float)(-a->priority_weight); S.beta_is_one = a->priority_weight == 1.0;
    S.seed = a->seed; S.counter = a->counter; S.u_table = a->u_table; S.max_attempts = a->max_attempts;
    S.banks = a->banks; S.choose = choose;
    S.tree_index = a->tree_index; S.states = a->states; S.actions = a->actions; S.returns = a->returns;
    S.next_states = a->next_states; S.nonterminals = a->nonterminals; S.weights = a->weights; S.error = a->error;
    DeviceGuard guard(device_of(banks->tree));
    cudaStream_t s = (cudaStream_t)stream;
    if (choose) irbpp_replay_choose_kernel<<<1, 32, 0, s>>>(a->banks, m, N, a->seed, a->counter);
    const int warps = std::min(per, REPLAY_MAX_WARPS);
    irbpp_replay_sample_kernel<<<m, warps * 32, 0, s>>>(*banks, S);
    return launch_status("replay sample");
}

int irbpp_replay_update_priorities(const irbpp_replay_banks* banks, const int64_t* tree_index, const float* priority,
                                   int32_t count, void* stream) {
    int rc = replay_check(banks); if (rc) return rc;
    if (count < 0 || (count > 0 && (!tree_index || !priority))) return fail(nullptr, IRBPP_EINVAL, "bad replay update arguments");
    if (count == 0) return IRBPP_OK;
    DeviceGuard guard(device_of(banks->tree));
    irbpp_replay_update_kernel<<<1, REPLAY_UPDATE_THREADS, 0, (cudaStream_t)stream>>>(*banks, tree_index, priority, count);
    return launch_status("replay update");
}

int irbpp_debug_phase_cycles(irbpp_handle h, int32_t enable, uint64_t* out8) {
    if (!h) return IRBPP_EINVAL;
    DeviceGuard guard(h->cfg.device);
#ifdef IRBPP_PROBE_TRACE
    const size_t trace_words = 8 + ((size_t)h->P.N * h->P.K + 1) * 8;     // profiling build: per-CTA timelines behind the counters
#else
    const size_t trace_words = 8;
#endif
    if (!h->phase_dev) CUDA_TRY(h, dev_alloc(h, &h->phase_dev, trace_words));
    CUDA_TRY(h, cudaDeviceSynchronize());
    if (out8) CUDA_TRY(h, cudaMemcpy(out8, h->phase_dev, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
#ifdef IRBPP_PROBE_TRACE
    if (const char* path = getenv("IRBPP_TRACE_FILE")) {
        std::vector<unsigned long long> tr(trace_words);
        CUDA_TRY(h, cudaMemcpy(tr.data(), h->phase_dev, trace_words * 8, cudaMemcpyDeviceToHost));
        if (FILE* f = fopen(path, "wb")) { fwrite(tr.data(), 8, trace_words, f); fclose(f); }
    }
#endif
    CUDA_TRY(h, cudaMemset(h->phase_dev, 0, trace_words * sizeof(uint64_t)));
    h->P.phase_cycles = enable ? h->phase_dev : nullptr;
    return IRBPP_OK;
}

}  // extern "C"
