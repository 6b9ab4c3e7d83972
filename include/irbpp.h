/*
 * irbpp.h -- C ABI of the B200-native IR-BPP packing-environment hot path.
 *
 * The reference (alexfrom0815/IR-BPP) has no FFI layer: its boundary is the Python VecEnv class
 * contract of envs.py:67-165 / wrapper/vec_env.py:29-108 / wrapper/shmem_vec_env.py:20-157.
 * Each entry point below states the reference interface it replaces (paths relative to the
 * reference root).  Host code (Python `irbpp_b200.vec_env.GpuVecEnv`) binds these with ctypes;
 * INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++ / torch types cross this boundary
 *   - every function returns 0 on success or a negative IRBPP_E* code; the message is available
 *     from irbpp_last_error(handle) (thread-unsafe per handle; one host thread per handle)
 *   - "dev" pointers are CUDA device pointers owned by the caller (e.g. torch tensors);
 *     "host" pointers are ordinary host memory owned by the caller
 *   - all GPU work is ordered on the `stream` argument (a cudaStream_t passed as void*, NULL =
 *     default stream); the library owns its internal state and result staging buffers
 *   - there is no CPU fallback: without a CUDA device irbpp_create fails with IRBPP_ECUDA
 */
#ifndef IRBPP_H_
#define IRBPP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IRBPP_ABI_VERSION 2

#define IRBPP_OK        0
#define IRBPP_EINVAL   -1   /* bad argument / unsupported configuration */
#define IRBPP_ECUDA    -2   /* CUDA runtime error */
#define IRBPP_ESTATE   -3   /* call order violated (e.g. step_async twice; vec_env.py:7-26) */
#define IRBPP_EDEVICE  -4   /* a kernel flagged an environment error (see irbpp_last_error) */

typedef struct irbpp_env* irbpp_handle;

/* PackingGame.__init__ / Space.__init__ settings that reach the hot path
 * (environment/physics0/binPhy.py:25-49, space.py:15-24, arguments.py:11-96,115). */
typedef struct irbpp_config {
    int32_t num_envs;          /* N bins resident on this GPU (args.num_processes) */
    int32_t num_rotations;     /* ZRotNum = --resolutionRot (arguments.py:85,117) */
    int32_t selected_action;   /* --selectedAction, candidate rows per observation (default 500) */
    int32_t buffer_size;       /* --bufferSize k; k > 1 selects the order->location protocol */
    double  bin_dimension[3];  /* [0.32, 0.32, 0.30] (arguments.py:115) */
    double  resolution_act;    /* --resolutionA 0.02 */
    double  resolution_h;      /* --resolutionH 0.01 */
    double  resolution_z;      /* --resolutionZ 0.01 (cvTools.py:77 heightResolution) */
    int32_t device;            /* CUDA device ordinal */
    int32_t approx_legacy;     /* 0: approxPolyDP as cv2 4.13 (segment distance); 1: legacy line distance */
} irbpp_config;

/* Views of the per-env results of the last step.  Replaces the (rews, dones, infos) tuple of ShmemVecEnv.step_wait
 * (wrapper/shmem_vec_env.py:76-81) and the Monitor episode info (wrapper/monitor.py:58-75).  The eight arrays lie in
 * one library-owned block of 31 bytes per env, in the order ratio | ep_reward | reward | counter | ep_len | done |
 * valid | error.  irbpp_step_wait returns host views into one of two pinned blocks that alternate, so they stay valid
 * until the SECOND next irbpp_step_async on the handle; irbpp_step_wait_device and irbpp_device_results return
 * device views of the one device block (irbpp_device_result is the same struct). */
typedef struct irbpp_step_result {
    const float*   reward;      /* [N]  10*volume/bin_volume on success, 0 otherwise (binPhy.py:299-322) */
    const uint8_t* done;        /* [N]  1 when the placement failed and the bin was auto-reset */
    const uint8_t* valid;       /* [N]  info['Valid'] (always 1 without the PyBullet settle) */
    const uint8_t* error;       /* [N]  non-zero: kernel-detected error for that env */
    const int32_t* counter;     /* [N]  info['counter'] = items packed, meaningful where done */
    const int32_t* ep_len;      /* [N]  info['episode']['l'], meaningful where done */
    const double*  ratio;       /* [N]  info['ratio'] = packed volume / bin volume, where done */
    const double*  ep_reward;   /* [N]  unrounded sum of episode rewards (Monitor rounds to 6 dp) */
} irbpp_step_result;

/* Device-resident copies of the same arrays (for callers that keep the loop on the GPU). */
typedef irbpp_step_result irbpp_device_result;

int irbpp_abi_version(void);

/* Replaces: make_vec_envs + N x PackingGame(args) construction (envs.py:67-99, binPhy.py:22-116). */
int irbpp_create(const irbpp_config* cfg, irbpp_handle* out);
int irbpp_destroy(irbpp_handle h);
const char* irbpp_last_error(irbpp_handle h);   /* h may be NULL: error of the last failed create */

/* Observation lengths: binPhy.py:87-98.  loc = selected_action*5 + 9 + Hx*Hy; order = k + Hx*Hy;
 * obs_len = (k > 1) ? order : loc. */
int irbpp_obs_len(irbpp_handle h, int32_t* obs_len, int32_t* loc_obs_len, int32_t* order_obs_len);

/* Replaces: args.shotInfo / args.shapeDict / args.infoDict (tools.py:248-279, binPhy.py:31-33).
 * Host arrays: dims[S,R,4] = (w, h, wA, hA) from space.py:104-106; ext[S,R,3] raw mesh extents;
 * vol[S]; maps = float64 pool with the four [w,h] row-major tables T | B | maskT | maskB of (s,r)
 * starting at offsets[s,r] (in doubles). */
int irbpp_load_shapes(irbpp_handle h, int32_t num_shapes, int32_t num_rotations,
                      const int32_t* dims, const double* ext, const double* vol,
                      const double* maps, const int64_t* offsets, int64_t maps_len);

/* Replaces: the item creators (environment/physics0/IRcreator.py:6-103).  ids[N,L] host int32; env e
 * draws ids[e, cursor % L] on every generate_item; the cursor persists across episodes.  Calling it again
 * replaces the sequences and restarts the cursors. */
int irbpp_set_sequences(irbpp_handle h, const int32_t* ids, int32_t length);

/* Alternative to explicit sequences: env e draws  id = mix(seed, e, draw counter) mod num_shapes  on the device
 * (splitmix64 finaliser, csrc/irbpp_kernels.cuh item_rng) -- i.i.d. uniform ids without a period, the stand-in
 * for RandomItemCreator (environment/physics0/IRcreator.py:26-33: np.random.choice on every generate_item). */
int irbpp_set_item_rng(irbpp_handle h, uint64_t seed);

/* Replaces: envs.reset() (envs.py:149-152 -> ShmemVecEnv.reset, shmem_vec_env.py:60-66; and
 * reset_specific, :113-118, when `which` (host uint8[N], 1 = reset) is not NULL).
 * obs_out: dev float32 [N, obs_len]; rows of envs not reset are left untouched. */
int irbpp_reset(irbpp_handle h, const uint8_t* which, float* obs_out, void* stream);

/* Replaces: envs.step_async (envs.py:154-159 -> shmem_vec_env.py:70-74).  actions: int64[N], a host
 * pointer (copied through pinned staging) or a device pointer when actions_on_device != 0.
 * obs_out: dev float32 [N, obs_len], written in stream order.  Returns IRBPP_ESTATE if a step is
 * already pending. */
int irbpp_step_async(irbpp_handle h, const int64_t* actions, int32_t actions_on_device,
                     float* obs_out, void* stream);

/* Replaces: envs.step_wait (envs.py:161-165 -> shmem_vec_env.py:76-81).  Copies the per-env results to
 * pinned host memory, synchronises the step's stream and fills *out.  out may be NULL (sync only). */
int irbpp_step_wait(irbpp_handle h, irbpp_step_result* out);

/* Device-side loop variant: marks the pending step as consumed without any host copy or sync and
 * returns device views of the result arrays (valid in stream order). */
int irbpp_step_wait_device(irbpp_handle h, irbpp_device_result* out);

/* The device copies of the per-env result arrays (fixed for the life of the handle; every step writes them in
 * stream order, also when its results are delivered to the host): what a device-resident replay buffer reads. */
int irbpp_device_results(irbpp_handle h, irbpp_device_result* out);

/* Replaces: envs.get_action_candidates(order_actions) (wrapper/shmem_vec_env.py:99-102 ->
 * binPhy.py:161-169), buffer_size > 1 only.  order_actions: int64[N] host or device.
 * loc_obs_out: dev float32 [N, loc_obs_len]. */
int irbpp_get_action_candidates(irbpp_handle h, const int64_t* order_actions, int32_t on_device,
                                float* loc_obs_out, void* stream);

/* Replaces: PackingGame.get_all_possible_observation (binPhy.py:171-180), buffer_size > 1 only.
 * out: dev float32 [N, k * loc_obs_len].  Leaves the candidate state of slot k-1 current. */
int irbpp_get_all_possible_observation(irbpp_handle h, float* out, void* stream);

/* Replaces: Space.get_heuristic_action(dirIdx, method, next_item_ID, next_item)
 * (environment/physics0/space.py:162-227) for every bin, over the drop heights / feasibility mask of
 * the bin's current item (the scan of the last reset / step (buffer_size 1) or
 * get_action_candidates).  method: IRBPP_HEUR_*; dir_idx 0..3 selects the X/Y flips (:163-166).
 * poses_out: int32[N,3] (rotIdx, lx, ly); index_out: int64[N] row of that pose in the bin's candidate
 * table (what envs.step takes), -1 if the pose is not a candidate; either may be NULL; both host
 * pointers, or device pointers when outputs_on_device != 0 (then nothing is synchronised).
 * The reference's RANDOM branch raises on every call and has no counterpart.
 * Returns IRBPP_ESTATE when no current scan exists (before reset, or buffer_size > 1 without
 * get_action_candidates). */
#define IRBPP_HEUR_MINZ      0
#define IRBPP_HEUR_DBLF      1
#define IRBPP_HEUR_FIRSTFIT  2
#define IRBPP_HEUR_HM        3
int irbpp_heuristic_actions(irbpp_handle h, int32_t method, int32_t dir_idx, int32_t* poses_out,
                            int64_t* index_out, int32_t outputs_on_device, void* stream);

/* irbpp_step_async with explicit poses instead of candidate rows: poses int64[N], each
 * (rotIdx * Ax + lx) * Ay + ly -- the (rotIdx, lx, ly) binPhy.action_to_position (binPhy.py:234-236)
 * would have read from candidates[action].  Everything after that line of PackingGame.step is
 * unchanged (prejudge, placement, reward, auto-reset); pair with irbpp_step_wait as usual. */
int irbpp_step_poses_async(irbpp_handle h, const int64_t* poses, int32_t poses_on_device,
                           float* obs_out, void* stream);

/* ---- parity / debugging views (float64, host destinations; any pointer may be NULL) ---- */

/* Current bin state: heightmap [N,Hx,Hy] row-major; int32 next item ids queue [N, max(k,1)], sequence
 * cursor [N] and packed_count [N], the items packed in the current episode. */
int irbpp_debug_state(irbpp_handle h, double* heightmap, int32_t* queue, int32_t* cursor,
                      int32_t* packed_count);
int irbpp_debug_set_heightmap(irbpp_handle h, const double* heightmap /* host [N,Hx,Hy] */);

/* Run the scan + candidate extraction of space.py:98-129 / cvTools.py:61-103 / binPhy.py:205-225 for
 * item_ids[N] (host int32) on the CURRENT heightmaps without touching env state.  Host outputs:
 * posZmap, posZValid, naiveMask float64 [N,R,Ax,Ay]; cand float64 [N,selected_action,5];
 * num_hull int32 [N] = K before select/pad (0 = fallback path taken). */
int irbpp_debug_scan(irbpp_handle h, const int32_t* item_ids, double* posZmap, double* posZValid,
                     double* naiveMask, double* cand, int32_t* num_hull);

/* Candidate extraction alone on caller-supplied maps: posZValid, mask host float64 [N,R,Ax,Ay] ->
 * cand [N,selected_action,5], num_hull [N]  (cvTools.getConvexHullActions + binPhy.py:205-225). */
int irbpp_debug_hulls(irbpp_handle h, const double* posZValid, const double* mask, double* cand,
                      int32_t* num_hull);

/* Kernel launches issued by this handle so far (bench.py's gpu_launches). */
int64_t irbpp_launch_count(irbpp_handle h);

/* ---- compact observations for the rollout gather (SURVEY.md 8e) ----------------------------------------------
 * The float32 location observation [N, sel*5 + 9 + 1024] (binPhy.py:196-227) re-encoded without loss as u16 poses, f32
 * heights, one mask bit per row, the item id and the f32 heightmap: irbpp_packed_obs_bytes(sel) bytes per bin (7 184 at
 * sel = 500, 51 %).  What `sharding.CompactRolloutGather` sends between GPUs; device pointers, handle-free. */
int irbpp_packed_obs_bytes(int32_t selected_action);
int irbpp_pack_observations(const float* obs, int64_t obs_stride, int32_t selected_action, int32_t n, void* packed, void* stream);
int irbpp_unpack_observations(const void* packed, int32_t selected_action, int32_t n, float* obs, int64_t obs_stride, void* stream);

/* ---- point clouds of the next items (SURVEY.md 8(f)3) --------------------------------------------------------
 * Replaces model.py:328-335 / :366-372: `shapeArray[next_item_ID.cpu()]` (a HOST gather of [B, P, 3] float32 rows),
 * `np.random.randint(P, size=samplePointsNum)` (one index set shared by the batch) and the host-to-device copy
 * of [B, n, 3] on every forward pass.  Handle-free; every pointer is a DEVICE pointer owned by the caller;
 * errors are reported through irbpp_last_error(NULL).
 *   shape_array  float32 [S, P, 3], resident on the device (agent.py:26 `args.shapeArray`)
 *   item ids     ids int32 [B] when not NULL, else (int) obs[b * obs_stride + item_col]  (the next_item_vec slot of
 *                the observation: item_col = selected_action * 5, binPhy.py:191,227; model.py:327)
 *   index set    index j = mix(seed, counter, j) mod P  (counter-based, uniform with replacement like randint;
 *                csrc/irbpp_pointnet.cuh pn_index; pass a new counter per forward pass)
 * irbpp_sample_point_clouds: out float32 [B, n_points, 3] = shapeArray[item_b][indices] (drop-in for `nextShape`);
 *   indices_out int32 [n_points] or NULL.
 * irbpp_shape_features: the fused path -- shapeEncoder (model.py:266-270: Linear(3,128), LeakyReLU, Linear(128,128),
 *   LeakyReLU; weights in nn.Linear layout, float32) and the max over the points (model.py:335), evaluated once per
 *   library SHAPE (the index set is shared by the batch, so the feature depends on the shape only) and gathered per
 *   bin: out float32 [B, 128].  scratch_keys: int32 [S * 128] work space. */
int irbpp_sample_point_clouds(const float* shape_array, int32_t S, int32_t P, const float* obs, int64_t obs_stride,
                              int32_t item_col, const int32_t* ids, int32_t B, uint64_t seed, uint64_t counter,
                              int32_t n_points, float* out, int32_t* indices_out, void* stream);
int irbpp_shape_features(const float* shape_array, int32_t S, int32_t P, const float* obs, int64_t obs_stride,
                         int32_t item_col, const int32_t* ids, int32_t B, uint64_t seed, uint64_t counter,
                         int32_t n_points, const float* W1, const float* b1, const float* W2, const float* b2,
                         float negative_slope, int32_t* scratch_keys, float* out, void* stream);

/* ---- prioritized n-step replay, one bank per bin (SURVEY.md 8(f)2; csrc/irbpp_replay.cuh) ------------------------
 * Replaces: the N ReplayMemory objects of main.py:61-63 (memory.py:95-208), their appends in trainer.py:184-186 and the
 * sample / update_priorities calls of agent.py:68-124.  Bank b is exactly ReplayMemory(args, capacity, obs_len): a
 * sum tree of 2C-1 float32 nodes (leaves C-1 .. 2C-2, any C), a cyclic slot index, `full`, the running max priority
 * (starts at 1) and the episode timestep t.  Handle-free: the caller owns every buffer (device pointers); the calls
 * are ordered on `stream` and none synchronises with the host; errors through irbpp_last_error(NULL). */
#define IRBPP_REPLAY_MAX_STEPS 16

typedef struct irbpp_replay_banks {
    int32_t  num_banks;        /* N */
    int32_t  capacity;         /* C transitions per bank */
    int32_t  obs_len;          /* L floats per state */
    int32_t  row_stride;       /* floats between stored states: >= obs_len, a multiple of 4 (16-byte aligned rows) */
    float*   tree;             /* [N, 2C-1] sum trees */
    float*   states;           /* [N, C, row_stride] */
    int64_t* actions;          /* [N, C] */
    float*   rewards;          /* [N, C] */
    uint8_t* nonterminals;     /* [N, C] */
    int32_t* index;            /* [N] next slot (transitions.index) */
    uint8_t* full;             /* [N] */
    float*   max_priority;     /* [N] transitions.max, 1 initially */
    int32_t* timestep;         /* [N] ReplayMemory.t */
} irbpp_replay_banks;

/* memory.py:110-113 for every bank b with valid[b] != 0 (valid may be NULL: all):  state row b (stride state_stride
 * floats), action[b] (int64), reward[b] (float32, clamped to +-reward_clip when reward_clip > 0, trainer.py:181-182),
 * done[b] (uint8).  Reads the step's arrays in stream order (e.g. irbpp_device_results), so it can follow a step in
 * the same stream or CUDA graph without a host round trip. */
int irbpp_replay_append(const irbpp_replay_banks* banks, const float* state, int64_t state_stride, const int64_t* action,
                        const float* reward, const uint8_t* done, const uint8_t* valid, float reward_clip, void* stream);

/* ReplayMemory.sample (memory.py:191-203) as agent.learn draws it (agent.py:68-82).  N <= batch: every bank gives
 * batch / N stratified draws; N > batch: `batch` banks chosen uniformly without replacement on the device, one draw each
 * (the reference's formula then gives every weight 1).  Rows = banks * per, bank-major.  Draw (row, attempt) uses
 * u_table[row * max_attempts + attempt] (device float64) when u_table is not NULL, else a counter-based stream of
 * (seed, counter); a row still rejected after max_attempts gets error[row] = 1 (the reference would retry forever).
 * Outputs (device): banks int32 [rows / per], tree_index int64 [rows] = bank * (2C-1) + node, states / next_states
 * float32 [rows, obs_len], actions int64 [rows], returns / nonterminals / weights float32 [rows], error int32 [rows]. */
typedef struct irbpp_replay_sample_args {
    int32_t       batch;
    int32_t       multi_step;                             /* n <= IRBPP_REPLAY_MAX_STEPS */
    float         n_step_scaling[IRBPP_REPLAY_MAX_STEPS]; /* float32(discount ** k), memory.py:107 */
    double        priority_weight;                        /* beta */
    uint64_t      seed, counter;
    const double* u_table;
    int32_t       max_attempts;
    int32_t*      banks;
    int64_t*      tree_index;
    float*        states;
    int64_t*      actions;
    float*        returns;
    float*        next_states;
    float*        nonterminals;
    float*        weights;
    int32_t*      error;
} irbpp_replay_sample_args;
int irbpp_replay_sample(const irbpp_replay_banks* banks, const irbpp_replay_sample_args* args, void* stream);

/* ReplayMemory.update_priorities after np.power (memory.py:206-208): tree_index int64 [count] as irbpp_replay_sample
 * returned it, priority float32 [count] (device); applied in order (a later duplicate wins), max over every value. */
int irbpp_replay_update_priorities(const irbpp_replay_banks* banks, const int64_t* tree_index, const float* priority,
                                   int32_t count, void* stream);

/* Profiling aid: when enabled, thread 0 of every CTA adds the SM cycles it spent in each kernel phase
 * (0 scan kernel: load + apply action, 1 scan kernel: observation heightmap + scan + level bitmaps,
 * 2 candidates kernel: contour tasks, 3 candidates kernel: select / pad) to counters 0-3; counters 4-7 count
 * level images, (image, start pixel) micro-tasks, rounds and >64-point overflow redos.  The call
 * returns the counters accumulated so far in out8 (may be NULL), clears them and sets the switch. */
int irbpp_debug_phase_cycles(irbpp_handle h, int32_t enable, uint64_t* out8);

#ifdef __cplusplus
}
#endif
#endif /* IRBPP_H_ */
