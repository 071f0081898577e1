/*
 * piml_b200.h -- C ABI of libpiml_b200.so: the B200 (sm_100a) implementation of PIML's per-timestep
 * crowd-rollout hot path.
 *
 * The reference (tsinghua-fib-lab/PIML) is pure Python/PyTorch and has no FFI; the "operator interface" of the
 * hot path is a set of Python call signatures (SURVEY.md section 8b).  Each entry point below replaces the
 * reference function cited next to it and is what a binding for that function would call; the Python host
 * (piml_b200/*.py) keeps the reference's signatures and forwards to these through ctypes.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host; all floating point is fp32, indices int64
 *   - tensors are dense row-major with the shapes given per function; nothing is allocated by the library
 *     except where a workspace is explicitly passed in
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls are asynchronous
 *   - return value: 0 = success, non-zero = error code (PIML_ERR_*); piml_last_error() gives the message of the
 *     calling thread's last failure.  Nothing throws across the ABI.  There is NO CPU fallback.
 */
#ifndef PIML_B200_H
#define PIML_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define PIML_API __attribute__((visibility("default")))
#else
#define PIML_API
#endif

#define PIML_OK 0
#define PIML_ERR_INVALID 1   /* bad argument (shape, k too large, misaligned pointer, ...) */
#define PIML_ERR_CUDA 2      /* a CUDA runtime call or kernel launch failed */
#define PIML_ERR_UNSUPPORTED 3

PIML_API int piml_version(void);
PIML_API const char *piml_last_error(void);
/* Number of kernels this library has launched in the calling process (bench.py's gpu_launches counter). */
PIML_API int64_t piml_launch_count(void);
/* compute capability major*10+minor of the current device, SM count; <0 on error */
PIML_API int piml_device_info(int *sm_count, int *cc);

/* Pipe-throughput probes used by bench.py for the roofline denominators (no reference counterpart).  `ctas` CTAs x
 * 256 threads each run iters*4 "units" on independent dependent chains; out: ctas*256 floats.
 *   which = 0: unit = 8 FFMA                         (FLOPs = ctas*256*iters*32*2)
 *   which = 1: unit = 8 MUFU.EX2                     (ops   = ctas*256*iters*32)
 *   which = 2: unit = 8 FFMA2 (fma.rn.f32x2, packed) (FLOPs = ctas*256*iters*32*4)
 *   which = 3..6: unit = 8 FFMA2 + {2,4,0,4} MUFU.EX2 + {0,0,4,4} FSETP/FSEL pairs (co-issue test)
 *   which = 7..12: unit = 8 ops with all-distinct register operands: fma2(x,y,z), mul2, add2, fma2(y,y,x),
 *                  scalar fma(x,y,z), fma2(y,z',x)  (register-read-bandwidth test) */
PIML_API int piml_pipe_probe(int which, int ctas, int iters, float *out, void *stream);

/* ---- features: src/data/data.py:351-512 ------------------------------------------------------------------ */

/* Pedestrians.get_heading_direction (data.py:351-395).  vel (C,T,N,2) -> head (C,T,N,2): zero-speed frames take
 * the nearest later, else nearest earlier, non-zero velocity of the same pedestrian; then v/||v|| (0 stays 0). */
PIML_API int piml_heading_f32(const float *vel, int C, int T, int N, float *head, void *stream);

/* The desired-speed double loop of TimeIndexedPedData.make_dataset (data.py:797-806).  vel (T,N,2) -> out (N):
 * mean of ||v|| over frames [s, min(s+skip_frames,T)) with s the pedestrian's first frame of non-zero velocity
 * (0 if none).  The mean is accumulated in fp64 (torch.mean's fp32 summation order is not specified): <= 1 ulp. */
PIML_API int piml_desired_speed_f32(const float *vel, int T, int N, int skip_frames, float *out, void *stream);

/* Pedestrians.get_relative_quantity (data.py:398-414): out (frames,N,M,d) = B (frames,M,d)[m] - A (frames,N,d)[n].
 * Only for callers that ask for the dense tensor (the reference's polar / symbolic paths); the hot path fuses it. */
PIML_API int piml_relative_quantity_f32(const float *A, const float *B, int64_t frames, int N, int M, int d, float *out,
                                        void *stream);

/* Pedestrians.get_filtered_features (data.py:449-464): features (rows,M,d), idx int64 / dist (rows,k) ->
 * out (rows,k,d) = features[row, idx] with every slot of distance > dist_threshold zeroed. */
PIML_API int piml_filtered_features_f32(const float *features, const int64_t *idx, const float *dist, int64_t rows, int M,
                                        int k, int d, float dist_threshold, float *out, void *stream);

/* Pedestrians.get_nearby_obj_in_sight (data.py:416-447).  pos (B,N,2), obj (B,M,2) [obj_frame_stride = M*2] or
 * (M,2) shared by all frames [obj_frame_stride = 0], head (B,N,2).  k <= 32.
 * out_dist (B,N,kk) fp32 / out_idx (B,N,kk) int64, kk = min(k,M): the kk nearest objects inside the field of view
 * (cos(rel,head) >= cos_thr), ascending by (distance, index); out-of-view / NaN objects carry distance +inf. */
PIML_API int piml_select_neighbors_f32(const float *pos, const float *obj, int64_t obj_frame_stride, const float *head,
                              int B, int N, int M, int k, float cos_thr, float *out_dist, int64_t *out_idx,
                              void *stream);

/* Pedestrians.get_relative_features (data.py:466-512) with get_relative_quantity (:398-414),
 * get_nearby_obj_in_sight (:416-447) and get_filtered_features (:449-464) fused: nothing of size N*N is
 * materialised.  pos/vel/acc/dest (C,T,N,2); vel and acc get NaN->0 IN PLACE (data.py:483-484).
 * head: (C,T,N,2) from piml_heading_f32, or NULL when T == 1 (then heading = v/||v|| is computed inline).
 * obs (M,2) [obs_per_channel=0] or (C,M,2) [obs_per_channel=1]; M may be 0.
 * Outputs ped_f (C,T,N,kp',6), obs_f (C,T,N,ko',6), dest_f (C,T,N,2); kp'=min(kp,N), ko'=min(ko,M); kp,ko <= 32.
 * Optional (NULL to skip) selection outputs: *_idx int64 (-1 = empty slot) and *_dist (+inf = empty slot),
 * holding only neighbours with distance <= threshold. */
PIML_API int piml_relative_features_f32(const float *pos, float *vel, float *acc, const float *dest, const float *head,
                               const float *obs, int obs_per_channel, int C, int T, int N, int M, int kp,
                               float cos_thr_ped, float dist_thr_ped, int ko, float cos_thr_obs,
                               float dist_thr_obs, float *ped_f, float *obs_f, float *dest_f, int64_t *ped_idx,
                               float *ped_dist, int64_t *obs_idx, float *obs_dist, void *stream);

/* The per-step feature rebuild of the rollout loops (simulators.py:642-652 / :772-778) for S scenes of N slots
 * (one frame each): get_relative_features as above (heading = v/||v||) plus
 * self_f (S,N,7) = cat(dest_features, hist_v, acceleration, desired_speed) written by the same kernel.
 * obs (M,2) [obs_per_scene=0] or (S,M,2).  hist_v (S,N,2), desired_speed (S,N). */
PIML_API int piml_state_features_f32(const float *pos, float *vel, float *acc, const float *dest, const float *obs,
                            int obs_per_scene, int S, int N, int M, int kp, float cos_thr_ped, float dist_thr_ped,
                            int ko, float cos_thr_obs, float dist_thr_obs, const float *hist_v,
                            const float *desired_speed, float *ped_f, float *obs_f, float *self_f, float *dest_f,
                            void *stream);

/* piml_state_features_f32 for the rows [row0,row1) of ONE scene of N slots against all N agents and M obstacles
 * (agent-sharded crowd, SURVEY.md 8e): ped_f (row1-row0,kp,6), obs_f, self_f (row1-row0,7), dest_f (row1-row0,2) hold
 * only those rows.  pos / vel / acc / dest / hist_v / desired_speed are the WHOLE scene (every rank keeps all of it);
 * the in-place NaN -> 0 of data.py:483-484 is applied to all N rows so that the replicas stay identical.
 * Always the cell-list evaluation (needs finite distance thresholds); identical results to the unsharded call. */
PIML_API int piml_state_features_rows_f32(const float *pos, float *vel, float *acc, const float *dest, const float *obs,
                                 int N, int M, int64_t row0, int64_t row1, int kp, float cos_thr_ped,
                                 float dist_thr_ped, int ko, float cos_thr_obs, float dist_thr_obs,
                                 const float *hist_v, const float *desired_speed, float *ped_f, float *obs_f,
                                 float *self_f, float *dest_f, void *stream);

/* Pedestrians.calculate_collision_label (data.py:515-535). ped_f (S,6) -> out (S) in {0,1}. */
PIML_API int piml_collision_label_f32(const float *ped_f, int64_t S, float *out, void *stream);

/* piml_relative_features_f32 / piml_state_features_f32 pick between two evaluations that return the identical result:
 * all pairs (every agent scans all N + M candidates, like the reference) and a uniform-grid cell list (cells as wide
 * as the larger distance threshold; only the 3 x 3 cells around an agent are scanned) used from 4096 agents per frame.
 * algo: 0 = automatic (default), 1 = always all pairs, 2 = always cell list.  Process-wide setting. */
PIML_API int piml_set_feature_algorithm(int algo);
/* Frees the device scratch the library caches between calls: the cell-list path's grid arrays (per stream) and the
 * tensor-core forward's per-agent sums / compact-mode lists (per calling thread, device and stream).  Everything else
 * the library touches is passed in by the caller. */
PIML_API int piml_free_workspace(void);

/* Backward of piml_relative_features_f32 / the feature rebuild inside the differentiable rollout
 * (simulators.py:772-778 -> data.py:466-512; autograd through the subtractions of get_relative_quantity and the
 * gather of get_filtered_features; the sort indices carry no gradient).  B frames of N agents.
 * ped_idx (B,N,kp), obs_idx (B,N,ko): the selection the forward reported (-1 = zero-padded slot).
 * g_ped_f (B,N,kp,6), g_obs_f (B,N,ko,6) [NULL if ko == 0], g_dest_f (B,N,2) [may be NULL].
 * Outputs g_pos, g_vel, g_acc, g_dest (B,N,2); neighbour contributions are scattered with fp32 atomics. */
PIML_API int piml_relative_features_backward_f32(const float *pos, const float *dest, const int64_t *ped_idx,
                                        const int64_t *obs_idx, int B, int N, int kp, int ko, const float *g_ped_f,
                                        const float *g_obs_f, const float *g_dest_f, float *g_pos, float *g_vel,
                                        float *g_acc, float *g_dest, void *stream);

/* Pedestrians.collision_detection (data.py:538-601).  mode 3: position (T,N,2) [pass C = 1]; pairs that are closer
 * than `threshold` in more than 25 frames of position (or of real_position (T,N,2) when given) are friends and do not
 * count.  mode 4: position (C,T,N,2); pairs that touch in any of the first 4 frames of a channel are friends.
 * out_full (C,T,N,N) 0/1 and/or out_rowsum (C,T,N) = sum over the last axis (the only use the training rollout makes
 * of it, simulators.py:707-724); either may be NULL. */
PIML_API int piml_collision_detection_f32(const float *position, const float *real_position, int C, int T, int N,
                                 float threshold, int mode, float *out_full, float *out_rowsum, void *stream);

/* ---- MLAPM: src/models/mlapm.py:10-58, loop src/main_mlapm.py:18-36 ----------------------------------------- */

typedef struct {
    int version;        /* 0 = 'raw' (mlapm.py:28-29), 1 = 'GC' (:30-39).  'UCY' crashes in the reference. */
    float tau, A, B, C, D;
    float theta_deg;    /* self.args['theta'] */
    int exact_math;     /* 1: IEEE div/sqrt/expf per pair in the reference's op order; 0: rsqrt/ex2 fast path */
} piml_mlapm_params;

/* Bytes of workspace piml_mlapm_step_f32 needs for N agents (column-split partial sums). */
PIML_API int64_t piml_mlapm_workspace_bytes(int64_t N);

/* MLAPM.step for rows [row0,row1) against all N columns: action (row1-row0,2) = velocity + force*dt.
 * pos, vel, dest (N,2); desired_speed (N,ds_dim), ds_dim 1 or 2.  workspace >= piml_mlapm_workspace_bytes(N).
 * Dense all-pairs O(N^2), no cut-off, like the reference.  (row0,row1) lets an agent-sharded rank compute its
 * own rows after an all-gather of (pos,vel). */
PIML_API int piml_mlapm_step_f32(const float *pos, const float *vel, const float *desired_speed, int ds_dim,
                        const float *dest, int64_t N, int64_t row0, int64_t row1, const piml_mlapm_params *prm,
                        float dt, float *action, void *workspace, void *stream);

/* MLAPM.step fused with the rest of the loop body main_mlapm.py:26,34 for rows [row0,row1):
 *   action = MLAPM.step(..) ; pos_new = pos + action*dt ; arrived = ||pos_new - dest|| < radius  (uint8 0/1).
 * The caller compacts away inactive agents first, exactly as the reference's boolean-mask indexing does
 * (main_mlapm.py:20-23).  pos_new / arrived may be NULL. */
PIML_API int piml_mlapm_advance_f32(const float *pos, const float *vel, const float *desired_speed, int ds_dim,
                           const float *dest, int64_t N, int64_t row0, int64_t row1,
                           const piml_mlapm_params *prm, float dt, float radius, float *action, float *pos_new,
                           uint8_t *arrived, void *workspace, void *stream);

/* piml_mlapm_advance_f32 with the size of the caller's workspace stated.  With workspace_bytes >=
 * piml_mlapm_workspace_bytes_sym(N) and the whole crowd (row0 = 0, row1 = N) the library may evaluate every UNORDERED
 * pair once for both rows (the smooth part of mlapm.py:25-39 is symmetric under n <-> m; the two gates keep the
 * reference's exact fp32 arithmetic in both directions), which needs room for per-agent fixed-point sums, a spatial
 * sort of the crowd and a work list (O(N + (N/512)^2) bytes).  The symmetric path skips every pair farther apart than
 * piml_mlapm_cull_radius, where the fp32 weight is exactly 0.  Same results to fp32 summation order.
 * piml_set_mlapm_algorithm: 0 = automatic (symmetric, culled, from 16 384 agents), 1 = ordered pairs, 2 = symmetric,
 * culled, 3 = symmetric, dense (every pair, no culling). */
PIML_API int64_t piml_mlapm_workspace_bytes_sym(int64_t N);
PIML_API int piml_set_mlapm_algorithm(int algo);
/* Distance (m) beyond which the production math's weight of a pair is exactly +0 for these parameters:
 * (127 + |C log2 e|) / -(B + |D|) log2 e for 'GC', 127 / -(B log2 e) for 'raw' (exp2 of the exponent flushes to 0
 * below -126), plus 1 % + 0.01 m for approximate rsqrt and fp32 rounding.  +inf where nothing can be skipped:
 * exact_math, or a weight that does not decay with distance (B + |D| >= 0). */
PIML_API float piml_mlapm_cull_radius(const piml_mlapm_params *prm);
/* Diagnostics: the length of the work list (row block x 128-column stage items) that the last culled symmetric step
 * of N agents built in `workspace`.  Synchronous (waits for the device). */
PIML_API int piml_mlapm_cull_items(const void *workspace, int64_t N, int64_t *items);
PIML_API int piml_mlapm_advance_ws_f32(const float *pos, const float *vel, const float *desired_speed, int ds_dim,
                              const float *dest, int64_t N, int64_t row0, int64_t row1,
                              const piml_mlapm_params *prm, float dt, float radius, float *action, float *pos_new,
                              uint8_t *arrived, void *workspace, int64_t workspace_bytes, void *stream);

/* Many independent crowds (scenes) in one launch: for every scene s, piml_mlapm_advance_f32 on the scene's active
 * agents alone, with the scene's own constants.  Padded layout: pos, vel, dest, action, pos_new (S,N,2);
 * desired_speed (S,N,ds_dim), ds_dim 1 or 2; active, arrived (S,N) uint8.  Inactive slots take part in no pair (their
 * inputs may hold anything, NaN included) and get action = pos_new = NaN, arrived = 0.
 * prm: version and exact_math for the whole call, and the constants when scene_params is NULL.
 * scene_params: NULL, or device (S,6) float = tau, A, B, C, D, theta_deg per scene.
 * Each active agent sums over its scene's active agents in ascending slot order in one thread: a scene's result does
 * not depend on the other scenes, on S or on the launch shape, and is deterministic.  No workspace, no allocation.
 * 1 <= N <= PIML_MLAPM_SCENES_MAX_N (a scene's columns stay in shared memory), S >= 1, S*N < 2^31. */
#define PIML_MLAPM_SCENES_MAX_N 8192
PIML_API int piml_mlapm_scenes_advance_f32(const float *pos, const float *vel, const float *desired_speed, int ds_dim,
                                  const float *dest, const uint8_t *active, int64_t S, int64_t N,
                                  const piml_mlapm_params *prm, const float *scene_params, float dt, float radius,
                                  float *action, float *pos_new, uint8_t *arrived, void *stream);

/* piml_mlapm_advance_f32 for an agent-sharded crowd with the path's one exchange FUSED into it (SURVEY.md 8e): the
 * finalize kernel stores the new position and velocity of its rows [row0,row1) straight into every rank's next-state
 * arrays over NVLink / NVSwitch peer memory, instead of a separate all-gather.
 * peer_pos_next_host / peer_vel_next_host: HOST arrays of `world` (<= 16) device addresses -- rank g's (N,2) next-state
 * position / velocity arrays as mapped into this process (e.g. torch symmetric memory `buffer_ptrs` + offset), the
 * calling rank included.  The caller double-buffers the state and places one cross-rank barrier after the call.
 * Production math path only (prm->exact_math == 0). */
PIML_API int piml_mlapm_advance_push_f32(const float *pos, const float *vel, const float *desired_speed, int ds_dim,
                                const float *dest, int64_t N, int64_t row0, int64_t row1,
                                const piml_mlapm_params *prm, float dt, float radius, int world,
                                const uint64_t *peer_pos_next_host, const uint64_t *peer_vel_next_host,
                                uint8_t *arrived, void *workspace, void *stream);

/* Host-buffer entry of an agent-sharded step (piml_b200.sharded.ShardedCrowd.scatter_rows): this rank's rows
 * [row0, row0 + nrows) of position / velocity (and destination, may be NULL) -- device copies of what the rank uploaded
 * from the host -- are stored into EVERY rank's state arrays over NVLink peer memory by one kernel.  peer_*_host: host
 * arrays of `world` device pointers to each rank's (N,2) arrays.  The caller follows with a cross-rank barrier. */
PIML_API int piml_scatter_rows_push_f32(const float *pos_rows, const float *vel_rows, const float *dest_rows, int64_t row0,
                                        int64_t nrows, int world, const uint64_t *peer_pos_host,
                                        const uint64_t *peer_vel_host, const uint64_t *peer_dest_host, void *stream);

/* Agent-sharded crowd on the symmetric (unordered-pair) evaluation (SURVEY.md 8e).  Rank g owns the 512-agent blocks
 * [g T / G, (g+1) T / G), T = ceil(N / 512) (piml_mlapm_sym_shard_rows), and evaluates the block pairs of its own row
 * blocks; the exchange is fused into two kernels over NVLink / NVSwitch peer memory:
 *   piml_mlapm_sym_pairs_push_f32     pair kernel + per-rank reduction of the column-direction sums, stored into the
 *                                     inbox of the rank that owns each agent (peer_inbox_host: `world` device
 *                                     addresses of the ranks' inboxes, piml_mlapm_sym_inbox_bytes(N, world) each);
 *   -- cross-rank barrier (caller) --
 *   piml_mlapm_sym_finalize_push_f32  adds the ranks' shares in rank order, destination term, Euler update, arrival
 *                                     test (main_mlapm.py:26,34) and stores the new rows into every rank's next-state
 *                                     arrays like piml_mlapm_advance_push_f32;
 *   -- cross-rank barrier (caller) --
 * workspace >= piml_mlapm_sym_shard_workspace_bytes(N, world), the same buffer for both calls. */
PIML_API int piml_mlapm_sym_shard_rows(int64_t N, int world, int rank, int64_t *row0, int64_t *row1);
PIML_API int64_t piml_mlapm_sym_inbox_bytes(int64_t N, int world);
PIML_API int64_t piml_mlapm_sym_shard_workspace_bytes(int64_t N, int world);
PIML_API int piml_mlapm_sym_pairs_push_f32(const float *pos, const float *vel, const float *dest, int64_t N, int world,
                                  int rank, const piml_mlapm_params *prm, const uint64_t *peer_inbox_host,
                                  void *workspace, int64_t workspace_bytes, void *stream);
PIML_API int piml_mlapm_sym_finalize_push_f32(const float *pos, const float *vel, const float *desired_speed,
                                     int ds_dim, const float *dest, int64_t N, int world, int rank,
                                     const piml_mlapm_params *prm, float dt, float radius, const float *inbox_local,
                                     const uint64_t *peer_pos_next_host, const uint64_t *peer_vel_next_host,
                                     uint8_t *arrived, void *workspace, int64_t workspace_bytes, void *stream);

/* ---- SFM repulsion: src/utils/utils.py:31-100 ------------------------------------------------------------ */

/* UTILS.calc_acceleration.  rel (S, stride) with stride >= 4 floats per slot -> out (S,2).
 * version 0/1/2 = 'v0'/'v1'/'v2'; constants as the reference selects them per dataset. */
PIML_API int piml_calc_acceleration_f32(const float *rel, int64_t S, int stride, int version, float A, float B, float C,
                               float D, float theta, float eps, float *out, void *stream);

/* Pure social-force "model" with the model(ped, obs, self) -> [acc, ped_msgs, obs_msgs] interface of model.py:1185
 * (BASELINE config 2).  The reference's own simulator (models.socialforce) is not shipped; this is the composition of
 * shipped reference code that SURVEY.md 8c names: per slot the v0 repulsion of utils.py:53-58 with the ped constants
 * (A_ped, B_ped = 8.75, -2.5 for GC; 10.67, -3.33 for UCY, utils.py:47-52) and with the obstacle constants
 * (src/configs/socialforce.yaml:52-56: intensity 10 / radius 0.2 -> A_obs = 50, B_obs = -5), summed over slots, plus
 * the destination term model.py:1205-1210 (tau = 0.5, socialforce.yaml:29).  ped_f (R,kp,6), obs_f (R,ko,6) or NULL
 * with ko = 0, self_f (R,7) -> acc (R,2); ped_msgs (R,kp,2) / obs_msgs (R,ko,2) may be NULL. */
typedef struct { float A_ped, B_ped, A_obs, B_obs, eps, tau; } piml_sfm_params;
PIML_API int piml_sfm_forward_f32(const piml_sfm_params *prm, const float *ped_f, const float *obs_f,
                         const float *self_f, int64_t R, int kp, int ko, float *acc, float *ped_msgs,
                         float *obs_msgs, void *stream);

/* ---- interaction networks: src/models/model.py:40-119, :720-792, :1062-1305 -------------------------------- */

typedef struct {
    int n_enc; int enc_dims[9];   /* enc_dims[0] = 6, then n_enc encoder widths (MLP, model.py:40-65) */
    int proc_mode;                /* 0: ResDNN == 2x (processor_hidden_layers > 1, model.py:115-119) ; 1: relu(Wx+b)+x */
    int n_dec; int dec_dims[9];   /* dec_dims[0] = processor width, then n_dec decoder widths */
    int n_coll; int coll_dims[5]; /* collision head incl. input width; n_coll = 0: none */
    int kind;                     /* 0: per-slot decode, sum 2-d messages (pinnsf_bottleneck, pinnsf_bm);
                                     1: sum embeddings over slots, then decode (pinnsf, pinnsf_m) */
} piml_net_desc;

/* Number of floats of the device parameter layout of `desc` (both branches + collision head); <0 on a bad desc. */
PIML_API int64_t piml_pinnsf_packed_floats(const piml_net_desc *desc);

/* Re-layout the parameters for the fused forward.  params_torch (device): the Linears' parameters concatenated in
 * torch's own layout and forward order -- pedestrian branch (encoder, [processor block 0 if proc_mode==1], decoder,
 * predictor), obstacle branch (same), collision head; per Linear `weight` (out,in) row-major then `bias` (out) --
 * i.e. the reference module's state_dict tensors, untouched.  packed (device, 16-byte aligned,
 * piml_pinnsf_packed_floats floats): per Linear W^T padded to 16*NJ columns in the tile kernel's column order, then the
 * bias.  Call once per weight update. */
PIML_API int piml_pinnsf_pack_f32(const piml_net_desc *desc, const float *params_torch, float *packed, void *stream);

/* Forward of a PINNSF-family model (eval mode, or train mode with caller-supplied dropout multipliers).
 * params: the vector written by piml_pinnsf_pack_f32.  Layer widths <= 128.
 * ped (R,kp,6), obs (R,ko,6) (ignored if has_obs==0), self (R,7).  norm_group = 0: destination norm per row
 * (the (N,7) call); = N: reduce over the agent axis per component ((C,N,7) call, model.py:1206 dim=1 quirk).
 * drop_ped / drop_obs: NULL, or (R,k,pw) multipliers applied to the processor output (Dropout in train()).
 * Outputs acc (R,2), ped_msgs (R,kp,msgw), obs_msgs (R,ko,msgw), coll (R,kp); any of the last three may be NULL.
 * Uses a small stream-keyed scratch buffer owned by the library (per-agent message sums). */
PIML_API int piml_pinnsf_forward_f32(const piml_net_desc *desc, const float *params, int has_obs, float tau,
                            const float *ped, const float *obs, const float *self, int64_t R, int kp, int ko,
                            int norm_group, const float *drop_ped, const float *drop_obs, float *acc,
                            float *ped_msgs, float *obs_msgs, float *coll, void *stream);

/* Self test of the tensor-core path (tcgen05 kind::tf32, A in TMEM, accumulator in TMEM): y (128,N) = x (128,K) w^T
 * with w (N,K) row-major; terms = 1: plain TF32, 3: 3xTF32 split (fp32-grade).  K % 8 == 0, N % 16 == 0, both <= 128. */
PIML_API int piml_tc_selftest_f32(const float *x, const float *w, int K, int N, int terms, float *y, void *stream);

/* The same product on the 16-bit path (tcgen05 kind::f16): x and w split into fp16 hi + lo, terms = 3:
 * x_lo w_hi + x_hi w_lo + x_hi w_hi with fp32 accumulation in TMEM (fp32-grade, like 3xTF32, at twice the K per
 * instruction and half the TMEM / shared-memory footprint).  K % 16 == 0, N % 16 == 0, both <= 128.  swap = 0. */
PIML_API int piml_tc16_selftest_f32(const float *x, const float *w, int K, int N, int terms, int swap, float *y,
                                    void *stream);

/* Tensor-core forward (tcgen05 kind::tf32 with the 3xTF32 split, accumulators and activations in TMEM): the inference
 * path of the rollouts.  Same contract as piml_pinnsf_forward_f32 in eval mode without the collision head:
 * acc (R,2) and, for kind 0 models, optional 2-d messages ped_msgs (R,kp,2) / obs_msgs (R,ko,2) (NULL to skip).
 * Needs processor_hidden_layers > 1 and hidden widths that are multiples of 32 (<= 128);
 * piml_pinnsf_packed_tc_floats returns -1 for networks it cannot run (callers then use piml_pinnsf_forward_f32).
 * packed_tc: written by piml_pinnsf_pack_tc_f32 from the torch-layout vector (see piml_pinnsf_pack_f32). */
PIML_API int64_t piml_pinnsf_packed_tc_floats(const piml_net_desc *desc);
PIML_API int piml_pinnsf_pack_tc_f32(const piml_net_desc *desc, const float *params_torch, float *packed_tc, void *stream);
PIML_API int piml_pinnsf_forward_tc_f32(const piml_net_desc *desc, const float *packed_tc, int has_obs, float tau,
                               const float *ped, const float *obs, const float *self, int64_t R, int kp, int ko,
                               int norm_group, float *acc, float *ped_msgs, float *obs_msgs, void *stream);

/* ---- training: forward with activation stash + backward (loss.backward(), simulators.py:359, through the models) -- */

/* Floats of the activation stash of the training-mode forward for R agents (every Linear's post-activation output,
 * row-major per layer) and of the backward's workspace (per-layer pre-activation gradients + dW split partials). */
PIML_API int64_t piml_pinnsf_stash_floats(const piml_net_desc *desc, int has_obs, int64_t R, int kp, int ko);
PIML_API int64_t piml_pinnsf_backward_workspace_floats(const piml_net_desc *desc, int has_obs, int64_t R, int kp, int ko);

/* piml_pinnsf_forward_f32 that also fills `stash` (piml_pinnsf_stash_floats floats) for piml_pinnsf_backward_f32.
 * coll must be non-NULL when the model has a collision head.  processor_hidden_layers == 1 -> PIML_ERR_UNSUPPORTED. */
PIML_API int piml_pinnsf_forward_train_f32(const piml_net_desc *desc, const float *params, int has_obs, float tau,
                                  const float *ped, const float *obs, const float *self, int64_t R, int kp, int ko,
                                  int norm_group, const float *drop_ped, const float *drop_obs, float *acc,
                                  float *ped_msgs, float *obs_msgs, float *coll, float *stash, void *stream);

/* Backward-pass parameter layout: per Linear torch's own (out,in) matrix with tile-permuted columns (dX = dY W). */
PIML_API int64_t piml_pinnsf_packed_bwd_floats(const piml_net_desc *desc);
PIML_API int piml_pinnsf_pack_bwd_f32(const piml_net_desc *desc, const float *params_torch, float *packed_bwd, void *stream);

/* Backward of the forward above.  Inputs: the forward's inputs and stash, and the gradients of its outputs
 * g_acc (R,2) [required], g_ped_msgs (R,kp,msgw), g_obs_msgs (R,ko,msgw), g_coll (R,kp) [each may be NULL = zero].
 * Outputs: g_params = gradient in the layout of params_torch (piml_pinnsf_pack_f32's input; ped branch, obs branch,
 * collision head; per Linear weight (out,in) then bias); g_ped (R,kp,6), g_obs (R,ko,6), g_self (R,7) [may be NULL].
 * workspace: piml_pinnsf_backward_workspace_floats floats, 16-byte aligned.  Deterministic (no atomics). */
PIML_API int piml_pinnsf_backward_f32(const piml_net_desc *desc, const float *packed_bwd, int has_obs, float tau,
                             const float *ped, const float *obs, const float *self, int64_t R, int kp, int ko,
                             int norm_group, const float *drop_ped, const float *drop_obs, const float *stash,
                             const float *g_acc, const float *g_ped_msgs, const float *g_obs_msgs,
                             const float *g_coll, float *g_params, float *g_ped, float *g_obs, float *g_self,
                             float *workspace, void *stream);

/* ---- rollout losses: src/models/simulators.py:172-249 --------------------------------------------------------- */

/* multiple_rollout_mse_loss (:172), multiple_rollout_collision_loss (:195) for the collision and the hard-collision
 * counts, each with reduction 'sum', as test_multiple_rollouts_for_training calls them (:795-813), in one pass:
 *   out[0] = sum decay_t (pred - labels)^2,  decay_t = time_decay^(T-t-1)  (time_decay^t if reverse, :822-823)
 *   out[1] = sum w_cn decay_t (P pred - P labels)^2 with w from `collisions` (C,T,N), out[2] likewise from
 *            `hard_collisions`; either may be NULL (-> 0); abnormal_mask (N) or NULL (:222-224).
 * pred (C,T,N,2) contiguous; labels: row (c,t,n) starts at labels + ((c*T+t)*N+n)*label_stride and its first two
 * floats are used (data.labels[..., :2] has stride 6 + k; pass labels + 4 for the acceleration labels of :822).
 * workspace >= piml_rollout_losses_workspace_floats(C, N) floats.  T <= 256.
 * Backward: g_pred (C,T,N,2) = d(g_out[0] out[0] + g_out[1] out[1] + g_out[2] out[2]) / d pred, g_out on the device. */
PIML_API int64_t piml_rollout_losses_workspace_floats(int C, int N);
PIML_API int piml_rollout_losses_f32(const float *pred, const float *labels, int64_t label_stride, int C, int T, int N,
                            float time_decay, int reverse, const float *collisions, const float *hard_collisions,
                            const float *abnormal_mask, float *out, float *workspace, void *stream);
PIML_API int piml_rollout_losses_backward_f32(const float *pred, const float *labels, int64_t label_stride, int C, int T,
                                     int N, float time_decay, int reverse, const float *collisions,
                                     const float *hard_collisions, const float *abnormal_mask, const float *g_out,
                                     float *g_pred, void *stream);

/* l1_reg_loss(embeddings, weight, 'sum') (simulators.py:169-170, called at :735-737): out[0] = sum weight*|x|; and
 * its gradient g_x = g_out[0] * weight * sign(x).  One CTA, fixed summation order. */
PIML_API int piml_l1_sum_f32(const float *x, int64_t n, float weight, float *out, void *stream);
PIML_API int piml_l1_sum_backward_f32(const float *x, int64_t n, float weight, const float *g_out, float *g_x,
                                      void *stream);

/* The collision-prediction loss of the training rollout (simulators.py:826-830):
 * out[0] = F.binary_cross_entropy(pred, target, reduction='sum') (log clamped at -100 like ATen),
 * out[1] = number of elements with round(pred) == target;  backward: g_pred = g_out[0] (p - t) / max((1-p) p, 1e-12). */
PIML_API int piml_bce_sum_f32(const float *pred, const float *target, int64_t n, float *out, void *stream);
PIML_API int piml_bce_sum_backward_f32(const float *pred, const float *target, int64_t n, const float *g_out,
                                       float *g_pred, void *stream);

/* ---- evaluation metrics: src/functions/metrics.py ----------------------------------------------------------------- */

/* Per frame t of a rollout, over the agents with mask[t][n] == 1 (p, q (T,N,2); mask (T,N) uint8):
 *   out_mae[t]  sum ||p - q||_2                      mae_with_time_mask  metrics.py:29-42
 *   out_ot[t]   SinkhornDistance(eps, max_iter)      ot_with_time_mask   :45-67, :108-199 (log-domain updates, equal
 *               weights, stops when sum |u - u_prev| < 0.1, exactly the reference's per-frame loop)
 *   out_mmd[t]  MaximumMeanDiscrepancy, kernel_mul / kernel_num bandwidths   mmd_with_time_mask :70-91, :207-273
 *   out_count[t] number of masked agents; frames with count <= 1 are skipped by the reference: ot / mmd are NaN there
 *   (ot / mmd of a frame with more than PIML_METRICS_MAX_AGENTS = 1024 masked agents are NOT computed: NaN, and the
 *   caller must treat count[t] > 1024 as an error; out_mae has no such limit).  out_ot / out_mmd may be NULL.
 *   One CTA per frame. */
#define PIML_METRICS_MAX_AGENTS 1024
PIML_API int piml_metrics_frames_f32(const float *p, const float *q, const uint8_t *mask, int T, int N, float eps,
                            int max_iter, float kernel_mul, int kernel_num, float *out_mae, float *out_ot,
                            float *out_mmd, int *out_count, void *stream);

/* ---- integrator: src/models/simulators.py:603-639 ---------------------------------------------------------- */

/* One state update of get_multiple_rollouts for S scenes of N slots (SURVEY A.2 steps 3-6): lagged explicit
 * Euler, arrival / waypoint switch, removal on arrival, teacher-forced entry; also records the pre-update state.
 *   p,v,a,dest (S,N,2) in/out; dest_idx (S,N) int64 in/out; a_next (S,N,2); dest_num (S,N) int64;
 *   waypoints (S,D,N,2); hist_v (S,N,2) out; entry (S,N) int64 or NULL; *_gt = ground truth at t+1, (S,N,..).
 *   rec_p/rec_v/rec_a (S,N,2) and rec_mask (S,N) fp32: where to record the state at t (NULL to skip). */
PIML_API int piml_integrate_step_f32(float *p, float *v, float *a, const float *a_next, float *dest, int64_t *dest_idx,
                            const int64_t *dest_num, const float *waypoints, int S, int D, int N, float dt,
                            int remove_on_arrival, const int64_t *entry, const float *p_gt, const float *v_gt,
                            const float *a_gt, const float *dest_gt, const int64_t *dest_idx_gt, float *hist_v,
                            float *rec_p, float *rec_v, float *rec_a, float *rec_mask, void *stream);

/* ---- whole rollout loop: src/models/simulators.py:595-652 ---------------------------------------------------------- */

/* Everything BaseSimulator.get_multiple_rollouts' `for t in range(t_start, T)` loop touches, for S scenes of N slots
 * rolled together.  Time-major ground truth (frame t of all scenes contiguous); all pointers are device pointers. */
typedef struct {
    const piml_net_desc *desc;      /* network (NULL when sfm is given) */
    const float *packed;            /* piml_pinnsf_pack_f32 vector (FP32-pipe kernel), or NULL if packed_tc is given */
    const float *packed_tc;         /* piml_pinnsf_pack_tc_f32 vector (tensor-core kernel), or NULL */
    int has_obs; float tau;
    int S, N, M, D, T, t_start; float dt;
    int kp; float cos_p, thr_p; int ko; float cos_o, thr_o;            /* topk / cos(sight angle) / distance threshold */
    const float *obstacles; int obs_per_scene;                          /* (M,2) or (S,M,2) */
    const float *pos_tm, *vel_tm, *acc_tm, *dest_tm;                    /* (T,S,N,2) data.position ... data.destination */
    const int64_t *dest_idx_tm;                                         /* (T,S,N) */
    const int64_t *entry_tm;                                            /* (T,S,N) mask_p - mask_p_pred (simulators.py:593) */
    const int64_t *dest_num;                                            /* (S,N) */
    const float *waypoints;                                             /* (S,D,N,2) */
    const float *desired_speed;                                         /* (S,N) */
    float *p, *v, *a, *dest; int64_t *dest_idx; float *hist_v;          /* (S,N,..) state at t_start, updated in place */
    float *ped_f, *obs_f, *self_f, *dest_f;                             /* features of the state at t_start, in/out */
    float *a_next;                                                      /* (S,N,2) scratch */
    float *rec_p, *rec_v, *rec_a, *rec_mask;                            /* (T,S,N,2) x3, (T,S,N): rows t >= t_start written */
    const piml_sfm_params *sfm;     /* non-NULL: the pure social-force model replaces the network (desc, packed* unused) */
} piml_rollout_args;

/* Enqueues the whole loop (3-4 launches per step, no host synchronisation) on `stream`. */
PIML_API int piml_rollout_f32(const piml_rollout_args *args, void *stream);

/* ---- social-force constants sweep: one clip rolled out under S constant sets ------------------------------------- */

/* The pure social-force rollout of piml_rollout_f32 (sfm mode) of ONE clip from t_start to T, under S constant sets at
 * once.  The clip's ground truth, waypoints and obstacles are shared by all sets (no scene axis).  For each set s the
 * trajectory equals piml_rollout_f32 on the clip alone with params[s], bit for bit, on either route (persistent kernel
 * or per-step launches, chosen as piml_rollout_f32 chooses them).  Score per set, over t in [t_start, T) and the slots n
 * whose simulated position at t is not NaN and mask_p[t][n] == 1:
 *   err_sum[s] = sum ||p_sim[t][s][n] - pos_tm[t][n]||_2 (float64),  err_count[s] = number of terms.
 * Each slot sums its own terms in time order, then the slots of a set are added in slot order: the score does not
 * depend on S, on the set's position in the batch or on the route.  All pointers are device pointers. */
typedef struct {
    int S, N, M, D, T, t_start; float dt;
    int kp; float cos_p, thr_p; int ko; float cos_o, thr_o;            /* topk / cos(sight angle) / distance threshold */
    const float *obstacles;                                             /* (M,2), NULL when M == 0 */
    const float *pos_tm, *vel_tm, *acc_tm, *dest_tm;                    /* (T,N,2) */
    const int64_t *dest_idx_tm;                                         /* (T,N) */
    const int64_t *entry_tm;                                            /* (T,N) mask_p - mask_p_pred (simulators.py:593) */
    const float *mask_p;                                                /* (T,N): the slots the score compares */
    const int64_t *dest_num;                                            /* (N) */
    const float *waypoints;                                             /* (D,N,2) */
    const float *desired_speed;                                         /* (N) */
    const float *p, *v, *a, *dest; const int64_t *dest_idx;             /* (N,..) state at t_start (read only) */
    const float *ped_f, *obs_f, *self_f;                                /* (N,kp',6), (N,ko',6), (N,7) its features */
    const piml_sfm_params *params;                                      /* (S) constant sets */
    double *err_sum; int64_t *err_count;                                /* (S) out */
    float *rec_p, *rec_v, *rec_a, *rec_mask;  /* (T,S,N,2) x3, (T,S,N): rows t >= t_start written as piml_rollout_f32
                                                 writes them; all four NULL for a score-only sweep */
    void *workspace; int64_t workspace_bytes;                           /* >= piml_sfm_sweep_workspace_bytes(args) */
} piml_sfm_sweep_args;

/* Workspace bytes piml_sfm_sweep_f32 needs for these sizes and the route it will take: O(S N), never O(S T N). */
PIML_API int64_t piml_sfm_sweep_workspace_bytes(const piml_sfm_sweep_args *args);
PIML_API int piml_sfm_sweep_f32(const piml_sfm_sweep_args *args, void *stream);

/* ---- one NN-augmented rollout step, fused: src/models/simulators.py:595-652 ----------------------------------------- */

/* The loop body of get_multiple_rollouts re-ordered around the state: features of the current state
 * (get_relative_features without a heading argument, data.py:466-512, incl. the in-place NaN -> 0 of v and a) ->
 * a_next = model(features) (model.py:1185-1221) -> record / Euler / arrival / entry (simulators.py:596-639), as ONE call:
 * cell-list features in compact form -> tensor cores -> slot sums + destination term + state update (nn_step.cu).
 * Bit-identical to piml_state_features_f32 -> piml_pinnsf_forward_tc_f32 -> piml_integrate_step_f32 on the same state.
 * For the networks piml_nn_step_supported() accepts (per-slot decoders with hidden widths 32 / 64 / 128: pinnsf_bm,
 * pinnsf_bottleneck) and finite distance thresholds; otherwise PIML_ERR_UNSUPPORTED / PIML_ERR_INVALID and the caller
 * uses the three calls. */
typedef struct {
    const piml_net_desc *desc;      /* network */
    const float *packed_tc;         /* piml_pinnsf_pack_tc_f32 vector */
    int has_obs; float tau;
    int S, N, M, D; float dt; int remove_on_arrival;
    int kp; float cos_p, thr_p; int ko; float cos_o, thr_o;            /* topk / cos(sight angle) / distance threshold */
    const float *obstacles; int obs_per_scene;                          /* (M,2) or (S,M,2) */
    const int64_t *dest_num;                                            /* (S,N) */
    const float *waypoints;                                             /* (S,D,N,2) */
    const float *desired_speed;                                         /* (S,N) */
    float *p, *v, *a, *dest; int64_t *dest_idx; float *hist_v;          /* (S,N,..) state, updated in place */
    const int64_t *entry;                                               /* (S,N) or NULL: teacher-forced entry ... */
    const float *p_gt, *v_gt, *a_gt, *dest_gt; const int64_t *dest_idx_gt;   /* ... from the data at t+1, (S,N,..) */
    float *rec_p, *rec_v, *rec_a, *rec_mask;                            /* (S,N,2) x3, (S,N): the state at t, or NULL */
    float *a_next;                                                      /* (S,N,2) out: the model output, or NULL */
    float *ped_f, *obs_f, *self_f, *dest_f;   /* optional dense features of the state at t (all or none): (S,N,kp,6), ... */
} piml_nn_step_args;

PIML_API int piml_nn_step_supported(const piml_net_desc *desc);         /* 1 if piml_nn_step_f32 can run this network */
PIML_API int piml_nn_step_f32(const piml_nn_step_args *args, void *stream);

/* The same step for ONE RANK of an agent-sharded crowd (one scene): the rank holds the whole current state (args->p, v,
 * a: every agent's, read only), evaluates rows [row0, row1) -- features against all agents, network, state update --
 * and stores the new p, v, a of its rows into EVERY rank's next-state arrays p_next[g], v_next[g], a_next[g] (device
 * pointers of `world` <= 8 peers, this rank's own arrays included; NVLink peer memory) from the epilogue of its last
 * kernel.  dest / dest_idx / hist_v are updated in place for the own rows only (nobody else reads them).  The caller
 * separates steps with a cross-rank barrier and swaps current / next.  No dense feature outputs. */
PIML_API int piml_nn_step_shard_f32(const piml_nn_step_args *args, int64_t row0, int64_t row1, int world,
                                    const uint64_t *p_next, const uint64_t *v_next, const uint64_t *a_next,
                                    void *stream);

/* Backward of the differentiable rollout's state update (simulators.py:741-769: v' = v + a dt, p' = p + v dt,
 * a' = model output; agents overwritten by teacher-forced entry get no gradient).  n = S*N agents.
 * entry (n) int64 or NULL; g_p2,g_v2,g_a2 (n,2) = gradients of the updated state -> g_p,g_v,g_a,g_a_next (n,2). */
PIML_API int piml_integrate_step_backward_f32(const int64_t *entry, int64_t n, float dt, const float *g_p2,
                                     const float *g_v2, const float *g_a2, float *g_p, float *g_v, float *g_a,
                                     float *g_a_next, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PIML_B200_H */
