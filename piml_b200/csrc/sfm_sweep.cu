// sfm_sweep.cu -- one clip rolled out by the pure social-force model under S constant sets at once, scored on the
// device: what a calibration of A_ped, B_ped, A_obs, B_obs, tau runs thousands of times.
//
// The clip's ground truth (teacher-forced entry, waypoints, obstacles) is shared by all sets instead of copied per
// scene, and the recorded trajectories are optional, so the memory is O(S N) and not O(S T N).  Both routes of
// piml_rollout_f32's social-force mode run it, chosen the same way:
//   persistent   sfm_rollout_kernel<G, true> (rollout_sfm.cu): CTA s rolls set s, scores in registers
//   per step     sfm_forward_sets_kernel -> integrate_sweep_kernel -> piml_state_features_f32 on the (S,N) state
// Both add a slot's terms in time order with the same helper (sweep_err_term), and sweep_score_kernel adds the slots
// of a set in slot order, so a set's score does not depend on S, on its position or on the route.
#include "integrate_common.cuh"

namespace piml {
bool sfm_persistent_fits(int S, int N, int M, int kp, int ko, float thr_p, float thr_o);             // rollout_sfm.cu
int sfm_sweep_persistent_launch(const piml_sfm_sweep_args *w, double *err_acc, int64_t *err_cnt, cudaStream_t st);
int sfm_forward_sets_launch(const piml_sfm_params *sets, int N, const float *ped_f, const float *obs_f,  // sfm.cu
                            const float *self_f, int64_t R, int kp, int ko, float *acc, cudaStream_t st);
int integrate_sweep_launch(const IntArgs &g, cudaStream_t st);                                          // integrate.cu

// dst[s][k] = src[k] for s < S: the clip's initial state and features handed to every set
__global__ void sweep_broadcast_kernel(const uint32_t *__restrict__ src, int64_t words, int64_t total,
                                       uint32_t *__restrict__ dst) {
    for (int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; k < total;
         k += static_cast<int64_t>(gridDim.x) * blockDim.x)
        dst[k] = src[k % words];
}

// err_sum[s] / err_count[s]: the slots of set s added in slot order
__global__ void sweep_score_kernel(const double *__restrict__ acc, const int64_t *__restrict__ cnt, int S, int N,
                                   double *__restrict__ err_sum, int64_t *__restrict__ err_count) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    double e = 0.0;
    int64_t c = 0;
    for (int n = 0; n < N; ++n) {
        e = __dadd_rn(e, acc[static_cast<int64_t>(s) * N + n]);
        c += cnt[static_cast<int64_t>(s) * N + n];
    }
    err_sum[s] = e;
    err_count[s] = c;
}

// Workspace layout; every block 256-byte aligned.  The persistent route needs the score accumulators only.
struct SweepWs {
    double *err_acc; int64_t *err_cnt;                                         // (S,N)
    float *p, *v, *a, *dest, *hist_v, *dest_f, *a_next;                        // (S,N,2)
    int64_t *dest_idx;                                                         // (S,N)
    float *ped_f, *obs_f, *self_f, *ds;                                        // (S,N,kp,6), (S,N,ko,6), (S,N,7), (S,N)
};

static int64_t sweep_layout(const piml_sfm_sweep_args *w, bool persistent, SweepWs *out) {
    const int64_t SN = static_cast<int64_t>(w->S) * w->N;
    const int kp = w->kp < w->N ? w->kp : w->N;
    const int ko = w->M > 0 ? (w->ko < w->M ? w->ko : w->M) : 0;
    char *base = static_cast<char *>(w->workspace);
    int64_t off = 0;
    auto take = [&](int64_t bytes) -> void * {
        void *p = base ? base + off : nullptr;
        off += (bytes + 255) / 256 * 256;
        return p;
    };
    SweepWs ws = {};
    ws.err_acc = static_cast<double *>(take(SN * 8));
    ws.err_cnt = static_cast<int64_t *>(take(SN * 8));
    if (!persistent) {
        float **f2[] = {&ws.p, &ws.v, &ws.a, &ws.dest, &ws.hist_v, &ws.dest_f, &ws.a_next};
        for (float **f : f2) *f = static_cast<float *>(take(SN * 8));
        ws.dest_idx = static_cast<int64_t *>(take(SN * 8));
        ws.ped_f = static_cast<float *>(take(SN * kp * 24));
        ws.obs_f = ko > 0 ? static_cast<float *>(take(SN * ko * 24)) : nullptr;
        ws.self_f = static_cast<float *>(take(SN * 28));
        ws.ds = static_cast<float *>(take(SN * 4));
    }
    if (out) *out = ws;
    return off;
}

static bool sweep_persistent(const piml_sfm_sweep_args *w) {
    return sfm_persistent_fits(w->S, w->N, w->M, w->kp, w->ko, w->thr_p, w->thr_o);
}

static int broadcast(const void *src, int64_t bytes, int S, void *dst, cudaStream_t st) {
    const int64_t words = bytes / 4, total = words * S;
    if (total == 0) return PIML_OK;
    const int threads = 256;
    const int64_t blocks = (total + threads - 1) / threads;
    sweep_broadcast_kernel<<<static_cast<unsigned>(blocks < 65536 ? blocks : 65536), threads, 0, st>>>(
        static_cast<const uint32_t *>(src), words, total, static_cast<uint32_t *>(dst));
    count_launch();
    return check_launch("sweep_broadcast_kernel");
}

// The feature rebuild takes at most 65535 scenes per call; a power of two keeps every chunk's rows 256-byte aligned.
constexpr int SWEEP_FEATURE_SETS = 32768;

// The per-step route: the loop of rollout_step (rollout.cu) on the (S,N) state, with the set's constants per row.
static int sweep_per_step(const piml_sfm_sweep_args *w, const SweepWs &ws, cudaStream_t st) {
    const int S = w->S, N = w->N;
    const int64_t SN = static_cast<int64_t>(S) * N;
    const int kp = w->kp < N ? w->kp : N;
    const int ko = w->M > 0 ? (w->ko < w->M ? w->ko : w->M) : 0;
    int rc;
    const struct { const void *src; void *dst; int64_t bytes; } init[] = {
        {w->p, ws.p, N * 8}, {w->v, ws.v, N * 8}, {w->a, ws.a, N * 8}, {w->dest, ws.dest, N * 8},
        {w->dest_idx, ws.dest_idx, N * 8}, {w->ped_f, ws.ped_f, static_cast<int64_t>(N) * kp * 24},
        {w->obs_f, ws.obs_f, static_cast<int64_t>(N) * ko * 24}, {w->self_f, ws.self_f, N * 28},
        {w->desired_speed, ws.ds, N * 4}};
    for (const auto &c : init)
        if (c.bytes > 0 && (rc = broadcast(c.src, c.bytes, S, c.dst, st))) return rc;
    PIML_CUDA(cudaMemsetAsync(ws.err_acc, 0, SN * 8, st));
    PIML_CUDA(cudaMemsetAsync(ws.err_cnt, 0, SN * 8, st));
    IntArgs g = {};
    g.p = reinterpret_cast<float2 *>(ws.p); g.v = reinterpret_cast<float2 *>(ws.v); g.a = reinterpret_cast<float2 *>(ws.a);
    g.a_next = reinterpret_cast<const float2 *>(ws.a_next); g.dest = reinterpret_cast<float2 *>(ws.dest);
    g.dest_idx = ws.dest_idx; g.dest_num = w->dest_num; g.waypoints = reinterpret_cast<const float2 *>(w->waypoints);
    g.S = S; g.D = w->D; g.N = N; g.dt = w->dt; g.remove_on_arrival = 1;
    g.hist_v = reinterpret_cast<float2 *>(ws.hist_v);
    g.err_acc = ws.err_acc; g.err_cnt = ws.err_cnt;
    const float2 *pos = reinterpret_cast<const float2 *>(w->pos_tm), *vel = reinterpret_cast<const float2 *>(w->vel_tm);
    const float2 *acc = reinterpret_cast<const float2 *>(w->acc_tm), *dst = reinterpret_cast<const float2 *>(w->dest_tm);
    for (int t = w->t_start; t < w->T; ++t) {
        // a_next = model(*state_features)[0]                                           (simulators.py:602)
        rc = sfm_forward_sets_launch(w->params, N, ws.ped_f, ws.obs_f, ws.self_f, SN, kp, ko, ws.a_next, st);
        if (rc) return rc;
        // record, score, Euler, arrival / waypoint switch, entry from the clip at t+1      (:596-639)
        const int64_t f = static_cast<int64_t>(t) * N, f1 = f + N, q = static_cast<int64_t>(t) * SN;
        const bool last = t >= w->T - 1;
        g.entry = last ? nullptr : w->entry_tm + f1;
        g.p_gt = last ? nullptr : pos + f1; g.v_gt = last ? nullptr : vel + f1;
        g.a_gt = last ? nullptr : acc + f1; g.dest_gt = last ? nullptr : dst + f1;
        g.dest_idx_gt = last ? nullptr : w->dest_idx_tm + f1;
        g.score_p = pos + f; g.score_mask = w->mask_p + f;
        if (w->rec_p) {
            g.rec_p = reinterpret_cast<float2 *>(w->rec_p) + q; g.rec_v = reinterpret_cast<float2 *>(w->rec_v) + q;
            g.rec_a = reinterpret_cast<float2 *>(w->rec_a) + q; g.rec_mask = w->rec_mask + q;
        }
        rc = integrate_sweep_launch(g, st);
        if (rc) return rc;
        // features of the new state + self_features, at most SWEEP_FEATURE_SETS sets per call       (:642-652)
        for (int s0 = 0; s0 < S; s0 += SWEEP_FEATURE_SETS) {
            const int n = S - s0 < SWEEP_FEATURE_SETS ? S - s0 : SWEEP_FEATURE_SETS;
            const int64_t r0 = static_cast<int64_t>(s0) * N;
            rc = piml_state_features_f32(ws.p + 2 * r0, ws.v + 2 * r0, ws.a + 2 * r0, ws.dest + 2 * r0, w->obstacles,
                                         0, n, N, w->M, w->kp, w->cos_p, w->thr_p, w->ko, w->cos_o, w->thr_o,
                                         ws.hist_v + 2 * r0, ws.ds + r0, ws.ped_f + 6 * kp * r0,
                                         ws.obs_f ? ws.obs_f + 6 * ko * r0 : nullptr, ws.self_f + 7 * r0,
                                         ws.dest_f + 2 * r0, st);
            if (rc) return rc;
        }
    }
    return PIML_OK;
}

}  // namespace piml

using namespace piml;

extern "C" int64_t piml_sfm_sweep_workspace_bytes(const piml_sfm_sweep_args *w) {
    if (!w || w->S < 0 || w->N < 1 || w->M < 0 || w->kp < 0 || w->ko < 0) return -1;
    return sweep_layout(w, sweep_persistent(w), nullptr);
}

extern "C" int piml_sfm_sweep_f32(const piml_sfm_sweep_args *w, void *stream) {
    PIML_REQUIRE(w, "piml_sfm_sweep_f32: null arguments");
    PIML_REQUIRE(w->S >= 0 && w->N >= 1 && w->T >= 1 && w->D >= 1 && w->M >= 0 && w->t_start >= 0 &&
                     w->t_start < w->T && w->kp >= 0 && w->ko >= 0,
                 "piml_sfm_sweep_f32: bad dimensions S=%d N=%d T=%d D=%d M=%d t_start=%d kp=%d ko=%d", w->S, w->N,
                 w->T, w->D, w->M, w->t_start, w->kp, w->ko);
    if (w->S == 0) return PIML_OK;
    PIML_REQUIRE(w->pos_tm && w->vel_tm && w->acc_tm && w->dest_tm && w->dest_idx_tm && w->entry_tm && w->mask_p &&
                     w->dest_num && w->waypoints && w->desired_speed,
                 "piml_sfm_sweep_f32: null ground-truth / static input");
    const int ko = w->M > 0 ? (w->ko < w->M ? w->ko : w->M) : 0;
    PIML_REQUIRE(w->p && w->v && w->a && w->dest && w->dest_idx && w->ped_f && w->self_f &&
                     (w->M == 0 || w->obstacles) && (ko == 0 || w->obs_f),
                 "piml_sfm_sweep_f32: null initial state / features");
    PIML_REQUIRE(w->params && w->err_sum && w->err_count, "piml_sfm_sweep_f32: null constants / score output");
    const bool rec = w->rec_p || w->rec_v || w->rec_a || w->rec_mask;
    PIML_REQUIRE(!rec || (w->rec_p && w->rec_v && w->rec_a && w->rec_mask),
                 "piml_sfm_sweep_f32: record outputs must be all given or all NULL");
    const bool persistent = sweep_persistent(w);
    SweepWs ws;
    const int64_t need = sweep_layout(w, persistent, &ws);
    PIML_REQUIRE(w->workspace && w->workspace_bytes >= need,
                 "piml_sfm_sweep_f32: workspace of %lld bytes, %lld needed (piml_sfm_sweep_workspace_bytes)",
                 static_cast<long long>(w->workspace_bytes), static_cast<long long>(need));
    PIML_REQUIRE((reinterpret_cast<uintptr_t>(w->workspace) & 255u) == 0, "piml_sfm_sweep_f32: workspace must be "
                 "256-byte aligned");
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int rc = persistent ? sfm_sweep_persistent_launch(w, ws.err_acc, ws.err_cnt, st) : sweep_per_step(w, ws, st);
    if (rc) return rc;
    const int threads = 128;
    sweep_score_kernel<<<static_cast<unsigned>((w->S + threads - 1) / threads), threads, 0, st>>>(
        ws.err_acc, ws.err_cnt, w->S, w->N, w->err_sum, w->err_count);
    count_launch();
    return check_launch("sweep_score_kernel");
}
