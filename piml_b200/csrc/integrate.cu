// integrate.cu -- fused rollout state update for sm_100a.
//
// Replaces the elementwise / gather / masked-write chain of BaseSimulator.get_multiple_rollouts
// (reference src/models/simulators.py:596-639, ~25 eager launches and 5 host syncs per step) by one kernel: record
// the state at t, lagged explicit Euler, arrival / waypoint switch, removal on arrival, teacher-forced entry and the
// history-velocity update.  One thread per (scene, slot); state is read and written once.
#include "integrate_common.cuh"

namespace piml {

template <bool SWEEP = false>
__device__ __forceinline__ void integrate_body(const IntArgs &g) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<int64_t>(g.S) * g.N) return;
    integrate_agent<SWEEP>(g, i, g.a_next[i]);
}

__global__ void integrate_kernel(IntArgs g) { integrate_body(g); }

// The step of a constants sweep (sfm_sweep.cu): S sets of one clip, whose ground truth has no scene axis; the
// recorded position is added to the slot's score.
__global__ void integrate_sweep_kernel(IntArgs g) { integrate_body<true>(g); }

// The same step with the frame index read from device memory: `g` carries the BASE pointers of the time-major
// ground-truth / record arrays, frame t = *t_dev selects the slices (record into frame t, entries from frame t + 1).
// Every launch of a rollout step then has constant arguments, so one captured CUDA graph replays the whole loop
// (rollout.cu); a one-thread kernel advances the counter at the end of the step.
__global__ void integrate_indirect_kernel(IntArgs g, const int *__restrict__ t_dev) {
    const int t = *t_dev;
    const int64_t SN = static_cast<int64_t>(g.S) * g.N;
    g.entry += (t + 1) * SN; g.dest_idx_gt += (t + 1) * SN;
    g.p_gt += (t + 1) * SN; g.v_gt += (t + 1) * SN; g.a_gt += (t + 1) * SN; g.dest_gt += (t + 1) * SN;
    g.rec_p += t * SN; g.rec_v += t * SN; g.rec_a += t * SN; g.rec_mask += t * SN;
    integrate_body(g);
}

__global__ void advance_counter_kernel(int *t_dev) { *t_dev += 1; }

// rollout.cu: one step of the captured loop (frames t_start + 1 .. T - 2 all have a successor frame to enter from)
int integrate_step_indirect(const piml_rollout_args *r, const int *t_dev, cudaStream_t st) {
    IntArgs g;
    g.p = reinterpret_cast<float2 *>(r->p); g.v = reinterpret_cast<float2 *>(r->v); g.a = reinterpret_cast<float2 *>(r->a);
    g.a_next = reinterpret_cast<const float2 *>(r->a_next); g.dest = reinterpret_cast<float2 *>(r->dest);
    g.dest_idx = r->dest_idx; g.dest_num = r->dest_num; g.waypoints = reinterpret_cast<const float2 *>(r->waypoints);
    g.S = r->S; g.D = r->D; g.N = r->N; g.dt = r->dt; g.remove_on_arrival = 1; g.entry = r->entry_tm;
    g.p_gt = reinterpret_cast<const float2 *>(r->pos_tm); g.v_gt = reinterpret_cast<const float2 *>(r->vel_tm);
    g.a_gt = reinterpret_cast<const float2 *>(r->acc_tm); g.dest_gt = reinterpret_cast<const float2 *>(r->dest_tm);
    g.dest_idx_gt = r->dest_idx_tm; g.hist_v = reinterpret_cast<float2 *>(r->hist_v);
    g.rec_p = reinterpret_cast<float2 *>(r->rec_p); g.rec_v = reinterpret_cast<float2 *>(r->rec_v);
    g.rec_a = reinterpret_cast<float2 *>(r->rec_a); g.rec_mask = r->rec_mask;
    const int64_t tot = static_cast<int64_t>(r->S) * r->N;
    const int threads = 128;
    integrate_indirect_kernel<<<static_cast<unsigned>((tot + threads - 1) / threads), threads, 0, st>>>(g, t_dev);
    count_launch();
    return check_launch("integrate_indirect_kernel");
}

int integrate_sweep_launch(const IntArgs &g, cudaStream_t st) {
    const int64_t tot = static_cast<int64_t>(g.S) * g.N;
    const int threads = 128;
    integrate_sweep_kernel<<<static_cast<unsigned>((tot + threads - 1) / threads), threads, 0, st>>>(g);
    count_launch();
    return check_launch("integrate_sweep_kernel");
}

int advance_counter(int *t_dev, cudaStream_t st) {
    advance_counter_kernel<<<1, 1, 0, st>>>(t_dev);
    count_launch();
    return check_launch("advance_counter_kernel");
}

// backward of v' = v + a dt, p' = p + v dt, a' = a_next with teacher-forced entry (simulators.py:741-769)
__global__ void integrate_bwd_kernel(const int64_t *__restrict__ entry, int64_t n, float dt,
                                     const float2 *__restrict__ g_p2, const float2 *__restrict__ g_v2,
                                     const float2 *__restrict__ g_a2, float2 *__restrict__ g_p,
                                     float2 *__restrict__ g_v, float2 *__restrict__ g_a, float2 *__restrict__ g_an) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float2 gp = g_p2[i], gv = g_v2[i], ga = g_a2[i];
    if (entry && entry[i] == 1) gp = gv = ga = make_float2(0.f, 0.f);           // overwritten from the data
    g_p[i] = gp;
    g_v[i] = make_float2(fmaf(gp.x, dt, gv.x), fmaf(gp.y, dt, gv.y));
    g_a[i] = make_float2(gv.x * dt, gv.y * dt);
    g_an[i] = ga;
}

}  // namespace piml

using namespace piml;

extern "C" int piml_integrate_step_f32(float *p, float *v, float *a, const float *a_next, float *dest,
                                       int64_t *dest_idx, const int64_t *dest_num, const float *waypoints, int S,
                                       int D, int N, float dt, int remove_on_arrival, const int64_t *entry,
                                       const float *p_gt, const float *v_gt, const float *a_gt, const float *dest_gt,
                                       const int64_t *dest_idx_gt, float *hist_v, float *rec_p, float *rec_v,
                                       float *rec_a, float *rec_mask, void *stream) {
    PIML_REQUIRE(p && v && a && a_next && dest && dest_idx && dest_num && waypoints,
                 "piml_integrate_step_f32: null pointer");
    PIML_REQUIRE(S >= 0 && D >= 1 && N >= 0, "piml_integrate_step_f32: bad dimensions S=%d D=%d N=%d", S, D, N);
    PIML_REQUIRE(!entry || (p_gt && v_gt && a_gt && dest_gt && dest_idx_gt),
                 "piml_integrate_step_f32: entry mask given without ground-truth arrays");
    const int64_t tot = static_cast<int64_t>(S) * N;
    if (tot == 0) return PIML_OK;
    IntArgs g;
    g.p = reinterpret_cast<float2 *>(p); g.v = reinterpret_cast<float2 *>(v); g.a = reinterpret_cast<float2 *>(a);
    g.a_next = reinterpret_cast<const float2 *>(a_next); g.dest = reinterpret_cast<float2 *>(dest);
    g.dest_idx = dest_idx; g.dest_num = dest_num; g.waypoints = reinterpret_cast<const float2 *>(waypoints);
    g.S = S; g.D = D; g.N = N; g.dt = dt; g.remove_on_arrival = remove_on_arrival; g.entry = entry;
    g.p_gt = reinterpret_cast<const float2 *>(p_gt); g.v_gt = reinterpret_cast<const float2 *>(v_gt);
    g.a_gt = reinterpret_cast<const float2 *>(a_gt); g.dest_gt = reinterpret_cast<const float2 *>(dest_gt);
    g.dest_idx_gt = dest_idx_gt; g.hist_v = reinterpret_cast<float2 *>(hist_v);
    g.rec_p = reinterpret_cast<float2 *>(rec_p); g.rec_v = reinterpret_cast<float2 *>(rec_v);
    g.rec_a = reinterpret_cast<float2 *>(rec_a); g.rec_mask = rec_mask;
    const int threads = 128;
    integrate_kernel<<<static_cast<unsigned>((tot + threads - 1) / threads), threads, 0,
                       static_cast<cudaStream_t>(stream)>>>(g);
    count_launch();
    return check_launch("integrate_kernel");
}

extern "C" int piml_integrate_step_backward_f32(const int64_t *entry, int64_t n, float dt, const float *g_p2,
                                                const float *g_v2, const float *g_a2, float *g_p, float *g_v,
                                                float *g_a, float *g_a_next, void *stream) {
    PIML_REQUIRE(g_p2 && g_v2 && g_a2 && g_p && g_v && g_a && g_a_next, "piml_integrate_step_backward_f32: null pointer");
    PIML_REQUIRE(n >= 0, "piml_integrate_step_backward_f32: negative size");
    if (n == 0) return PIML_OK;
    const int threads = 128;
    integrate_bwd_kernel<<<static_cast<unsigned>((n + threads - 1) / threads), threads, 0,
                           static_cast<cudaStream_t>(stream)>>>(
        entry, n, dt, reinterpret_cast<const float2 *>(g_p2), reinterpret_cast<const float2 *>(g_v2),
        reinterpret_cast<const float2 *>(g_a2), reinterpret_cast<float2 *>(g_p), reinterpret_cast<float2 *>(g_v),
        reinterpret_cast<float2 *>(g_a), reinterpret_cast<float2 *>(g_a_next));
    count_launch();
    return check_launch("integrate_bwd_kernel");
}
