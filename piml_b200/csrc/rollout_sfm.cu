// rollout_sfm.cu -- persistent rollout kernel for the pure social-force model (BASELINE configs 2 and 5b).
//
// The whole `for t in range(t_start, T)` loop of BaseSimulator.get_multiple_rollouts (reference
// src/models/simulators.py:595-652) for GC-shaped scenes in ONE launch: one CTA per scene, 2-4 lanes per agent slot.
// Per step a thread evaluates the social-force model on its current features (sfm_common.cuh), applies the state update
// (integrate_common.cuh: lagged Euler, arrival / waypoint switch, teacher-forced entry from the time-major ground
// truth), publishes its new position in shared memory and rebuilds its own neighbour features against the scene's
// positions and obstacles in shared memory (the same exact-arithmetic gate and (distance, index) top-k as
// relative_features_kernel).  Agent state and features live in registers for all T steps: a step reads nothing but
// the entry data of frame t+1 from HBM and writes nothing but the recorded trajectory -- "one rollout step reads and
// writes agent state once" (north star (c)) -- and there is no launch per step (the per-step path is launch-bound at
// 31 us per step for one scene).  Results are bit-identical to the per-step path (piml_rollout_f32 with three launches
// per step), which remains the route for scenes with more than 256 slots or 2048 obstacle points and for more than
// two waves of scenes (measured: 19 us per step and CTA, dependent IEEE div / sqrt / exp chains and two CTA barriers).
// The SWEEP instantiation runs a constants sweep (sfm_sweep.cu): CTA s rolls the ONE clip under constant set s.
#include <stdlib.h>

#include "features_common.cuh"
#include "integrate_common.cuh"
#include "sfm_common.cuh"

namespace piml {

constexpr int RS_THREADS = 512;                   // threads per CTA = lanes per agent x agent slots
constexpr int RS_MAXN = 256;                      // agent slots per scene (2 lanes each; 4 lanes up to 128 slots)
constexpr int RS_MAXM = 2048;                     // obstacle points per scene held in shared memory
constexpr int RS_KP = 8, RS_KO = 16;              // register top-k capacities (kp <= 8, ko <= 16)

struct SfmRollArgs {
    piml_sfm_params prm;
    int S, N, M, D, T, t_start; float dt;
    int kp, ko; float cos_p, thr_p, pre2_p, cos_o, thr_o, pre2_o;
    const float2 *obstacles; int obs_per_scene;
    const float2 *pos_tm, *vel_tm, *acc_tm, *dest_tm; const int64_t *dest_idx_tm, *entry_tm, *dest_num;
    const float2 *waypoints; const float *desired_speed;
    float2 *p, *v, *a, *dest; int64_t *dest_idx; float2 *hist_v;
    const float *ped_f, *obs_f, *self_f;          // features of the state at t_start
    float2 *rec_p, *rec_v, *rec_a; float *rec_mask;
    // constants sweep (SWEEP = true, sfm_sweep.cu): CTA s is constant set s of ONE clip, whose ground truth, initial
    // state and features have no scene axis; recording is optional and the positions are scored against the clip
    const piml_sfm_params *prm_sets;
    const float2 *score_pos; const float *score_mask;  // (T,N) the clip's positions and mask_p
    double *err_acc; int64_t *err_cnt;                 // (S,N) per-slot score, summed in time order
};

// G lanes per agent slot (threads per CTA = G * N <= RS_THREADS): a single warp per scheduler cannot hide the latency
// of the dependent IEEE div / sqrt / exp chains, so the slots of an agent (forward) and the candidates (feature
// rebuild) are spread over G lanes; sums are formed in slot order on every lane, so nothing changes numerically.
template <int G, bool SWEEP>
__global__ void __launch_bounds__(RS_THREADS) sfm_rollout_kernel(const __grid_constant__ SfmRollArgs r) {
    constexpr int PS = RS_KP / G, OS = RS_KO / G;               // slots per lane: slot j lives on lane j % G, [j / G]
    extern __shared__ __align__(16) float2 rs_smem[];
    float2 *spos = rs_smem;                                       // [N] current positions of the scene
    float2 *sobs = rs_smem + r.N;                                 // [M]
    const int s = blockIdx.x, n = threadIdx.x / G, g = threadIdx.x % G;
    const bool live = n < r.N;
    const int nn = live ? n : r.N - 1;                            // idle lanes shadow the last slot and never write
    const int64_t i = static_cast<int64_t>(s) * r.N + nn;
    const int64_t SN = static_cast<int64_t>(r.S) * r.N;
    const int64_t gi = SWEEP ? nn : i;                            // ground truth / initial state of the slot
    const int64_t GSN = SWEEP ? r.N : SN;                         // ... and of one frame
    piml_sfm_params set_prm;
    if constexpr (SWEEP) set_prm = r.prm_sets[s];
    const piml_sfm_params &prm = SWEEP ? set_prm : r.prm;
    const int kp = r.kp < r.N ? r.kp : r.N;
    const int ko = r.M > 0 ? (r.ko < r.M ? r.ko : r.M) : 0;
    const float2 *obs = r.obstacles + (r.obs_per_scene ? static_cast<int64_t>(s) * r.M : 0);
    for (int m = threadIdx.x; m < r.M; m += blockDim.x) sobs[m] = obs[m];

    // every lane of an agent's group carries the same state (the update is recomputed redundantly, lane 0 records)
    AgentState st{r.p[gi], r.v[gi], r.a[gi], r.dest[gi], r.dest_idx[gi], make_float2(0.f, 0.f)};
    const int64_t dnum = r.dest_num[gi];
    const float2 *wp = r.waypoints + (SWEEP ? 0 : static_cast<int64_t>(s) * r.D * r.N) + nn;
    double err = 0.0;
    int64_t err_n = 0;
    // features of the state at t_start, as handed over by the caller (data.ped_features[t_start] ...)
    float fx[PS], fy[PS], ox[OS], oy[OS];
#pragma unroll
    for (int q = 0; q < PS; ++q) {
        const int j = q * G + g;
        fx[q] = fy[q] = 0.f;
        if (j < kp) { fx[q] = r.ped_f[(gi * kp + j) * 6]; fy[q] = r.ped_f[(gi * kp + j) * 6 + 1]; }
    }
#pragma unroll
    for (int q = 0; q < OS; ++q) {
        const int j = q * G + g;
        ox[q] = oy[q] = 0.f;
        if (j < ko) { ox[q] = r.obs_f[(gi * ko + j) * 6]; oy[q] = r.obs_f[(gi * ko + j) * 6 + 1]; }
    }
    float dfx = r.self_f[gi * 7], dfy = r.self_f[gi * 7 + 1], hvx = r.self_f[gi * 7 + 2], hvy = r.self_f[gi * 7 + 3];
    float v0 = r.self_f[gi * 7 + 6];
    const float v0_later = r.desired_speed[gi];
    __syncthreads();

    for (int t = r.t_start; t < r.T; ++t) {
        // ---- a_next = model(*state_features)[0]                                            (simulators.py:602)
        float2 pm[PS], om[OS];
#pragma unroll
        for (int q = 0; q < PS; ++q)
            pm[q] = (q * G + g < kp) ? sfm_v0(fx[q], fy[q], prm.A_ped, prm.B_ped, prm.eps) : make_float2(0.f, 0.f);
#pragma unroll
        for (int q = 0; q < OS; ++q)
            om[q] = (q * G + g < ko) ? sfm_v0(ox[q], oy[q], prm.A_obs, prm.B_obs, prm.eps) : make_float2(0.f, 0.f);
        float ax = 0.f, ay = 0.f, bx = 0.f, by = 0.f;              // slot order, like torch.sum over dim -2
#pragma unroll
        for (int j = 0; j < RS_KP; ++j) {
            if (j >= kp) break;                                   // uniform
            const float mx = __shfl_sync(0xffffffffu, pm[j / G].x, j % G, G);
            const float my = __shfl_sync(0xffffffffu, pm[j / G].y, j % G, G);
            ax = __fadd_rn(ax, mx); ay = __fadd_rn(ay, my);
        }
#pragma unroll
        for (int j = 0; j < RS_KO; ++j) {
            if (j >= ko) break;
            const float mx = __shfl_sync(0xffffffffu, om[j / G].x, j % G, G);
            const float my = __shfl_sync(0xffffffffu, om[j / G].y, j % G, G);
            bx = __fadd_rn(bx, mx); by = __fadd_rn(by, my);
        }
        const float2 a_next = sfm_total(ax, ay, bx, by, dfx, dfy, hvx, hvy, v0, prm.tau);
        // ---- record the state at t, update, teacher-forced entry                           (:596-639)
        const int64_t q0 = static_cast<int64_t>(t) * SN + i;
        if (live && g == 0 && (!SWEEP || r.rec_p)) {
            r.rec_p[q0] = st.p; r.rec_v[q0] = st.v; r.rec_a[q0] = st.a;
            if (!(st.p.x != st.p.x)) r.rec_mask[q0] = 1.0f;
        }
        if constexpr (SWEEP) {
            const int64_t c = static_cast<int64_t>(t) * r.N + nn;
            sweep_err_term(st.p, r.score_pos[c], r.score_mask[c], err, err_n);
        }
        integrate_update(st, a_next, r.dt, 1, dnum, wp, r.N);
        if (t < r.T - 1) {
            const int64_t o = static_cast<int64_t>(t + 1) * GSN + gi;
            if (r.entry_tm[o] == 1) {
                st.p = r.pos_tm[o]; st.v = r.vel_tm[o]; st.a = r.acc_tm[o]; st.dest = r.dest_tm[o];
                st.di = r.dest_idx_tm[o];
                st.hv = st.v;
            }
        }
        // ---- features of the new state                                                     (:642-652, data.py:466-512)
        __syncthreads();                                          // everyone has finished reading the old positions
        if (live && g == 0) spos[n] = st.p;
        __syncthreads();
        st.v = make_float2(nan_to_zero(st.v.x), nan_to_zero(st.v.y));          // in place, data.py:483-484
        st.a = make_float2(nan_to_zero(st.a.x), nan_to_zero(st.a.y));
        float2 h;
        {
            float nv = norm2_rn(st.v.x, st.v.y);
            if (nv == 0.0f) nv = 0.1f;
            h = make_float2(__fdiv_rn(st.v.x, nv), __fdiv_rn(st.v.y, nv));
            const float nh = fmaxf(norm2_rn(h.x, h.y), 1e-8f);
            h = make_float2(__fdiv_rn(h.x, nh), __fdiv_rn(h.y, nh));
        }
        {
            TopK<RS_KP> best;
            best.init();
            for (int m = g; m < r.N; m += G) {
                const float2 o = spos[m];
                const float rx = __fsub_rn(o.x, st.p.x), ry = __fsub_rn(o.y, st.p.y);
                if (!(__fmaf_rn(ry, ry, __fmul_rn(rx, rx)) <= r.pre2_p)) continue;
                const float d = gated_distance(rx, ry, h.x, h.y, r.cos_p);
                if (d <= r.thr_p) best.insert(make_key(d, m));
            }
#pragma unroll
            for (int j = 0; j < RS_KP; ++j) {                     // merge the G lists: k smallest keys, smallest first
                if (j >= kp) break;                               // uniform: slots beyond kp stay zero
                const uint64_t w = group_min<G>(best.key[0]);
                if (w != EMPTY_KEY && best.key[0] == w) best.pop_front();
                if (j % G == g) {
                    fx[j / G] = fy[j / G] = 0.f;
                    if (j < kp && w != EMPTY_KEY) {
                        const float2 pmm = spos[key_idx(w)];
                        fx[j / G] = __fsub_rn(pmm.x, st.p.x); fy[j / G] = __fsub_rn(pmm.y, st.p.y);
                    }
                }
            }
        }
        if (r.M > 0) {
            TopK<RS_KO> best;
            best.init();
            for (int m = g; m < r.M; m += G) {
                const float2 o = sobs[m];
                const float rx = __fsub_rn(o.x, st.p.x), ry = __fsub_rn(o.y, st.p.y);
                if (!(__fmaf_rn(ry, ry, __fmul_rn(rx, rx)) <= r.pre2_o)) continue;
                const float d = gated_distance(rx, ry, h.x, h.y, r.cos_o);
                if (d <= r.thr_o) best.insert(make_key(d, m));
            }
#pragma unroll
            for (int j = 0; j < RS_KO; ++j) {
                if (j >= ko) break;
                const uint64_t w = group_min<G>(best.key[0]);
                if (w != EMPTY_KEY && best.key[0] == w) best.pop_front();
                if (j % G == g) {
                    ox[j / G] = oy[j / G] = 0.f;
                    if (j < ko && w != EMPTY_KEY) {
                        const float2 omm = sobs[key_idx(w)];
                        ox[j / G] = __fsub_rn(omm.x, st.p.x); oy[j / G] = __fsub_rn(omm.y, st.p.y);
                    }
                }
            }
        }
        dfx = nan_to_zero(__fsub_rn(st.dest.x, st.p.x));                       // data.py:496-497
        dfy = nan_to_zero(__fsub_rn(st.dest.y, st.p.y));
        hvx = st.hv.x; hvy = st.hv.y;
        v0 = v0_later;
    }
    if (live && g == 0) {
        if constexpr (SWEEP) {
            r.err_acc[i] = err; r.err_cnt[i] = err_n;
        } else {                                                  // leave the state buffers as the per-step path does
            r.p[i] = st.p; r.v[i] = st.v; r.a[i] = st.a; r.dest[i] = st.dest; r.dest_idx[i] = st.di;
            r.hist_v[i] = st.hv;
        }
    }
}

// Whether the persistent kernel may run S scenes (or constant sets) of these sizes (PIML_SFM_PERSISTENT=0 disables
// it, =2 forces it whatever S is).
bool sfm_persistent_fits(int S, int N, int M, int kp_, int ko_, float thr_p, float thr_o) {
    const char *e = getenv("PIML_SFM_PERSISTENT");                 // read per call: tests compare both routes
    const bool off = e && atoi(e) == 0;
    const int kp = kp_ < N ? kp_ : N;
    const int ko = M > 0 ? (ko_ < M ? ko_ : M) : 0;
    // one CTA per scene and one resident CTA per SM: latency-bound at ~19 us per step whatever S is, so it wins up to
    // about two waves of scenes (S = 64: 6.2 vs 15.4 ms per 300-step rollout; S = 4096: the per-step route's
    // throughput-bound 0.45 ms per step wins)
    if (S > 2 * sm_count() && !(e && atoi(e) == 2)) return false;
    return !off && N <= RS_MAXN && M <= RS_MAXM && kp <= RS_KP && ko <= RS_KO &&
           thr_p > 0.f && thr_p < 1e18f && (M == 0 || (thr_o > 0.f && thr_o < 1e18f));
}

// Whether piml_rollout_f32 may use the persistent kernel.
bool sfm_rollout_fits(const piml_rollout_args *r) {
    return r->sfm && sfm_persistent_fits(r->S, r->N, r->M, r->kp, r->ko, r->thr_p, r->thr_o);
}

template <bool SWEEP>
static int sfm_rollout_launch_args(const SfmRollArgs &a, cudaStream_t st) {
    const int G = a.N * 4 <= RS_THREADS ? 4 : 2;
    const int threads = (a.N * G + 31) / 32 * 32;
    const size_t smem = sizeof(float2) * (a.N + a.M);
    if (G == 4) sfm_rollout_kernel<4, SWEEP><<<static_cast<unsigned>(a.S), threads, smem, st>>>(a);
    else sfm_rollout_kernel<2, SWEEP><<<static_cast<unsigned>(a.S), threads, smem, st>>>(a);
    count_launch();
    return check_launch("sfm_rollout_kernel");
}

int sfm_rollout_launch(const piml_rollout_args *r, cudaStream_t st) {
    SfmRollArgs a;
    a.prm = *r->sfm;
    a.S = r->S; a.N = r->N; a.M = (r->has_obs && r->M > 0) ? r->M : 0; a.D = r->D; a.T = r->T; a.t_start = r->t_start;
    a.dt = r->dt; a.kp = r->kp; a.ko = r->ko;
    a.cos_p = r->cos_p; a.thr_p = r->thr_p; a.pre2_p = prefilter_sq(r->thr_p);
    a.cos_o = r->cos_o; a.thr_o = r->thr_o; a.pre2_o = prefilter_sq(r->thr_o);
    a.obstacles = reinterpret_cast<const float2 *>(r->obstacles); a.obs_per_scene = r->obs_per_scene;
    a.pos_tm = reinterpret_cast<const float2 *>(r->pos_tm); a.vel_tm = reinterpret_cast<const float2 *>(r->vel_tm);
    a.acc_tm = reinterpret_cast<const float2 *>(r->acc_tm); a.dest_tm = reinterpret_cast<const float2 *>(r->dest_tm);
    a.dest_idx_tm = r->dest_idx_tm; a.entry_tm = r->entry_tm; a.dest_num = r->dest_num;
    a.waypoints = reinterpret_cast<const float2 *>(r->waypoints); a.desired_speed = r->desired_speed;
    a.p = reinterpret_cast<float2 *>(r->p); a.v = reinterpret_cast<float2 *>(r->v); a.a = reinterpret_cast<float2 *>(r->a);
    a.dest = reinterpret_cast<float2 *>(r->dest); a.dest_idx = r->dest_idx; a.hist_v = reinterpret_cast<float2 *>(r->hist_v);
    a.ped_f = r->ped_f; a.obs_f = r->obs_f; a.self_f = r->self_f;
    a.rec_p = reinterpret_cast<float2 *>(r->rec_p); a.rec_v = reinterpret_cast<float2 *>(r->rec_v);
    a.rec_a = reinterpret_cast<float2 *>(r->rec_a); a.rec_mask = r->rec_mask;
    return sfm_rollout_launch_args<false>(a, st);
}

// The constants sweep on the persistent kernel: CTA s rolls the clip under w->params[s] and leaves its slots' scores
// in err_acc / err_cnt (S,N).  The initial state is read, never written.
int sfm_sweep_persistent_launch(const piml_sfm_sweep_args *w, double *err_acc, int64_t *err_cnt, cudaStream_t st) {
    SfmRollArgs a = {};
    a.S = w->S; a.N = w->N; a.M = w->M; a.D = w->D; a.T = w->T; a.t_start = w->t_start;
    a.dt = w->dt; a.kp = w->kp; a.ko = w->ko;
    a.cos_p = w->cos_p; a.thr_p = w->thr_p; a.pre2_p = prefilter_sq(w->thr_p);
    a.cos_o = w->cos_o; a.thr_o = w->thr_o; a.pre2_o = prefilter_sq(w->thr_o);
    a.obstacles = reinterpret_cast<const float2 *>(w->obstacles); a.obs_per_scene = 0;
    a.pos_tm = reinterpret_cast<const float2 *>(w->pos_tm); a.vel_tm = reinterpret_cast<const float2 *>(w->vel_tm);
    a.acc_tm = reinterpret_cast<const float2 *>(w->acc_tm); a.dest_tm = reinterpret_cast<const float2 *>(w->dest_tm);
    a.dest_idx_tm = w->dest_idx_tm; a.entry_tm = w->entry_tm; a.dest_num = w->dest_num;
    a.waypoints = reinterpret_cast<const float2 *>(w->waypoints); a.desired_speed = w->desired_speed;
    // read only in the sweep instantiation
    a.p = const_cast<float2 *>(reinterpret_cast<const float2 *>(w->p));
    a.v = const_cast<float2 *>(reinterpret_cast<const float2 *>(w->v));
    a.a = const_cast<float2 *>(reinterpret_cast<const float2 *>(w->a));
    a.dest = const_cast<float2 *>(reinterpret_cast<const float2 *>(w->dest));
    a.dest_idx = const_cast<int64_t *>(w->dest_idx);
    a.ped_f = w->ped_f; a.obs_f = w->obs_f; a.self_f = w->self_f;
    a.rec_p = reinterpret_cast<float2 *>(w->rec_p); a.rec_v = reinterpret_cast<float2 *>(w->rec_v);
    a.rec_a = reinterpret_cast<float2 *>(w->rec_a); a.rec_mask = w->rec_mask;
    a.prm_sets = w->params;
    a.score_pos = reinterpret_cast<const float2 *>(w->pos_tm); a.score_mask = w->mask_p;
    a.err_acc = err_acc; a.err_cnt = err_cnt;
    return sfm_rollout_launch_args<true>(a, st);
}

}  // namespace piml
