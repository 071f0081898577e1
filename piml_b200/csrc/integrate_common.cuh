// integrate_common.cuh -- one agent's state update of get_multiple_rollouts (simulators.py:603-626), shared by
// integrate_kernel and the persistent rollout kernel (rollout_sfm.cu).
#pragma once
#include <math_constants.h>

#include "common.cuh"

namespace piml {

struct AgentState { float2 p, v, a, dest; int64_t di; float2 hv; };

// Lagged explicit Euler with the OLD a and v, arrival / waypoint switch, removal on arrival.  `wp` points at
// waypoints[scene][0][n]; consecutive waypoints of the agent are `wp_stride` float2 apart.
__device__ __forceinline__ void integrate_update(AgentState &s, float2 a_next, float dt, int remove_on_arrival,
                                                 int64_t dest_num, const float2 *__restrict__ wp, int64_t wp_stride) {
    // v_next = v + a*dt ; p_next = p + v*dt                                   (simulators.py:603-604)
    const float2 vn = make_float2(__fadd_rn(s.v.x, __fmul_rn(s.a.x, dt)), __fadd_rn(s.v.y, __fmul_rn(s.a.y, dt)));
    float2 pn = make_float2(__fadd_rn(s.p.x, __fmul_rn(s.v.x, dt)), __fadd_rn(s.p.y, __fmul_rn(s.v.y, dt)));
    int64_t di = s.di;
    const float dis = norm2_rn(__fsub_rn(s.p.x, s.dest.x), __fsub_rn(s.p.y, s.dest.y));   // :608
    if (dis < 0.5f) di += 1;                                                   // :609
    if (di > dest_num - 1) {
        if (remove_on_arrival) pn = make_float2(CUDART_NAN_F, CUDART_NAN_F);   // :611
        di -= 1;                                                               // :613
    }
    s.dest = wp[di * wp_stride];                                               // :614-616
    s.p = pn; s.v = vn; s.a = a_next; s.di = di;
    s.hv = vn;                                                                 // :624-626
}

// One term of a constants sweep's score (sfm_sweep.cu): ||p - q||_2 in float64 where the simulated position p is not
// NaN (the rollout records mask 1 there) and the clip's mask_p is 1.  Explicit roundings: both routes of the sweep
// call this and must agree bit for bit.
__device__ __forceinline__ void sweep_err_term(float2 p, float2 q, float mask_p, double &sum, int64_t &count) {
    if (p.x != p.x || mask_p != 1.0f) return;
    const double dx = __dsub_rn(static_cast<double>(p.x), static_cast<double>(q.x));
    const double dy = __dsub_rn(static_cast<double>(p.y), static_cast<double>(q.y));
    sum = __dadd_rn(sum, __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))));
    count += 1;
}

// One thread's whole step of integrate_kernel (integrate.cu) / nn_finish_integrate_kernel (nn_step.cu): record the
// state at t, update, teacher-forced entry from the data at t + 1, history velocity.  simulators.py:596-639.
struct IntArgs {
    float2 *p, *v, *a; const float2 *a_next; float2 *dest; int64_t *dest_idx; const int64_t *dest_num;
    const float2 *waypoints; int S, D, N; float dt; int remove_on_arrival;
    const int64_t *entry; const float2 *p_gt, *v_gt, *a_gt, *dest_gt; const int64_t *dest_idx_gt;
    float2 *hist_v; float2 *rec_p, *rec_v, *rec_a; float *rec_mask;
    // constants sweep only (SWEEP = true): entry / *_gt / dest_num / waypoints are the ONE clip's (no scene axis), and
    // the recorded position is scored against the clip's frame t
    const float2 *score_p; const float *score_mask; double *err_acc; int64_t *err_cnt;
};

struct AgentNext { float2 p, v, a, dest, hv; int64_t di; };

// reads agent i's state, records it, returns the updated state (nothing of the state is written)
template <bool SWEEP = false>
__device__ __forceinline__ AgentNext integrate_agent_compute(const IntArgs &g, int64_t i, float2 a_next) {
    const int s = static_cast<int>(i / g.N), n = static_cast<int>(i % g.N);
    const int64_t gi = SWEEP ? n : i;                                          // the slot's ground truth
    const float2 p = g.p[i], v = g.v[i], a = g.a[i];
    // p_res[t] = p_cur ... mask_p_new[t][~isnan(p.x)] = 1          (simulators.py:596-600)
    if (g.rec_p) g.rec_p[i] = p;
    if (g.rec_v) g.rec_v[i] = v;
    if (g.rec_a) g.rec_a[i] = a;
    if (g.rec_mask && !(p.x != p.x)) g.rec_mask[i] = 1.0f;
    if constexpr (SWEEP) {
        double e = g.err_acc[i];
        int64_t c = g.err_cnt[i];
        sweep_err_term(p, g.score_p[n], g.score_mask[n], e, c);
        g.err_acc[i] = e; g.err_cnt[i] = c;
    }
    AgentState st{p, v, a, g.dest[i], g.dest_idx[i], make_float2(0.f, 0.f)};
    integrate_update(st, a_next, g.dt, g.remove_on_arrival, g.dest_num[gi],
                     g.waypoints + (SWEEP ? 0 : static_cast<int64_t>(s) * g.D * g.N) + n, g.N);
    AgentNext o{st.p, st.v, st.a, st.dest, st.hv, st.di};
    if (g.entry && g.entry[gi] == 1) {                                         // :629-639
        o.p = g.p_gt[gi]; o.v = g.v_gt[gi]; o.a = g.a_gt[gi]; o.dest = g.dest_gt[gi]; o.di = g.dest_idx_gt[gi];
        o.hv = o.v;
    }
    return o;
}

template <bool SWEEP = false>
__device__ __forceinline__ void integrate_agent(const IntArgs &g, int64_t i, float2 a_next) {
    const AgentNext o = integrate_agent_compute<SWEEP>(g, i, a_next);
    g.p[i] = o.p; g.v[i] = o.v; g.a[i] = o.a; g.dest[i] = o.dest; g.dest_idx[i] = o.di;
    if (g.hist_v) g.hist_v[i] = o.hv;
}

}  // namespace piml
