// nn_step.cu -- one NN-augmented rollout step as ONE C call and 7 launches: the body of the loop of
// BaseSimulator.get_multiple_rollouts (reference src/models/simulators.py:595-652) re-ordered around the state,
//     features(state_t) -> a_next = model(features) -> record / Euler / arrival / entry -> state_{t+1},
// for large crowds (cell list) and the per-slot-decoder networks the 16-bit tensor-core kernel runs (pinnsf_bm,
// pinnsf_bottleneck; model.py:1104-1135, :1185-1221).
//
// What is fused compared with the three-call route (piml_state_features_f32 -> piml_pinnsf_forward_tc_f32 ->
// piml_integrate_step_f32; 10 kernels + 2 memsets per step):
//   * the feature kernel (features_cells.cu, sorted order, 4 lanes per agent) emits the NON-EMPTY slot rows directly in
//     the compact layout the tensor-core kernel consumes, plus a slot -> row map: the dense (N,k,6) feature tensors are
//     not written and re-read (384 + 420 B per agent-step), and the separate compaction pass is gone;
//   * pinnsf_tc16_kernel reads those rows contiguously (no index list, no gather);
//   * nn_finish_integrate_kernel forms the slot sums (in slot order, f(0) for empty slots: the same additions in the
//     same order as the dense evaluation), adds the destination term (model.py:1205-1210) and applies the state update
//     of integrate_kernel in the same thread: the model output never round-trips through HBM between two launches;
//   * the cell-list build needs no memset and 4 launches (fused scan, counters zeroed by their reader).
//   * empty slots are not represented at all: a per-agent live-slot count (the live slots are a prefix of an agent's
//     slots) replaces map entries, and warps none of whose agents has a position skip the search (batches of mostly
//     empty scenes).
// Results are bit-identical to the three-call route (tests/test_gpu_nn_step.py; scripts/fuzz_parity.py family 5).
// piml_nn_step_shard_f32 is the same chain for one rank of an agent-sharded crowd: own agents only, new p, v, a stored
// into every rank's next-state arrays over NVLink peer memory by the finish kernel.
#include "features_common.cuh"
#include "integrate_common.cuh"
#include "mlp_tc16.cuh"

namespace piml {

struct FinishArgs {
    const float *cmsg_ped, *cmsg_obs;          // per compact row (2)
    const int *map_ped, *map_obs;              // (S*N, kp), (S*N, ko): compact row of each LIVE slot
    const uint16_t *live;                      // (S*N): live pedestrian | obstacle << 8 slots (a prefix of the slots)
    const float *f0;                           // [2][2] message of a zero row per branch
    const float *desired_speed;
    int kp, ko, has_obs; float tau;
    float2 *a_out;                             // optional copy of the model output
    int *counts;                               // the compact-row counters: zeroed here for the next step
};

// acc = sum over the k slots (slot order, f(0) for the empty ones) of both branches + destination term: the arithmetic
// of pinnsf_tc_finish_compact_kernel (mlp_tc.cu) for both components.
__device__ __forceinline__ float2 nn_agent_output(const IntArgs &g, const FinishArgs &f, int64_t i) {
    const float2 p = g.p[i], d = g.dest[i], hv = g.hist_v[i];
    const float ds = f.desired_speed[i];
    // self features: dest_f = nan_to_zero(dest - p) (data.py:502-503), hist_v, desired speed (simulators.py:651)
    const float sf0 = nan_to_zero(__fsub_rn(d.x, p.x)), sf1 = nan_to_zero(__fsub_rn(d.y, p.y));
    float nrm = norm2_rn(sf0, sf1);
    if (nrm == 0.f) nrm = __fadd_rn(nrm, 0.1f);
    const int lv = f.live[i], np = lv & 0xff, no = lv >> 8;
    float2 mm = make_float2(0.f, 0.f);
    for (int j = 0; j < f.kp; ++j) {                               // slot order; empty slots (the tail) yield f(0)
        float2 x = make_float2(f.f0[0], f.f0[1]);
        if (j < np) x = reinterpret_cast<const float2 *>(f.cmsg_ped)[f.map_ped[i * f.kp + j]];
        mm.x += x.x; mm.y += x.y;
    }
    if (f.has_obs) {
        float2 mo = make_float2(0.f, 0.f);
        for (int j = 0; j < f.ko; ++j) {
            float2 x = make_float2(f.f0[2], f.f0[3]);
            if (j < no) x = reinterpret_cast<const float2 *>(f.cmsg_obs)[f.map_obs[i * f.ko + j]];
            mo.x += x.x; mo.y += x.y;
        }
        mm = make_float2(__fadd_rn(mm.x, mo.x), __fadd_rn(mm.y, mo.y));
    }
    float acc[2];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        const float dir = __fdiv_rn(c == 0 ? sf0 : sf1, nrm);
        const float dterm = __fdiv_rn(__fsub_rn(__fmul_rn(ds, dir), c == 0 ? hv.x : hv.y), f.tau);
        acc[c] = __fadd_rn(c == 0 ? mm.x : mm.y, dterm);
    }
    return make_float2(acc[0], acc[1]);
}

// slot sums + destination term (model.py:1205-1210) followed by integrate_agent, one thread per agent
__global__ void __launch_bounds__(128) nn_finish_integrate_kernel(IntArgs g, FinishArgs f, const int *__restrict__ t_dev) {
    const int64_t SN = static_cast<int64_t>(g.S) * g.N;
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i == 0) { f.counts[0] = 0; f.counts[1] = 0; }
    if (i >= SN) return;
    if (t_dev) {                                                   // captured loop: frame index from device memory
        const int t = *t_dev;
        g.entry += (t + 1) * SN; g.dest_idx_gt += (t + 1) * SN;
        g.p_gt += (t + 1) * SN; g.v_gt += (t + 1) * SN; g.a_gt += (t + 1) * SN; g.dest_gt += (t + 1) * SN;
        g.rec_p += t * SN; g.rec_v += t * SN; g.rec_a += t * SN; g.rec_mask += t * SN;
    }
    const float2 a_next = nn_agent_output(g, f, i);
    if (f.a_out) f.a_out[i] = a_next;
    integrate_agent(g, i, a_next);
}

// Agent-sharded ranks: the same for the rank's own rows [row0, row0 + rows); the new p, v, a of a row are stored into
// EVERY rank's next-state arrays over NVLink peer memory (the step's only exchange, riding on this kernel's epilogue:
// 24 B per agent and peer); dest, dest_idx and hist_v of a row are only ever read by its owner and stay local.
struct PushTabs { float2 *p[8], *v[8], *a[8]; int world; };

__global__ void __launch_bounds__(128) nn_finish_integrate_push_kernel(IntArgs g, FinishArgs f, PushTabs t, int64_t row0,
                                                                       int64_t rows) {
    const int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (k == 0) { f.counts[0] = 0; f.counts[1] = 0; }
    if (k >= rows) return;
    const int64_t i = row0 + k;
    const float2 a_next = nn_agent_output(g, f, i);
    if (f.a_out) f.a_out[i] = a_next;
    const AgentNext o = integrate_agent_compute(g, i, a_next);
    g.dest[i] = o.dest; g.dest_idx[i] = o.di;
    if (g.hist_v) g.hist_v[i] = o.hv;
    for (int r = 0; r < t.world; ++r) { t.p[r][i] = o.p; t.v[r][i] = o.v; t.a[r][i] = o.a; }
    __threadfence_system();                                        // visible to the peers before the step's barrier
}

// scratch of the fused step, cached per calling thread, device and stream; released by piml_free_workspace()
struct NnScratch { cudaStream_t st; int dev; char *buf; size_t cap; };
static thread_local NnScratch g_nn_slots[8] = {};
static thread_local int g_nn_used = 0;

void nn_scratch_free() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return;
    for (int i = 0; i < g_nn_used; ++i)
        if (g_nn_slots[i].buf) {
            cudaSetDevice(g_nn_slots[i].dev);
            cudaStreamSynchronize(g_nn_slots[i].st);
            cudaFree(g_nn_slots[i].buf);
            g_nn_slots[i] = NnScratch{};
        }
    g_nn_used = 0;
    cudaSetDevice(dev);
}

// *fresh: the buffer was (re)allocated, its counters are not zero yet
static int nn_scratch_get(cudaStream_t st, size_t bytes, char **out, bool *fresh) {
    int dev = 0;
    PIML_CUDA(cudaGetDevice(&dev));
    NnScratch *s = nullptr;
    for (int i = 0; i < g_nn_used; ++i)
        if (g_nn_slots[i].st == st && g_nn_slots[i].dev == dev) s = &g_nn_slots[i];
    *fresh = false;
    if (!s) {
        s = &g_nn_slots[g_nn_used < 8 ? g_nn_used++ : 7];
        if (s->buf) { cudaSetDevice(s->dev); cudaFree(s->buf); cudaSetDevice(dev); }
        s->st = st; s->dev = dev; s->buf = nullptr; s->cap = 0;
    }
    if (s->cap < bytes) {
        if (s->buf) { PIML_CUDA(cudaStreamSynchronize(st)); PIML_CUDA(cudaFree(s->buf)); }
        s->buf = nullptr; s->cap = 0;
        PIML_CUDA(cudaMalloc(&s->buf, bytes));
        s->cap = bytes;
        *fresh = true;
    }
    *out = s->buf;
    return PIML_OK;
}

static size_t al256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

struct ShardInfo { int64_t row0, row1; PushTabs tabs; };

// t_dev != nullptr: entry_* / rec_* are the BASE pointers of time-major arrays and the frame comes from device memory
// sh != nullptr: this rank evaluates rows [row0, row1) only and pushes their new state to every rank
int nn_step_launch(const piml_nn_step_args *r, const int *t_dev, cudaStream_t st, const ShardInfo *sh = nullptr) {
    Tc16Plan P16;
    if (tc16_plan_for(r->desc, &P16))
        return fail(PIML_ERR_UNSUPPORTED, "piml_nn_step_f32: the network does not fit the 16-bit tensor-core kernel "
                                          "(per-slot decoder, hidden widths 32 / 64 / 128)");
    const int64_t SN = static_cast<int64_t>(r->S) * r->N;
    const int kp = r->kp < r->N ? r->kp : r->N;
    const int ko = r->M > 0 ? (r->ko < r->M ? r->ko : r->M) : 0;
    const int has_obs = (r->has_obs && ko > 0) ? 1 : 0;
    PIML_REQUIRE(kp >= 1 && kp <= 32 && ko <= 32, "piml_nn_step_f32: topk (%d,%d) out of range", r->kp, r->ko);
    PIML_REQUIRE(SN * (kp > ko ? kp : ko) < (1LL << 31), "piml_nn_step_f32: too many slot rows");
    const int64_t rows_ped = SN * kp, rows_obs = SN * ko;
    // scratch: f0 [4] + counts [2] (+ pad) | compact rows (+ 1 row of slack) | messages | maps
    const size_t b_head = 256, b_rp = al256(sizeof(float) * 6 * (rows_ped + 1)), b_ro = al256(sizeof(float) * 6 * (rows_obs + 1)),
                 b_mp = al256(sizeof(float) * 2 * (rows_ped + 1)), b_mo = al256(sizeof(float) * 2 * (rows_obs + 1)),
                 b_ip = al256(sizeof(int) * (rows_ped + 1)), b_io = al256(sizeof(int) * (rows_obs + 1)),
                 b_lv = al256(sizeof(uint16_t) * (SN + 1));
    char *base = nullptr;
    bool fresh = false;
    int rc = nn_scratch_get(st, b_head + b_rp + b_ro + b_mp + b_mo + b_ip + b_io + b_lv, &base, &fresh);
    if (rc) return rc;
    float *f0 = reinterpret_cast<float *>(base);
    int *counts = reinterpret_cast<int *>(base + 16);
    base += b_head;
    float *rows_p = reinterpret_cast<float *>(base); base += b_rp;
    float *rows_o = reinterpret_cast<float *>(base); base += b_ro;
    float *msg_p = reinterpret_cast<float *>(base); base += b_mp;
    float *msg_o = reinterpret_cast<float *>(base); base += b_mo;
    int *map_p = reinterpret_cast<int *>(base); base += b_ip;
    int *map_o = reinterpret_cast<int *>(base); base += b_io;
    uint16_t *live = reinterpret_cast<uint16_t *>(base);
    if (fresh) PIML_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(int), st));       // afterwards the finish kernel zeroes them

    // ---- features of the current state, compact rows only (dense copies on request)
    FeatArgs a;
    a.pos = r->p; a.vel = r->v; a.acc = r->a; a.dest = r->dest; a.head = nullptr; a.obs = r->obstacles;
    a.obs_frame_stride = r->obs_per_scene ? static_cast<int64_t>(r->M) * 2 : 0;
    a.obs_channel_T = r->obs_per_scene ? 1 : 0;
    a.B = r->S; a.N = r->N; a.M = r->M; a.kp = kp; a.ko = ko;
    a.cos_p = r->cos_p; a.thr_p = r->thr_p; a.pre2_p = prefilter_sq(r->thr_p);
    a.cos_o = r->cos_o; a.thr_o = r->thr_o; a.pre2_o = prefilter_sq(r->thr_o);
    a.ped_f = r->ped_f; a.obs_f = r->M > 0 ? r->obs_f : nullptr; a.dest_f = r->dest_f;
    a.ped_idx = nullptr; a.ped_dist = nullptr; a.obs_idx = nullptr; a.obs_dist = nullptr;
    a.hist_v = r->hist_v; a.desired_speed = r->desired_speed; a.self_f = r->dest_f ? r->self_f : nullptr;
    a.row0 = sh ? sh->row0 : 0; a.row1 = sh ? sh->row1 : 0;
    CompactOut co{rows_p, rows_o, map_p, map_o, live, counts};
    rc = relative_features_cells(a, r->obs_per_scene ? r->S : 1, st, &co);
    if (rc) return rc;

    // ---- network on the compact rows (+ one zero row per branch for f(0))
    Tc16Args b;
    b.params = r->packed_tc; b.ped = rows_p; b.obs = rows_o; b.R = SN; b.kp = kp; b.ko = ko;
    b.ag_ped = 128 / kp; b.ag_obs = ko ? 128 / ko : 1; b.n_ped_tiles = 0; b.n_obs_tiles = 0;
    b.sums = nullptr; b.ped_msgs = nullptr; b.obs_msgs = nullptr;
    b.compact = 1; b.has_obs = has_obs;
    b.list_ped = nullptr; b.list_obs = nullptr; b.counts = counts;
    b.cmsg_ped = msg_p; b.cmsg_obs = msg_o; b.f0 = f0;
    const int64_t tiles = (rows_ped + 128) / 128 + (has_obs ? (rows_obs + 128) / 128 : 0);
    rc = tc16_launch(P16, b, tiles < 2 ? 2 : tiles, st);
    if (rc) return rc;

    // ---- slot sums + destination term + state update
    IntArgs g;
    g.p = reinterpret_cast<float2 *>(r->p); g.v = reinterpret_cast<float2 *>(r->v); g.a = reinterpret_cast<float2 *>(r->a);
    g.a_next = nullptr; g.dest = reinterpret_cast<float2 *>(r->dest);
    g.dest_idx = r->dest_idx; g.dest_num = r->dest_num; g.waypoints = reinterpret_cast<const float2 *>(r->waypoints);
    g.S = r->S; g.D = r->D; g.N = r->N; g.dt = r->dt; g.remove_on_arrival = r->remove_on_arrival; g.entry = r->entry;
    g.p_gt = reinterpret_cast<const float2 *>(r->p_gt); g.v_gt = reinterpret_cast<const float2 *>(r->v_gt);
    g.a_gt = reinterpret_cast<const float2 *>(r->a_gt); g.dest_gt = reinterpret_cast<const float2 *>(r->dest_gt);
    g.dest_idx_gt = r->dest_idx_gt; g.hist_v = reinterpret_cast<float2 *>(r->hist_v);
    g.rec_p = reinterpret_cast<float2 *>(r->rec_p); g.rec_v = reinterpret_cast<float2 *>(r->rec_v);
    g.rec_a = reinterpret_cast<float2 *>(r->rec_a); g.rec_mask = r->rec_mask;
    FinishArgs f{msg_p, msg_o, map_p, map_o, live, f0, r->desired_speed, kp, ko, has_obs, r->tau,
                 reinterpret_cast<float2 *>(r->a_next), counts};
    const int threads = 128;
    if (sh) {
        const int64_t rows = sh->row1 - sh->row0;
        nn_finish_integrate_push_kernel<<<static_cast<unsigned>((rows + threads - 1) / threads), threads, 0, st>>>(
            g, f, sh->tabs, sh->row0, rows);
        count_launch();
        return check_launch("nn_finish_integrate_push_kernel");
    }
    nn_finish_integrate_kernel<<<static_cast<unsigned>((SN + threads - 1) / threads), threads, 0, st>>>(g, f, t_dev);
    count_launch();
    return check_launch("nn_finish_integrate_kernel");
}

}  // namespace piml

using namespace piml;

extern "C" int piml_nn_step_supported(const piml_net_desc *desc) {
    Tc16Plan P16;
    return (desc && tc16_plan_for(desc, &P16) == 0) ? 1 : 0;
}

extern "C" int piml_nn_step_f32(const piml_nn_step_args *r, void *stream) {
    PIML_REQUIRE(r && r->desc && r->packed_tc, "piml_nn_step_f32: null descriptor / parameters");
    PIML_REQUIRE(r->S >= 1 && r->N >= 1 && r->D >= 1 && r->M >= 0, "piml_nn_step_f32: bad dimensions S=%d N=%d D=%d M=%d",
                 r->S, r->N, r->D, r->M);
    PIML_REQUIRE(r->p && r->v && r->a && r->dest && r->dest_idx && r->hist_v && r->dest_num && r->waypoints &&
                     r->desired_speed && (r->M == 0 || r->obstacles),
                 "piml_nn_step_f32: null state / static input");
    PIML_REQUIRE(!r->entry || (r->p_gt && r->v_gt && r->a_gt && r->dest_gt && r->dest_idx_gt),
                 "piml_nn_step_f32: entry mask given without ground-truth arrays");
    PIML_REQUIRE(!r->dest_f || (r->ped_f && r->self_f && (r->M == 0 || r->obs_f)),
                 "piml_nn_step_f32: dense feature outputs must be given together");
    PIML_REQUIRE(aligned16(r->packed_tc), "piml_nn_step_f32: packed_tc must be 16-byte aligned");
    return nn_step_launch(r, nullptr, static_cast<cudaStream_t>(stream));
}

extern "C" int piml_nn_step_shard_f32(const piml_nn_step_args *r, int64_t row0, int64_t row1, int world,
                                      const uint64_t *p_next, const uint64_t *v_next, const uint64_t *a_next,
                                      void *stream) {
    PIML_REQUIRE(r && r->desc && r->packed_tc, "piml_nn_step_shard_f32: null descriptor / parameters");
    PIML_REQUIRE(r->S == 1 && r->N >= 1 && r->D >= 1 && r->M >= 0, "piml_nn_step_shard_f32: one scene per sharded crowd");
    PIML_REQUIRE(r->p && r->v && r->a && r->dest && r->dest_idx && r->hist_v && r->dest_num && r->waypoints &&
                     r->desired_speed && (r->M == 0 || r->obstacles),
                 "piml_nn_step_shard_f32: null state / static input");
    PIML_REQUIRE(!r->entry || (r->p_gt && r->v_gt && r->a_gt && r->dest_gt && r->dest_idx_gt),
                 "piml_nn_step_shard_f32: entry mask given without ground-truth arrays");
    PIML_REQUIRE(!r->dest_f && !r->ped_f && !r->obs_f && !r->self_f, "piml_nn_step_shard_f32: no dense feature outputs");
    PIML_REQUIRE(0 <= row0 && row0 < row1 && row1 <= r->N, "piml_nn_step_shard_f32: bad row range");
    PIML_REQUIRE(world >= 1 && world <= 8 && p_next && v_next && a_next, "piml_nn_step_shard_f32: bad peer tables");
    PIML_REQUIRE(aligned16(r->packed_tc), "piml_nn_step_shard_f32: packed_tc must be 16-byte aligned");
    ShardInfo sh;
    sh.row0 = row0; sh.row1 = row1; sh.tabs.world = world;
    for (int g = 0; g < world; ++g) {
        sh.tabs.p[g] = reinterpret_cast<float2 *>(p_next[g]);
        sh.tabs.v[g] = reinterpret_cast<float2 *>(v_next[g]);
        sh.tabs.a[g] = reinterpret_cast<float2 *>(a_next[g]);
    }
    return nn_step_launch(r, nullptr, static_cast<cudaStream_t>(stream), &sh);
}
