// mlp_tc.cu -- interaction-network forward on the 5th-generation tensor cores (tcgen05, TMEM), for sm_100a: the
// 3xTF32 kernel, the packing of both tensor-core weight images and the C entry points, which choose between this
// kernel and the 16-bit one (mlp_tc16.cu).
#include "common.cuh"
#include "tc.cuh"
#include "mlp_tc16.cuh"

// =====================================================================================================================
// Fused interaction-network forward on the tensor cores (inference: eval mode, acceleration output [+ 2-d messages]).
//
// Same mathematics as pinnsf_tile_kernel (mlp.cu) -- reference src/models/model.py:40-119, :762-792, :1104-1135,
// :1185-1212, :1271-1296 -- but every wide Linear of a 128-row tile is a chain of tcgen05.mma (kind::tf32) with the
// 3xTF32 split (x_lo w_hi + x_hi w_lo + x_hi w_hi, fp32 accumulation in TMEM): measured 1e-6 of fp64 per layer, i.e.
// fp32-grade, which the 1e-5 parity gate needs and plain TF32 (3e-4) does not give.
//
// Per CTA (persistent, one per SM, 320 threads):
//   warp 0  : TMA producer -- streams the layers' weight images (hi + lo, pre-split and pre-arranged as UMMA K-major
//             core matrices by piml_pinnsf_pack_tc_f32) through a 5-stage shared-memory ring with cp.async.bulk;
//   warp 1  : MMA issuer -- one thread issues the tcgen05.mma chain of a layer: A (activations, hi / lo) from TMEM,
//             B from the ring, D into TMEM; tcgen05.commit frees ring stages and signals "D ready";
//   warps 2-9: epilogue -- thread = tile row (two warps per TMEM lane quarter, alternating 32-column groups):
//             tcgen05.ld D, + bias, ReLU / ResDNN 2x fold, split into tf32 hi / lo and tcgen05.st as the NEXT layer's A
//             operand (activations never touch shared memory); the 2-wide predictor, the sum over an agent's slots
//             and (kind 1) the per-agent embedding sum run on the CUDA cores in fp32.
// TMEM columns: D0 [0,128), D1 [128,256) (alternating per layer), A_hi [256,384), A_lo [384,512).
namespace piml {

constexpr int TC_EPI_WARPS = 8;                 // two warps per TMEM lane quarter: column halves
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;
constexpr int TC_STAGES = 5;
constexpr int TC_STAGE_BYTES = 32768;          // hi + lo image of a 32-deep K chunk of a 128-wide layer
constexpr int TC_MAXL = 16;
constexpr int TC_MAXCH = 64;
constexpr int TC_COL_D0 = 0, TC_COL_D1 = 128, TC_COL_AH = 256, TC_COL_AL = 384;
constexpr int TC_STAGE_LD = 17;

struct TcLayer { int K, Kp, N, chunk0, nchunks, bias_off, relu; float scale; };   // bias_off: floats into the bias block
struct TcChunk { int off, bytes, cells; };          // float offset from the branch's weight base; 16-byte K cells (even)
struct TcPlan {
    int kind, n_enc, n_dec, nl, pw, dw;
    TcLayer L[TC_MAXL];
    int nch; TcChunk C[TC_MAXCH];
    int predw_off, predb_off, bias_floats;         // inside the bias block
    int64_t w_off[2], b_off[2];                    // float offsets of a branch's chunk images / bias block
    int64_t total;
};

struct TcArgs {
    const float *params; const float *ped; const float *obs;
    int64_t R; int kp, ko, ag_ped, ag_obs; int64_t n_ped_tiles, n_obs_tiles;
    float *sums; float *ped_msgs; float *obs_msgs;
    // Compact mode (kind 0): zero-padded slot rows all produce the same message f(0), so only the non-zero rows (+ one
    // zero row per branch that yields f(0)) go through the network; the slot sums are formed by the finish kernel.
    int compact; int has_obs;
    const int *list_ped, *list_obs;                // indices of the non-zero slot rows of each branch
    const int *counts;                             // [2] their number (written by tc_compact_kernel)
    float *cmsg_ped, *cmsg_obs;                    // per-row messages (R*kp,2), (R*ko,2): non-zero rows are written
    float *f0;                                     // [2][2] message of a zero row per branch
};

// mbarrier wait that can never hang the GPU: a protocol bug traps (launch error) after ~seconds instead of spinning.
__device__ __forceinline__ void tc_wait(uint64_t *bar, uint32_t parity) {
    if (!mbar_wait_bounded(bar, parity, 1u << 28)) __trap();
}

__device__ __forceinline__ void half_barrier(int half) {           // the 128 epilogue threads of one column half
    asm volatile("bar.sync %0, 128;" ::"r"(1 + half) : "memory");
}
__device__ __forceinline__ void epi_barrier_all() { asm volatile("bar.sync 3, 256;" ::: "memory"); }

// Pipeline inside a tile (layer l reads A, writes D[l & 1]):
//   epilogue of layer l   : waits "D[l&1] ready", then per 32-column group g: tcgen05.ld -> bias/ReLU -> hi/lo ->
//                           tcgen05.st into A columns [32g, 32g+32) -> arrives on a_ready[g]
//   MMAs of layer l + 1   : K chunk g starts as soon as a_ready[g] fired, i.e. while the epilogue is still converting
//                           groups g+1.. of layer l; they accumulate into the OTHER accumulator D[(l+1)&1].
// So tensor-core work of layer l+1 overlaps the CUDA-core epilogue of layer l; activations never leave TMEM.
__global__ void __launch_bounds__(TC_THREADS, 1) pinnsf_tc_kernel(const __grid_constant__ TcPlan P,
                                                                  const __grid_constant__ TcArgs a) {
    extern __shared__ __align__(128) unsigned char tc_smem[];
    unsigned char *ring = tc_smem;                                                       // TC_STAGES x 32 KB
    float *biasb = reinterpret_cast<float *>(ring + TC_STAGES * TC_STAGE_BYTES);         // [2][bias_floats]
    float *small = biasb + 2 * P.bias_floats;                                            // [2 halves][128][2]
    float *stage = small + 512;                                                          // [2 halves][128][33] (kind 1)
    uint64_t *bars = reinterpret_cast<uint64_t *>(
        (reinterpret_cast<uintptr_t>(stage + 2 * 128 * TC_STAGE_LD) + 15) & ~static_cast<uintptr_t>(15));
    uint64_t *full = bars, *empty = bars + TC_STAGES, *a_ready = bars + 2 * TC_STAGES, *d_ready = a_ready + 4;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(d_ready + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (warp == 0) tc::tmem_alloc(tmem_slot, 512);
    if (tid == 32) {
        for (int s = 0; s < TC_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int c = 0; c < 4; ++c) mbar_init(&a_ready[c], 256);
        mbar_init(&d_ready[0], 1);
        mbar_init(&d_ready[1], 1);
        mbar_fence_init();
    }
    for (int e = tid; e < 2 * P.bias_floats; e += TC_THREADS) {
        const int br = e / P.bias_floats, i = e - br * P.bias_floats;
        biasb[e] = (br == 0 || a.has_obs) ? a.params[P.b_off[br] + i] : 0.f;
    }
    // compact mode: rows = the listed non-zero rows followed by ONE zero row (index -1) per branch
    // (compact == 2, kind 1: the lists hold AGENTS with at least one non-zero slot, + one all-zero agent per branch)
    const int64_t cnt_ped = a.compact ? a.counts[0] + 1 : 0, cnt_obs = (a.compact && a.has_obs) ? a.counts[1] + 1 : 0;
    const int64_t per_ped = a.compact == 2 ? a.ag_ped : 128, per_obs = a.compact == 2 ? a.ag_obs : 128;
    const int64_t n_ped_tiles = a.compact ? (cnt_ped + per_ped - 1) / per_ped : a.n_ped_tiles;
    const int64_t n_obs_tiles = a.compact ? (cnt_obs + per_obs - 1) / per_obs : a.n_obs_tiles;
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tbase = *tmem_slot;
    const int64_t ntiles = n_ped_tiles + n_obs_tiles;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            uint32_t pc = 0;
            for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const int br = tile < n_ped_tiles ? 0 : 1;
                const float *wbase = a.params + P.w_off[br];
                for (int c = 0; c < P.nch; ++c, ++pc) {
                    const uint32_t s = pc % TC_STAGES, ph = (pc / TC_STAGES) & 1u;
                    tc_wait(&empty[s], ph ^ 1u);
                    const uint32_t bytes = static_cast<uint32_t>(P.C[c].bytes);   // <= TC_STAGE_BYTES
                    mbar_expect_tx(&full[s], bytes);
                    tma_bulk_g2s(ring + s * TC_STAGE_BYTES, reinterpret_cast<const unsigned char *>(wbase + P.C[c].off),
                                 bytes, &full[s]);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        // The whole warp runs the loop on warp-uniform values and one elected lane issues (tc::elect_one): with the
        // issuing code under `if (lane == 0)` ptxas wrapped every MMA in an R2UR waterfall loop (86 instead of 69 cycles
        // per MMA in round 1's profile).
        const uint32_t tb = __shfl_sync(0xffffffffu, tbase, 0);
        const uint32_t ring_addr = __shfl_sync(0xffffffffu, tc::smem_addr(ring), 0);
        const long long nt = __shfl_sync(0xffffffffu, static_cast<long long>(ntiles), 0);
        uint32_t pc = 0, aph = 0;                                  // aph: phase bit per a_ready barrier
        for (long long tile = blockIdx.x; tile < nt; tile += gridDim.x) {
            for (int li = 0; li < P.nl; ++li) {
                const TcLayer &Ly = P.L[li];
                const uint32_t dcol = tb + ((li & 1) ? TC_COL_D1 : TC_COL_D0);
                const uint32_t idesc = tc::idesc_tf32(Ly.N);
                const uint32_t lbo = Ly.N * 16, sbo = 128, kstep = 2 * lbo;
                bool acc = false;
                for (int c = 0; c < Ly.nchunks; ++c, ++pc) {
                    tc_wait(&a_ready[c], (aph >> c) & 1u);         // A columns of this K chunk are in TMEM
                    aph ^= (1u << c);
                    const uint32_t s = pc % TC_STAGES, ph = (pc / TC_STAGES) & 1u;
                    tc_wait(&full[s], ph);
                    tc::fence_after_sync();
                    const TcChunk &Ch = P.C[Ly.chunk0 + c];
                    const uint32_t hi_addr = ring_addr + s * TC_STAGE_BYTES;
                    uint64_t bh = tc::smem_desc(hi_addr, lbo, sbo);
                    uint64_t bl = tc::smem_desc(hi_addr + Ch.cells * lbo, lbo, sbo);
                    const uint64_t dstep = kstep >> 4;             // start-address field advances by one K = 8 step
                    uint32_t ah = tb + TC_COL_AH + c * 32, al = tb + TC_COL_AL + c * 32;
                    const int nks = Ch.cells / 2;
                    if (tc::elect_one()) {
#pragma unroll 4
                        for (int ks = 0; ks < nks; ++ks, bh += dstep, bl += dstep, ah += 8, al += 8) {
                            tc::mma_tf32_ts(dcol, al, bh, idesc, acc);      // x_lo w_hi
                            tc::mma_tf32_ts(dcol, ah, bl, idesc, true);     // x_hi w_lo
                            tc::mma_tf32_ts(dcol, ah, bh, idesc, true);     // x_hi w_hi
                            acc = true;
                        }
                        tc::commit(&empty[s]);                     // ring stage free once these MMAs have read it
                        if (c == Ly.nchunks - 1) tc::commit(&d_ready[li & 1]);   // accumulator of this layer complete
                    }
                    acc = true;
                    __syncwarp();
                }
            }
        }
    } else {
        // ===== epilogue warps: thread = tile row; the two warps of a lane quarter split the column groups =====
        const int q4 = warp & 3;                                   // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2;                          // 0: even 32-column groups, 1: odd groups
        const int m = q4 * 32 + lane;                              // tile row == TMEM lane
        const uint32_t tl = tbase + (static_cast<uint32_t>(q4 * 32) << 16);
        float *stg = stage + half * 128 * TC_STAGE_LD;
        uint32_t dph = 0;                                          // phase bit per d_ready barrier
        // The 6-d features of a tile row (and, in compact mode, the row's index through the list) are two dependent
        // global loads at the head of a tile's critical path: fetch them one tile ahead, into registers.
        struct RowFeat { int64_t crow; float f[6]; bool live; };
        auto load_row = [&](int64_t tile) {
            RowFeat rf;
            rf.crow = -1; rf.live = false;
#pragma unroll
            for (int q = 0; q < 6; ++q) rf.f[q] = 0.f;
            if (tile >= ntiles) return rf;
            const int br = tile < n_ped_tiles ? 0 : 1;
            const int k = br == 0 ? a.kp : a.ko;
            const int AG = br == 0 ? a.ag_ped : a.ag_obs;
            const int64_t tloc = br == 0 ? tile : tile - n_ped_tiles;
            const int64_t agent0 = tloc * AG;
            const int64_t cnt = br == 0 ? cnt_ped : cnt_obs;
            int64_t src;
            if (a.compact == 2) {                                  // listed agent (m / k), its slot m % k
                const int na = static_cast<int>(min(static_cast<int64_t>(AG), cnt - agent0));
                const int64_t ai = agent0 + m / k;
                int64_t ag = -1;
                if (m < na * k && ai < cnt - 1) ag = (br == 0 ? a.list_ped : a.list_obs)[ai];
                rf.live = ag >= 0;
                src = ag * k + m % k;
            } else if (a.compact) {
                const int nrows = static_cast<int>(min(static_cast<int64_t>(128), cnt - tloc * 128));
                if (m < nrows && tloc * 128 + m < cnt - 1) rf.crow = (br == 0 ? a.list_ped : a.list_obs)[tloc * 128 + m];
                rf.live = rf.crow >= 0;
                src = rf.crow;
            } else {
                const int na = static_cast<int>(min(static_cast<int64_t>(AG), a.R - agent0));
                rf.live = m < na * k;
                src = agent0 * k + m;
            }
            if (rf.live) {
                const float2 *f2 = reinterpret_cast<const float2 *>((br == 0 ? a.ped : a.obs) + src * 6);
                const float2 x0 = f2[0], x1 = f2[1], x2 = f2[2];
                rf.f[0] = x0.x; rf.f[1] = x0.y; rf.f[2] = x1.x; rf.f[3] = x1.y; rf.f[4] = x2.x; rf.f[5] = x2.y;
            }
            return rf;
        };
        RowFeat nxt = load_row(half == 0 ? static_cast<int64_t>(blockIdx.x) : ntiles);
        for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const int br = tile < n_ped_tiles ? 0 : 1;
            const int k = br == 0 ? a.kp : a.ko;
            const int AG = br == 0 ? a.ag_ped : a.ag_obs;
            const int64_t tloc = br == 0 ? tile : tile - n_ped_tiles;
            const int64_t agent0 = tloc * AG;
            const int64_t cnt = br == 0 ? cnt_ped : cnt_obs;
            const int na = a.compact == 2 ? static_cast<int>(min(static_cast<int64_t>(AG), cnt - agent0))
                                          : (a.compact ? 0 : static_cast<int>(min(static_cast<int64_t>(AG), a.R - agent0)));
            const int nrows = a.compact == 1 ? static_cast<int>(min(static_cast<int64_t>(128), cnt - tloc * 128)) : na * k;
            const int64_t row0 = agent0 * k;
            // compact mode: the slot row this tile row stands for (-1: the zero row that yields f(0))
            const int64_t crow = nxt.crow;
            const float *bb = biasb + br * P.bias_floats;
            if (half == 0) {   // stage the 6-d features of this row as the first A operand (K padded to 8 with zeros)
                uint32_t hi[8], lo[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float x = (q < 6 && nxt.live) ? nxt.f[q] : 0.f;
                    tc::split_tf32(x, hi[q], lo[q]);
                }
                tc::st8(tl + TC_COL_AH, hi);
                tc::st8(tl + TC_COL_AL, lo);
                tc::wait_st();
                tc::fence_before_sync();
            }
            tc::mbar_arrive(&a_ready[0]);
            if (half == 0) nxt = load_row(tile + gridDim.x);       // in flight while this tile runs
            float m0 = 0.f, m1 = 0.f;
            for (int li = 0; li < P.nl; ++li) {
                const TcLayer &Ly = P.L[li];
                const bool last = li == P.nl - 1;
                const bool to_sum = P.kind == 1 && li == P.n_enc - 1;        // kind 1: sum the slot embeddings per agent
                const uint32_t dcol = tl + ((li & 1) ? TC_COL_D1 : TC_COL_D0);
                tc_wait(&d_ready[li & 1], (dph >> (li & 1)) & 1u);
                dph ^= (1u << (li & 1));
                tc::fence_after_sync();
                const float *bias = bb + Ly.bias_off;
                // every 32-column group is converted by BOTH warps of the lane quarter (16 columns each), so that
                // the first K chunk of the next layer is released after half the latency
                for (int g = 0; g < Ly.N / 32; ++g) {
                    const int n0 = g * 32 + half * 16;
                    uint32_t r[16];
                    tc::ld16(dcol + n0, r);
                    tc::wait_ld();
                    float y[16];
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        float v = __uint_as_float(r[q]) + bias[n0 + q];      // (ResDNN's 2x is folded into W and b)
                        if (Ly.relu) v = fmaxf(v, 0.f);
                        y[q] = v;
                    }
                    if (last) {                                    // predictor Linear(dw, 2) on the CUDA cores
                        const float *w0 = bb + P.predw_off + n0, *w1 = w0 + P.dw;
#pragma unroll
                        for (int q = 0; q < 16; ++q) { m0 = fmaf(y[q], w0[q], m0); m1 = fmaf(y[q], w1[q], m1); }
                        continue;
                    }
                    if (to_sum) {                                  // torch.sum(dim=-2) over the k slots (model.py:1276)
#pragma unroll
                        for (int q = 0; q < 16; ++q) stg[m * TC_STAGE_LD + q] = y[q];
                        half_barrier(half);
#pragma unroll
                        for (int q = 0; q < 16; ++q) {
                            float s = 0.f;
                            if (m < na)
                                for (int j = 0; j < k; ++j) s += stg[(m * k + j) * TC_STAGE_LD + q];
                            y[q] = s;
                        }
                        half_barrier(half);
                    }
                    uint32_t lo[16];
#pragma unroll
                    for (int q = 0; q < 16; ++q) tc::split_tf32(y[q], r[q], lo[q]);
                    tc::st16(tl + TC_COL_AH + n0, r);
                    tc::st16(tl + TC_COL_AL + n0, lo);
                    tc::wait_st();
                    tc::fence_before_sync();
                    tc::mbar_arrive(&a_ready[g]);                  // K chunk g of the next layer may start
                }
            }
            // combine the two column halves of the predictor, then sum over an agent's slots
            small[(half * 128 + m) * 2] = m0;
            small[(half * 128 + m) * 2 + 1] = m1;
            epi_barrier_all();
            if (half == 0) {
                m0 = small[m * 2] + small[(128 + m) * 2] + bb[P.predb_off];
                m1 = small[m * 2 + 1] + small[(128 + m) * 2 + 1] + bb[P.predb_off + 1];
                if (P.kind == 0 && a.compact) {
                    if (m < nrows) {                               // slot sums are formed by the finish kernel
                        float *dst = crow >= 0 ? (br == 0 ? a.cmsg_ped : a.cmsg_obs) + crow * 2 : a.f0 + br * 2;
                        dst[0] = m0; dst[1] = m1;
                    }
                } else if (P.kind == 0) {
                    float *msgs_out = br == 0 ? a.ped_msgs : a.obs_msgs;
                    if (msgs_out && m < nrows) { msgs_out[(row0 + m) * 2] = m0; msgs_out[(row0 + m) * 2 + 1] = m1; }
                    half_barrier(0);                               // every partial read before the totals overwrite
                    small[m * 2] = m0; small[m * 2 + 1] = m1;
                    half_barrier(0);
                    for (int e = m; e < 2 * na; e += 128) {        // torch.sum(dim=-2) over the k slots (model.py:1194);
                        const int ag = e >> 1, c = e & 1;          // k = 1: 128 agents per tile, two sums per thread
                        float s = 0.f;
                        for (int j = 0; j < k; ++j) s += small[(ag * k + j) * 2 + c];
                        a.sums[(agent0 + ag) * 4 + br * 2 + c] = s;
                    }
                } else if (m < na) {
                    float *dst = a.sums + (agent0 + m) * 4 + br * 2;
                    if (a.compact == 2) {                          // listed agent, or the all-zero agent -> g(0)
                        const int64_t ag = agent0 + m < cnt - 1 ? (br == 0 ? a.list_ped : a.list_obs)[agent0 + m] : -1;
                        dst = ag >= 0 ? a.sums + ag * 4 + br * 2 : a.f0 + br * 2;
                    }
                    dst[0] = m0; dst[1] = m1;
                }
            }
            epi_barrier_all();                                     // small[] is free for the next tile
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tbase, 512);
}

// ---- plan + packing -------------------------------------------------------------------------------------------------
struct TcPackRec { int K, Kp, N; float scale; int64_t src_w, src_b, dst_w, dst_b; };
struct TcPackTab { int n; TcPackRec r[2 * TC_MAXL]; int dw; int64_t pred_src[2], predw_dst[2], predb_dst[2]; int64_t total; };

static int tc_build_plan(const piml_net_desc *d, TcPlan *P, TcPackTab *T) {
    PIML_REQUIRE(d->n_enc >= 1 && d->n_enc <= 8 && d->n_dec >= 1 && d->n_dec <= 8, "piml_pinnsf_tc: bad layer counts");
    PIML_REQUIRE(d->proc_mode == 0, "piml_pinnsf_tc: processor_hidden_layers == 1 is not supported on the tensor-core path");
    PIML_REQUIRE(d->enc_dims[0] == 6, "piml_pinnsf_tc: feature dim must be 6");
    PIML_REQUIRE(d->dec_dims[0] == d->enc_dims[d->n_enc], "piml_pinnsf_tc: decoder input != processor width");
    P->kind = d->kind; P->n_enc = d->n_enc; P->n_dec = d->n_dec; P->nl = d->n_enc + d->n_dec;
    P->pw = d->enc_dims[d->n_enc]; P->dw = d->dec_dims[d->n_dec];
    int nch = 0, woff = 0, boff = 0;
    int64_t src = 0;
    T->n = 0;
    auto layer = [&](int li, int K, int N, int relu, float scale) -> int {
        PIML_REQUIRE(N % 32 == 0 && N <= 128 && K <= 128 && (K % 8 == 0 || li == 0),
                     "piml_pinnsf_tc: layer %d (%d -> %d) needs widths that are multiples of 32 (<= 128)", li, K, N);
        TcLayer &L = P->L[li];
        L.K = K; L.Kp = (K + 7) & ~7; L.N = N; L.relu = relu; L.scale = scale; L.bias_off = boff; L.chunk0 = nch;
        L.nchunks = (L.Kp + 31) / 32;
        TcPackRec &r = T->r[T->n++];
        r.K = K; r.Kp = L.Kp; r.N = N; r.scale = scale; r.src_w = src; r.src_b = src + static_cast<int64_t>(K) * N; r.dst_w = woff; r.dst_b = boff;
        for (int c = 0; c < L.nchunks; ++c) {
            PIML_REQUIRE(nch < TC_MAXCH, "piml_pinnsf_tc: too many weight chunks");
            const int cells = (L.Kp - c * 32 < 32 ? L.Kp - c * 32 : 32) / 4;
            P->C[nch].off = woff; P->C[nch].cells = cells; P->C[nch].bytes = 2 * cells * N * 16;
            woff += 2 * cells * N * 4;
            ++nch;
        }
        boff += N;
        src += static_cast<int64_t>(K) * N + N;
        return PIML_OK;
    };
    int li = 0;
    for (int l = 0; l < d->n_enc; ++l, ++li) {
        const bool last = l == d->n_enc - 1;
        int rc = layer(li, d->enc_dims[l], d->enc_dims[l + 1], last ? 0 : 1, last ? 2.f : 1.f);   // ResDNN == 2x fold
        if (rc) return rc;
    }
    for (int l = 0; l < d->n_dec; ++l, ++li) {
        int rc = layer(li, d->dec_dims[l], d->dec_dims[l + 1], l < d->n_dec - 1 ? 1 : 0, 1.f);
        if (rc) return rc;
    }
    P->nch = nch;
    P->predw_off = boff; boff += 2 * P->dw;
    P->predb_off = boff; boff += 2;
    P->bias_floats = (boff + 3) & ~3;
    const int64_t branch_src = src + 2 * P->dw + 2;                // torch floats of one branch
    const int64_t branch_dst = static_cast<int64_t>(woff) + P->bias_floats;
    for (int br = 0; br < 2; ++br) {
        P->w_off[br] = br * branch_dst;
        P->b_off[br] = br * branch_dst + woff;
        T->pred_src[br] = br * branch_src + src;
        T->predw_dst[br] = P->b_off[br] + P->predw_off;
        T->predb_dst[br] = P->b_off[br] + P->predb_off;
    }
    T->dw = P->dw;
    // second branch: same records shifted
    const int n1 = T->n;
    for (int i = 0; i < n1; ++i) {
        TcPackRec r = T->r[i];
        r.src_w += branch_src; r.src_b += branch_src; r.dst_w += branch_dst; r.dst_b += P->b_off[1];
        T->r[T->n++] = r;
    }
    for (int i = 0; i < n1; ++i) T->r[i].dst_b += P->b_off[0];
    P->total = 2 * branch_dst;
    T->total = P->total;
    return PIML_OK;
}

// one thread per float of the packed vector
__global__ void pinnsf_pack_tc_kernel(const __grid_constant__ TcPackTab T, const float *__restrict__ src,
                                      float *__restrict__ dst, int nlayers_per_branch, int64_t branch_floats,
                                      int64_t wfloats) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= T.total) return;
    const int br = static_cast<int>(i / branch_floats);
    const int64_t off = i - br * branch_floats;
    float v = 0.f;
    if (off < wfloats) {
        // inside a weight image: find the layer, then (chunk, half, cell, n, kk)
        int l = 0;
        while (l + 1 < nlayers_per_branch && off >= T.r[l + 1].dst_w) ++l;
        const TcPackRec &R = T.r[br * nlayers_per_branch + l];
        int64_t e = off - T.r[l].dst_w;
        int c = 0;
        for (;;) {                                                 // chunks of this layer
            const int cells = (R.Kp - c * 32 < 32 ? R.Kp - c * 32 : 32) / 4;
            const int64_t cf = 2LL * cells * R.N * 4;
            if (e < cf) {
                const int half = static_cast<int>(e / (cells * R.N * 4));
                const int64_t r = e - static_cast<int64_t>(half) * cells * R.N * 4;
                const int cell = static_cast<int>(r / (R.N * 4)), n = static_cast<int>((r / 4) % R.N), kk = static_cast<int>(r & 3);
                const int kx = c * 32 + cell * 4 + kk;
                const float w = kx < R.K ? src[R.src_w + static_cast<int64_t>(n) * R.K + kx] * R.scale : 0.f;   // 2x: exact
                uint32_t hi, lo;
                tc::split_tf32(w, hi, lo);
                v = __uint_as_float(half == 0 ? hi : lo);
                break;
            }
            e -= cf; ++c;
        }
    } else {
        const int64_t b = off - wfloats;                           // inside the bias block
        const int64_t predw = T.predw_dst[0] - wfloats, predb = T.predb_dst[0] - wfloats;
        if (b >= predb) { if (b < predb + 2) v = src[T.pred_src[br] + 2LL * T.dw + (b - predb)]; }
        else if (b >= predw) { v = src[T.pred_src[br] + (b - predw)]; }
        else {
            int l = 0;
            while (l + 1 < nlayers_per_branch && b >= T.r[l + 1].dst_b - T.r[0].dst_b) ++l;
            const TcPackRec &R = T.r[br * nlayers_per_branch + l];
            const int64_t o = b - (T.r[l].dst_b - T.r[0].dst_b);
            if (o < R.N) v = src[R.src_b + o] * R.scale;
        }
    }
    dst[i] = v;
}

// per-agent sums scratch shared with mlp.cu's finish kernel
__global__ void pinnsf_tc_finish_kernel(const float *__restrict__ sums, const float *__restrict__ self,
                                        const float *__restrict__ dnorm, int64_t R, int has_obs, float tau,
                                        float *__restrict__ acc) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= 2 * R) return;
    const int64_t ag = i >> 1;
    const int c = static_cast<int>(i & 1);
    const float *s = self + ag * 7;
    float nrm = dnorm ? dnorm[ag * 2 + c] : norm2_rn(s[0], s[1]);
    if (nrm == 0.f) nrm = __fadd_rn(nrm, 0.1f);
    const float dir = __fdiv_rn(s[c], nrm);
    const float dterm = __fdiv_rn(__fsub_rn(__fmul_rn(s[6], dir), s[2 + c]), tau);
    float mm = sums[ag * 4 + c];
    if (has_obs) mm = __fadd_rn(mm, sums[ag * 4 + 2 + c]);
    acc[i] = __fadd_rn(mm, dterm);
}

__global__ void tc_colnorm_kernel(const float *__restrict__ self, int group, float *__restrict__ dnorm) {
    __shared__ float red[2][128];
    const int64_t base = static_cast<int64_t>(blockIdx.x) * group;
    float s0 = 0.f, s1 = 0.f;
    for (int i = threadIdx.x; i < group; i += blockDim.x) {
        const float x = self[(base + i) * 7], y = self[(base + i) * 7 + 1];
        s0 = fmaf(x, x, s0); s1 = fmaf(y, y, s1);
    }
    red[0][threadIdx.x] = s0; red[1][threadIdx.x] = s1;
    __syncthreads();
    for (int off = blockDim.x / 2; off > 0; off >>= 1) {
        if (threadIdx.x < off) { red[0][threadIdx.x] += red[0][threadIdx.x + off]; red[1][threadIdx.x] += red[1][threadIdx.x + off]; }
        __syncthreads();
    }
    const float n0 = sqrtf(red[0][0]), n1 = sqrtf(red[1][0]);
    for (int i = threadIdx.x; i < group; i += blockDim.x) { dnorm[(base + i) * 2] = n0; dnorm[(base + i) * 2 + 1] = n1; }
}

// Compact mode, pass 1: list the slot rows that are not all-zero (warp-aggregated append; a row's message does not
// depend on its place in a tile, so the order is irrelevant) and flag the zero rows for the finish kernel.
__global__ void tc_compact_kernel(const float *__restrict__ ped, const float *__restrict__ obs, int64_t rows_ped,
                                  int64_t rows_obs, int *__restrict__ list_ped, int *__restrict__ list_obs,
                                  int *__restrict__ counts, uint8_t *__restrict__ zero_ped,
                                  uint8_t *__restrict__ zero_obs) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const int br = i < rows_ped ? 0 : 1;
    const int64_t r = br == 0 ? i : i - rows_ped;
    const bool in = i < rows_ped + rows_obs;
    bool nz = false;
    if (in) {
        const float2 *f = reinterpret_cast<const float2 *>((br == 0 ? ped : obs) + r * 6);
        const float2 a = f[0], b = f[1], c = f[2];
        nz = !(a.x == 0.f && a.y == 0.f && b.x == 0.f && b.y == 0.f && c.x == 0.f && c.y == 0.f);
        (br == 0 ? zero_ped : zero_obs)[r] = nz ? 0 : 1;
    }
    // a warp may straddle the two branches: append per branch
#pragma unroll
    for (int b2 = 0; b2 < 2; ++b2) {
        const unsigned mask = __ballot_sync(0xffffffffu, in && nz && br == b2);
        if (!mask) continue;
        const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
        int base = 0;
        if (lane == leader) base = atomicAdd(&counts[b2], __popc(mask));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (in && nz && br == b2) (b2 == 0 ? list_ped : list_obs)[base + __popc(mask & ((1u << lane) - 1))] = static_cast<int>(r);
    }
}

// Compact mode 2 (summed-embedding networks, kind 1), pass 1: list the AGENTS of each branch that have a non-zero
// slot; an agent whose slots are all zero yields the same per-branch output g(0) = pred(dec(k * 2 enc(0))).
__global__ void tc_compact_agents_kernel(const float *__restrict__ ped, const float *__restrict__ obs, int64_t R,
                                         int kp, int ko, int *__restrict__ list_ped, int *__restrict__ list_obs,
                                         int *__restrict__ counts, uint8_t *__restrict__ zero_ped,
                                         uint8_t *__restrict__ zero_obs) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const int nb = obs ? 2 : 1;
    const int br = i < R ? 0 : 1;
    const int64_t ag = br == 0 ? i : i - R;
    const bool in = i < R * nb;
    bool nz = false;
    if (in) {
        const int k = br == 0 ? kp : ko;
        const float2 *f = reinterpret_cast<const float2 *>((br == 0 ? ped : obs) + ag * k * 6);
        for (int j = 0; j < 3 * k; ++j) {
            const float2 x = f[j];
            nz = nz || x.x != 0.f || x.y != 0.f;
        }
        (br == 0 ? zero_ped : zero_obs)[ag] = nz ? 0 : 1;
    }
#pragma unroll
    for (int b2 = 0; b2 < 2; ++b2) {
        const unsigned mask = __ballot_sync(0xffffffffu, in && nz && br == b2);
        if (!mask) continue;
        const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
        int base = 0;
        if (lane == leader) base = atomicAdd(&counts[b2], __popc(mask));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (in && nz && br == b2) (b2 == 0 ? list_ped : list_obs)[base + __popc(mask & ((1u << lane) - 1))] = static_cast<int>(ag);
    }
}

// Compact mode 2, finish: per-branch outputs of the listed agents, g(0) for the others, + the destination term.
__global__ void pinnsf_tc_finish_compact2_kernel(const float *__restrict__ sums, const uint8_t *__restrict__ zero_ped,
                                                 const uint8_t *__restrict__ zero_obs, const float *__restrict__ f0,
                                                 const float *__restrict__ self, const float *__restrict__ dnorm,
                                                 int64_t R, int has_obs, float tau, float *__restrict__ acc) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= 2 * R) return;
    const int64_t ag = i >> 1;
    const int c = static_cast<int>(i & 1);
    const float *s = self + ag * 7;
    float nrm = dnorm ? dnorm[ag * 2 + c] : norm2_rn(s[0], s[1]);
    if (nrm == 0.f) nrm = __fadd_rn(nrm, 0.1f);
    const float dir = __fdiv_rn(s[c], nrm);
    const float dterm = __fdiv_rn(__fsub_rn(__fmul_rn(s[6], dir), s[2 + c]), tau);
    float mm = zero_ped[ag] ? f0[c] : sums[ag * 4 + c];
    if (has_obs) mm = __fadd_rn(mm, zero_obs[ag] ? f0[2 + c] : sums[ag * 4 + 2 + c]);
    acc[i] = __fadd_rn(mm, dterm);
}

// Compact mode, finish: acc = sum over the k slots (in slot order, f(0) for the zero rows) of both branches + the
// destination term -- the same additions in the same order as the in-tile sums of the dense mode.
__global__ void pinnsf_tc_finish_compact_kernel(const float *__restrict__ cmsg_ped, const float *__restrict__ cmsg_obs,
                                                const uint8_t *__restrict__ zero_ped,
                                                const uint8_t *__restrict__ zero_obs, const float *__restrict__ f0,
                                                const float *__restrict__ self, const float *__restrict__ dnorm,
                                                int64_t R, int kp, int ko, int has_obs, float tau,
                                                float *__restrict__ acc) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= 2 * R) return;
    const int64_t ag = i >> 1;
    const int c = static_cast<int>(i & 1);
    const float *s = self + ag * 7;
    float nrm = dnorm ? dnorm[ag * 2 + c] : norm2_rn(s[0], s[1]);
    if (nrm == 0.f) nrm = __fadd_rn(nrm, 0.1f);
    const float dir = __fdiv_rn(s[c], nrm);
    const float dterm = __fdiv_rn(__fsub_rn(__fmul_rn(s[6], dir), s[2 + c]), tau);
    float mm = 0.f;
    for (int j = 0; j < kp; ++j) {
        const int64_t r = ag * kp + j;
        mm += zero_ped[r] ? f0[c] : cmsg_ped[r * 2 + c];
    }
    if (has_obs) {
        float mo = 0.f;
        for (int j = 0; j < ko; ++j) {
            const int64_t r = ag * ko + j;
            mo += zero_obs[r] ? f0[2 + c] : cmsg_obs[r * 2 + c];
        }
        mm = __fadd_rn(mm, mo);
    }
    acc[i] = __fadd_rn(mm, dterm);
}

// Internal scratch of the tensor-core forward (per-agent sums, compact-mode lists and messages), cached per calling
// thread, device and stream; released by piml_free_workspace().
struct TcScratch { cudaStream_t st; int dev; float *buf; int64_t cap; };
static thread_local TcScratch g_tc_slots[8] = {};
static thread_local int g_tc_used = 0;

void tc_scratch_free() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return;
    for (int i = 0; i < g_tc_used; ++i)
        if (g_tc_slots[i].buf) {
            cudaSetDevice(g_tc_slots[i].dev);
            cudaStreamSynchronize(g_tc_slots[i].st);
            cudaFree(g_tc_slots[i].buf);
            g_tc_slots[i] = TcScratch{};
        }
    g_tc_used = 0;
    cudaSetDevice(dev);
}

static int tc_scratch_get(cudaStream_t st, int64_t floats, float **out) {
    TcScratch *slots = g_tc_slots;
    int &used = g_tc_used;
    int dev = 0;
    PIML_CUDA(cudaGetDevice(&dev));
    TcScratch *s = nullptr;
    for (int i = 0; i < used; ++i)
        if (slots[i].st == st && slots[i].dev == dev) s = &slots[i];
    if (!s) {
        s = &slots[used < 8 ? used++ : 7];
        if (s->buf) { cudaSetDevice(s->dev); cudaFree(s->buf); cudaSetDevice(dev); }
        s->st = st; s->dev = dev; s->buf = nullptr; s->cap = 0;
    }
    if (s->cap < floats) {
        if (s->buf) { PIML_CUDA(cudaStreamSynchronize(st)); PIML_CUDA(cudaFree(s->buf)); }
        s->buf = nullptr; s->cap = 0;
        PIML_CUDA(cudaMalloc(&s->buf, sizeof(float) * floats));
        s->cap = floats;
    }
    *out = s->buf;
    return PIML_OK;
}

}  // namespace piml

using namespace piml;

extern "C" int64_t piml_pinnsf_packed_tc_floats(const piml_net_desc *desc) {
    if (!desc) return -1;
    TcPlan P;
    TcPackTab T;
    if (tc_build_plan(desc, &P, &T)) return -1;
    Tc16Plan P16;                                                  // the 16-bit images follow the tf32 images
    if (tc16_build_plan(desc, P.total, &P16) == 0) return P16.base + 2 * P16.branch_floats;
    return P.total;
}

namespace piml {
int tc16_plan_for(const piml_net_desc *d, Tc16Plan *P16) {
    TcPlan P;
    TcPackTab T;
    if (d->kind != 0 || d->proc_mode != 0 || tc_build_plan(d, &P, &T)) return 1;
    return tc16_build_plan(d, P.total, P16);
}
}  // namespace piml

static void tc16_sources(const TcPlan &P, const TcPackTab &T, Tc16Src *S) {
    for (int br = 0; br < 2; ++br) {
        for (int l = 0; l < P.nl; ++l) {
            S->src_w[br * P.nl + l] = T.r[br * P.nl + l].src_w;
            S->src_b[br * P.nl + l] = T.r[br * P.nl + l].src_b;
        }
        S->pred_src[br] = T.pred_src[br];
    }
    for (int l = 0; l < P.nl; ++l) S->scale[l] = T.r[l].scale;
}

extern "C" int piml_pinnsf_pack_tc_f32(const piml_net_desc *desc, const float *params_torch, float *packed_tc,
                                       void *stream) {
    PIML_REQUIRE(desc && params_torch && packed_tc, "piml_pinnsf_pack_tc_f32: null pointer");
    TcPlan P;
    TcPackTab T;
    int rc = tc_build_plan(desc, &P, &T);
    if (rc) return rc;
    PIML_REQUIRE(aligned16(packed_tc), "piml_pinnsf_pack_tc_f32: packed_tc must be 16-byte aligned");
    const int threads = 256;
    pinnsf_pack_tc_kernel<<<static_cast<unsigned>((P.total + threads - 1) / threads), threads, 0,
                            static_cast<cudaStream_t>(stream)>>>(T, params_torch, packed_tc, P.nl, P.total / 2,
                                                                 P.b_off[0]);
    count_launch();
    rc = check_launch("pinnsf_pack_tc_kernel");
    if (rc) return rc;
    Tc16Plan P16;
    if (tc16_build_plan(desc, P.total, &P16) == 0) {
        Tc16Src S;
        tc16_sources(P, T, &S);
        rc = tc16_pack(P16, S, params_torch, packed_tc, static_cast<cudaStream_t>(stream));
    }
    return rc;
}

extern "C" int piml_pinnsf_forward_tc_f32(const piml_net_desc *desc, const float *packed_tc, int has_obs, float tau,
                                          const float *ped, const float *obs, const float *self, int64_t R, int kp,
                                          int ko, int norm_group, float *acc, float *ped_msgs, float *obs_msgs,
                                          void *stream) {
    PIML_REQUIRE(desc && packed_tc && ped && self && acc, "piml_pinnsf_forward_tc_f32: null pointer");
    PIML_REQUIRE(!has_obs || obs, "piml_pinnsf_forward_tc_f32: has_obs set but obs is null");
    PIML_REQUIRE(R >= 0 && kp >= 1 && ko >= 0 && kp <= 128 && ko <= 128, "piml_pinnsf_forward_tc_f32: bad dimensions");
    PIML_REQUIRE(aligned16(packed_tc), "piml_pinnsf_forward_tc_f32: packed_tc must be 16-byte aligned");
    if (!has_obs || ko == 0) { has_obs = 0; ko = 0; }
    TcPlan P;
    TcPackTab T;
    int rc = tc_build_plan(desc, &P, &T);
    if (rc) return rc;
    PIML_REQUIRE(P.kind == 0 || (!ped_msgs && !obs_msgs),
                 "piml_pinnsf_forward_tc_f32: per-slot embedding messages (kind 1) are only produced by the FP32 path");
    if (R == 0) return PIML_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    float *scratch = nullptr;
    // compact mode: messages not requested and the dense tiles exceed one wave (a scene whose dense tiles fit one wave
    // gains nothing from it and would pay two more launches)
    const int64_t dense_tiles = (R + 128 / kp - 1) / (128 / kp) + ((has_obs && ko) ? (R + 128 / ko - 1) / (128 / ko) : 0);
    const bool compact_ok = !ped_msgs && !obs_msgs && dense_tiles > sm_count() &&
                            R * static_cast<int64_t>(kp > ko ? kp : ko) < (1LL << 31);
    const bool compact = compact_ok && P.kind == 0;               // row level (per-slot decoders)
    const bool compact2 = compact_ok && P.kind == 1;              // agent level (summed embeddings)
    const int64_t rows_ped = R * kp, rows_obs = has_obs ? R * ko : 0, rows_all = rows_ped + rows_obs;
    // scratch (floats): sums R*4 | dnorm R*2 | messages rows_all*2 | lists rows_all | f0 4 + counts 2 (+2 pad) | flags
    const int64_t f_sums = R * 4, f_norm = norm_group > 0 ? R * 2 : 0;
    const int64_t f_extra = compact ? rows_all * 2 + rows_all + 8 + (rows_all + 3) / 4 + 4
                                    : (compact2 ? 2 * R + 8 + (2 * R + 3) / 4 + 4 : 0);
    rc = tc_scratch_get(st, f_sums + f_norm + f_extra, &scratch);
    if (rc) return rc;
    const float *dnorm = nullptr;
    if (norm_group > 0) {
        PIML_REQUIRE(R % norm_group == 0, "piml_pinnsf_forward_tc_f32: R not a multiple of norm_group");
        float *dn = scratch + R * 4;
        tc_colnorm_kernel<<<static_cast<unsigned>(R / norm_group), 128, 0, st>>>(self, norm_group, dn);
        count_launch();
        rc = check_launch("tc_colnorm_kernel");
        if (rc) return rc;
        dnorm = dn;
    }
    TcArgs a;
    a.params = packed_tc; a.ped = ped; a.obs = obs; a.R = R; a.kp = kp; a.ko = ko;
    a.ag_ped = 128 / kp; a.ag_obs = ko ? 128 / ko : 1;
    a.n_ped_tiles = (R + a.ag_ped - 1) / a.ag_ped;
    a.n_obs_tiles = has_obs ? (R + a.ag_obs - 1) / a.ag_obs : 0;
    a.sums = scratch; a.ped_msgs = ped_msgs; a.obs_msgs = has_obs ? obs_msgs : nullptr;
    a.compact = compact ? 1 : (compact2 ? 2 : 0);
    a.has_obs = has_obs ? 1 : 0;
    a.list_ped = a.list_obs = nullptr; a.counts = nullptr; a.cmsg_ped = a.cmsg_obs = a.f0 = nullptr;
    uint8_t *zero_ped = nullptr, *zero_obs = nullptr;
    if (compact) {
        float *x = scratch + f_sums + f_norm;
        a.cmsg_ped = x; a.cmsg_obs = x + rows_ped * 2; x += rows_all * 2;
        int *lists = reinterpret_cast<int *>(x); x += rows_all;
        a.list_ped = lists; a.list_obs = lists + rows_ped;
        a.f0 = x; int *counts = reinterpret_cast<int *>(x + 4); x += 8;
        a.counts = counts;
        zero_ped = reinterpret_cast<uint8_t *>(x); zero_obs = zero_ped + rows_ped;
        PIML_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(int), st));
        const int threads = 256;
        tc_compact_kernel<<<static_cast<unsigned>((rows_all + threads - 1) / threads), threads, 0, st>>>(
            ped, obs, rows_ped, rows_obs, lists, lists + rows_ped, counts, zero_ped, zero_obs);
        count_launch();
        rc = check_launch("tc_compact_kernel");
        if (rc) return rc;
    }
    const size_t smem = static_cast<size_t>(TC_STAGES) * TC_STAGE_BYTES +
                        sizeof(float) * (2 * P.bias_floats + 512 + 2 * 128 * TC_STAGE_LD) + 8 * (2 * TC_STAGES + 6) + 64;
    static thread_local bool attr_set = false;
    if (!attr_set) {
        PIML_CUDA(cudaFuncSetAttribute(pinnsf_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
        attr_set = true;
    }
    PIML_REQUIRE(smem <= 216 * 1024, "piml_pinnsf_forward_tc_f32: network too large for the shared-memory plan");
    // compact mode: the tile count is only known on the device (at most (rows + 1) / 128 + 1 per branch)
    if (compact2) {
        float *x = scratch + f_sums + f_norm;
        int *lists = reinterpret_cast<int *>(x); x += 2 * R;
        a.list_ped = lists; a.list_obs = lists + R;
        a.f0 = x; int *counts = reinterpret_cast<int *>(x + 4); x += 8;
        a.counts = counts;
        zero_ped = reinterpret_cast<uint8_t *>(x); zero_obs = zero_ped + R;
        PIML_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(int), st));
        const int threads = 256;
        const int64_t n = R * (has_obs ? 2 : 1);
        tc_compact_agents_kernel<<<static_cast<unsigned>((n + threads - 1) / threads), threads, 0, st>>>(
            ped, has_obs ? obs : nullptr, R, kp, ko, lists, lists + R, counts, zero_ped, zero_obs);
        count_launch();
        rc = check_launch("tc_compact_agents_kernel");
        if (rc) return rc;
    }
    const int64_t tiles = compact ? (rows_ped + 128) / 128 + (has_obs ? (rows_obs + 128) / 128 : 0)
                                  : a.n_ped_tiles + a.n_obs_tiles + (compact2 ? 2 : 0);
    // 16-bit path (two tiles in flight, resident weights) for every network its plan accepts; the agent-compact mode
    // (summed-embedding networks) only exists in the tf32 kernel
    Tc16Plan P16;
    if (!compact2 && tc16_build_plan(desc, P.total, &P16) == 0) {
        Tc16Args b;
        b.params = packed_tc; b.ped = ped; b.obs = obs; b.R = R; b.kp = kp; b.ko = ko;
        b.ag_ped = a.ag_ped; b.ag_obs = a.ag_obs; b.n_ped_tiles = a.n_ped_tiles; b.n_obs_tiles = a.n_obs_tiles;
        b.sums = a.sums; b.ped_msgs = a.ped_msgs; b.obs_msgs = a.obs_msgs;
        b.compact = compact ? 1 : 0; b.has_obs = a.has_obs;
        b.list_ped = a.list_ped; b.list_obs = a.list_obs; b.counts = a.counts;
        b.cmsg_ped = a.cmsg_ped; b.cmsg_obs = a.cmsg_obs; b.f0 = a.f0;
        rc = tc16_launch(P16, b, tiles, st);
    } else {
        const int grid = static_cast<int>(tiles < sm_count() ? tiles : sm_count());
        pinnsf_tc_kernel<<<grid, TC_THREADS, smem, st>>>(P, a);
        count_launch();
        rc = check_launch("pinnsf_tc_kernel");
    }
    if (rc) return rc;
    const int threads = 256;
    if (compact2) {
        pinnsf_tc_finish_compact2_kernel<<<static_cast<unsigned>((2 * R + threads - 1) / threads), threads, 0, st>>>(
            scratch, zero_ped, zero_obs, a.f0, self, dnorm, R, has_obs, tau, acc);
        count_launch();
        return check_launch("pinnsf_tc_finish_compact2_kernel");
    }
    if (compact) {
        pinnsf_tc_finish_compact_kernel<<<static_cast<unsigned>((2 * R + threads - 1) / threads), threads, 0, st>>>(
            a.cmsg_ped, a.cmsg_obs, zero_ped, zero_obs, a.f0, self, dnorm, R, kp, ko, has_obs, tau, acc);
        count_launch();
        return check_launch("pinnsf_tc_finish_compact_kernel");
    }
    pinnsf_tc_finish_kernel<<<static_cast<unsigned>((2 * R + threads - 1) / threads), threads, 0, st>>>(
        scratch, self, dnorm, R, has_obs, tau, acc);
    count_launch();
    return check_launch("pinnsf_tc_finish_kernel");
}

namespace piml {
// S networks of one description, set s on rows [s N, (s+1) N): the 16-bit kernel in dense mode with one (set, branch)
// per CTA, then the finish kernel on all S N rows.  sums: S N 4 floats of scratch.
int tc16_forward_sets(const piml_net_desc *desc, const float *packed_tc, int64_t set_stride, int S, int has_obs,
                      float tau, const float *ped, const float *obs, const float *self, int64_t N, int kp, int ko,
                      float *sums, float *acc, cudaStream_t st) {
    Tc16Plan P16;
    if (tc16_plan_for(desc, &P16))
        return fail(PIML_ERR_UNSUPPORTED, "piml_pinnsf_forward_tc_sets_f32: the 16-bit tensor-core path does not take "
                    "this network (per-slot decoders with hidden widths 32 / 64 / 128 only)");
    PIML_REQUIRE(set_stride >= piml_pinnsf_packed_tc_floats(desc) && set_stride % 4 == 0,
                 "piml_pinnsf_forward_tc_sets_f32: set_stride %lld must be a multiple of 4 and >= %lld "
                 "(piml_pinnsf_packed_tc_floats)", static_cast<long long>(set_stride),
                 static_cast<long long>(piml_pinnsf_packed_tc_floats(desc)));
    PIML_REQUIRE(aligned16(packed_tc), "piml_pinnsf_forward_tc_sets_f32: packed_tc must be 16-byte aligned");
    if (!has_obs || ko == 0) { has_obs = 0; ko = 0; }
    PIML_REQUIRE(!has_obs || obs, "piml_pinnsf_forward_tc_sets_f32: has_obs set but obs is null");
    const int64_t R = static_cast<int64_t>(S) * N;
    if (R == 0) return PIML_OK;
    Tc16Args b = {};
    b.params = packed_tc; b.ped = ped; b.obs = obs; b.R = N; b.kp = kp; b.ko = ko;
    b.ag_ped = 128 / kp; b.ag_obs = ko ? 128 / ko : 1;
    b.n_ped_tiles = (N + b.ag_ped - 1) / b.ag_ped;
    b.n_obs_tiles = has_obs ? (N + b.ag_obs - 1) / b.ag_obs : 0;
    b.sums = sums; b.has_obs = has_obs; b.set_stride = set_stride;
    int rc = tc16_launch_sets(P16, b, S, st);
    if (rc) return rc;
    const int threads = 256;
    pinnsf_tc_finish_kernel<<<static_cast<unsigned>((2 * R + threads - 1) / threads), threads, 0, st>>>(
        sums, self, nullptr, R, has_obs, tau, acc);
    count_launch();
    return check_launch("pinnsf_tc_finish_kernel");
}
}  // namespace piml

extern "C" int piml_pinnsf_forward_tc_sets_f32(const piml_net_desc *desc, const float *packed_tc, int64_t set_stride,
                                               int S, int has_obs, float tau, const float *ped, const float *obs,
                                               const float *self, int64_t N, int kp, int ko, float *acc,
                                               void *stream) {
    PIML_REQUIRE(desc && packed_tc && ped && self && acc, "piml_pinnsf_forward_tc_sets_f32: null pointer");
    PIML_REQUIRE(S >= 0 && N >= 0 && kp >= 1 && ko >= 0 && kp <= 128 && ko <= 128 &&
                     N * (kp > ko ? kp : ko) < (1LL << 31),
                 "piml_pinnsf_forward_tc_sets_f32: bad dimensions S=%d N=%lld kp=%d ko=%d", S,
                 static_cast<long long>(N), kp, ko);
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    float *sums = nullptr;
    if (static_cast<int64_t>(S) * N > 0) {
        const int rc = tc_scratch_get(st, static_cast<int64_t>(S) * N * 4, &sums);
        if (rc) return rc;
    }
    return tc16_forward_sets(desc, packed_tc, set_stride, S, has_obs, tau, ped, obs, self, N, kp, ko, sums, acc, st);
}
