// mlp_bwd.cu -- backward of the fused interaction networks for sm_100a (training rollouts and single-step training).
//
// Replaces what autograd does for the reference's `loss.backward()` through MLP / ResDNN / PINNSF* forwards
// (reference src/models/simulators.py:359 through src/models/model.py:40-119, :762-792, :1104-1135, :1185-1221,
// :1271-1305): per Linear an addmm for dX, an addmm for dW, a column sum for db, plus threshold/mul kernels.
// Here the backward is three kernels:
//   1. pinnsf_bwd_tile_kernel -- the dX CHAIN of a whole branch for a tile of 128 slot rows: the same register-tiled
//      dense layer as the forward (mlp_tile.cuh) applied to torch's own (out,in) weight matrices streamed by TMA,
//      ReLU masks / the ResDNN 2x-and-dropout fold taken from the forward's activation stash, every layer's
//      pre-activation gradient G_l written row-major for step 2, and the gradient of the 6-d input features;
//   2. pinnsf_dw_kernel -- dW_l = G_l^T A_{l-1}, db_l = sum_r G_l for ALL Linears in one launch
//      (grid = row splits x layers; 8x8 register tiles, packed FP32 FMAs), partial sums per split;
//   3. pinnsf_dw_reduce_kernel -- adds the split partials in a fixed order (deterministic, no atomics) and emits the
//      gradient in torch's own parameter layout (pack_state_dict order), plus pinnsf_finish_bwd_kernel for the
//      destination term (incl. the dim=1 norm quirk of channelled inputs, SURVEY.md B-3).
// Dead weights of the reference (ResDNN block 0 when processor_hidden_layers > 1, SURVEY.md B-4) receive no gradient,
// like the reference's `grad is None`.
#include "mlp_tile.cuh"

namespace piml {

struct BArgs {
    const float *wT; const float *stash; float *G;
    const float *drop_ped; const float *drop_obs;
    const float *g_acc; const float *g_ped_msgs; const float *g_obs_msgs; const float *g_coll;
    float *g_ped; float *g_obs;
    int64_t R; int kp, ko, ag_ped, ag_obs; int64_t n_ped_tiles, n_obs_tiles; int has_coll;
};

// buf[i][r] *= (act[r][i] > 0);  gout[r][i] = buf[i][r]      (threshold_backward of ReLU)
__device__ __forceinline__ void relu_mask_store(float *buf, const float *__restrict__ act, float *__restrict__ gout,
                                                int64_t r0, int n, int width) {
    tile_pass(width, n, [&](int i, int r) {
        float g = buf[i * FT_TRP + r];
        if (!(act[(r0 + r) * width + i] > 0.f)) g = 0.f;
        buf[i * FT_TRP + r] = g;
        gout[(r0 + r) * width + i] = g;
    });
}

// P is the TRANSPOSED plan (build_plan(..., true)): P.enc[l].K = forward OUT, P.enc[l].OUT = forward K.
__global__ void __launch_bounds__(FT_THREADS, 1) pinnsf_bwd_tile_kernel(const __grid_constant__ FPlan P,
                                                                        const __grid_constant__ FTab T,
                                                                        const __grid_constant__ BArgs a,
                                                                        const __grid_constant__ SPlan S,
                                                                        const __grid_constant__ SPlan Gp) {
    extern __shared__ __align__(128) float smem[];
    float *bufA = smem;
    float *bufB = bufA + FT_MAXW * FT_TRP;
    float *wbuf = bufB + FT_MAXW * FT_TRP;
    float *small = wbuf + 2 * FT_KC * FT_MAXW;                    // [FT_SMALL][FT_TRP]
    uint64_t *bars = reinterpret_cast<uint64_t *>(small + FT_SMALL * FT_TRP);
    const int tid = threadIdx.x;

    const int64_t tile = blockIdx.x;
    const int br = tile < a.n_ped_tiles ? 0 : 1;
    const int k = br == 0 ? a.kp : a.ko;
    const int AG = br == 0 ? a.ag_ped : a.ag_obs;
    const int64_t agent0 = (br == 0 ? tile : tile - a.n_ped_tiles) * AG;
    const int na = static_cast<int>(min(static_cast<int64_t>(AG), a.R - agent0));
    const int nrows = na * k;
    const int64_t row0 = agent0 * k;
    const float *pbase = a.wT + P.branch_off[br];
    const float *cb = a.wT + P.coll_off;
    const bool coll = br == 0 && P.n_coll > 0 && a.has_coll;
    const float *gmsg = br == 0 ? a.g_ped_msgs : a.g_obs_msgs;
    const float *drop = br == 0 ? a.drop_ped : a.drop_obs;

    WPipe wp;
    wp.base = a.wT; wp.tab = T.c[br]; wp.n = T.n[br]; wp.cons = 0; wp.wbuf = wbuf; wp.bars = bars; wp.phase = 0;
    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
        wp.issue(0);
    }
    float *cur = bufA, *oth = bufB;
    const int nd = P.n_dec, ne = P.n_enc;
    const int npred = P.kind == 0 ? nrows : na;                    // rows the decoder / predictor ran on
    const int64_t pred0 = P.kind == 0 ? row0 : agent0;

    // ---- gradients arriving at the predictor output and at the collision logit ----
    for (int e = tid; e < npred * 2; e += FT_THREADS) {
        const int r = e >> 1, c = e & 1;
        float g;
        if (P.kind == 0) {                   // acc = sum_k msg (model.py:1194): every slot gets its agent's gradient
            g = a.g_acc[(agent0 + r / k) * 2 + c];
            if (gmsg) g += gmsg[(row0 + r) * 2 + c];
        } else {
            g = a.g_acc[(agent0 + r) * 2 + c];
        }
        small[c * FT_TRP + r] = g;
        a.G[Gp.pred[br] + (pred0 + r) * 2 + c] = g;
    }
    if (coll)
        for (int r = tid; r < nrows; r += FT_THREADS) {           // sigmoid backward (model.py:1215 / :1299)
            const float p = a.stash[S.prob + row0 + r];
            const float g = a.g_coll ? a.g_coll[row0 + r] * p * (1.f - p) : 0.f;
            small[2 * FT_TRP + r] = g;
            a.G[Gp.prob + row0 + r] = g;
        }
    __syncthreads();                                               // barrier init + small visible

    // collision head backward into `dstbuf` (+= ), input gradient of the head has width P.coll[0].OUT
    auto coll_backward = [&](float *dstbuf, float *scratch) {
        if (P.n_coll == 2) {
            dense_any(wp, P.coll[1], cb, small + 2 * FT_TRP, scratch, nrows, false, 1.f);
            __syncthreads();
            relu_mask_store(scratch, a.stash + S.collh, a.G + Gp.collh, row0, nrows, P.coll[1].OUT);
            dense_any(wp, P.coll[0], cb, scratch, dstbuf, nrows, false, 1.f, dstbuf);
        } else {
            dense_any(wp, P.coll[0], cb, small + 2 * FT_TRP, dstbuf, nrows, false, 1.f, dstbuf);
        }
    };

    dense_any(wp, P.pred, pbase, small, cur, npred, false, 1.f);  // gradient of the last decoder output
    if (P.kind == 0 && coll) coll_backward(cur, oth);
    __syncthreads();
    store_tile(cur, a.G + Gp.dec[br][nd - 1], pred0, npred, P.dec[nd - 1].K);
    for (int l = nd - 1; l >= 0; --l) {
        dense_any(wp, P.dec[l], pbase, cur, oth, npred, false, 1.f);
        __syncthreads();
        if (l > 0) relu_mask_store(oth, a.stash + S.dec[br][l - 1], a.G + Gp.dec[br][l - 1], pred0, npred, P.dec[l].OUT);
        float *t = cur; cur = oth; oth = t;
    }
    if (P.kind == 1) {
        // cur = gradient of the per-agent embedding sum: broadcast to the k slots, add the message gradients
        const int pw = P.pw;
        tile_pass(pw, nrows, [&](int i, int r) {
            float g = cur[i * FT_TRP + r / k];
            if (gmsg) g += gmsg[(row0 + r) * pw + i];
            oth[i * FT_TRP + r] = g;
        });
        float *t = cur; cur = oth; oth = t;
        if (coll) coll_backward(cur, oth);                         // (the dense calls synchronise before reading)
        __syncthreads();
    }
    if (P.proc_mode == 1) {
        // single ResBlock y = (relu(W e + b) + e) * drop (model.py:68-79,118): g_e = g_y drop + (g_y drop . mask) W
        const int pw = P.pw;
        const float *dr = drop ? drop + row0 * pw : nullptr;
        const float *hp = a.stash + S.proc_h[br];
        float *gproc = a.G + Gp.proc[br];
        tile_pass(pw, nrows, [&](int i, int r) {
            float g = cur[i * FT_TRP + r];
            if (dr) g *= dr[static_cast<int64_t>(r) * pw + i];
            cur[i * FT_TRP + r] = g;
            const float gm = hp[(row0 + r) * pw + i] > 0.f ? g : 0.f;
            oth[i * FT_TRP + r] = gm;
            gproc[(row0 + r) * pw + i] = gm;
        });
        dense_any(wp, P.proc, pbase, oth, cur, nrows, false, 1.f, cur);
        __syncthreads();
        store_tile(cur, a.G + Gp.enc[br][ne - 1], row0, nrows, pw);
    } else {
        // ResDNN == 2x (+ dropout multipliers) folded into the last encoder layer (model.py:115-119)
        const int pw = P.pw;
        float *gout = a.G + Gp.enc[br][ne - 1];
        const float *dr = drop ? drop + row0 * pw : nullptr;
        tile_pass(pw, nrows, [&](int i, int r) {
            float g = cur[i * FT_TRP + r] * 2.f;
            if (dr) g *= dr[static_cast<int64_t>(r) * pw + i];
            cur[i * FT_TRP + r] = g;
            gout[(row0 + r) * pw + i] = g;
        });
    }
    for (int l = ne - 1; l >= 0; --l) {
        dense_any(wp, P.enc[l], pbase, cur, oth, nrows, false, 1.f);
        __syncthreads();
        if (l > 0) {
            relu_mask_store(oth, a.stash + S.enc[br][l - 1], a.G + Gp.enc[br][l - 1], row0, nrows, P.enc[l].OUT);
        } else {
            float *gx = br == 0 ? a.g_ped : a.g_obs;
            if (gx) store_tile(oth, gx, row0, nrows, P.enc[0].OUT);
        }
        float *t = cur; cur = oth; oth = t;
    }
}

// chunk consumption order of one branch -- must mirror pinnsf_bwd_tile_kernel exactly
static int build_chunks_bwd(const FPlan &P, int br, bool want_coll, FTab *T) {
    int n = 0;
    auto add = [&](const FLayer &L, int base) -> int {
        const int nch = (L.K + FT_KC - 1) / FT_KC;
        for (int c = 0; c < nch; ++c) {
            if (n >= FT_MAXCH) return -1;
            const int kc = L.K - c * FT_KC < FT_KC ? L.K - c * FT_KC : FT_KC;
            T->c[br][n].off = base + L.w_off + c * FT_KC * L.OUTP;
            T->c[br][n].bytes = kc * L.OUTP * static_cast<int>(sizeof(float));
            ++n;
        }
        return 0;
    };
    const int base = P.branch_off[br];
    const bool coll = want_coll && br == 0 && P.n_coll > 0;
    int bad = 0;
    auto add_coll = [&]() {
        if (P.n_coll == 2) { bad |= add(P.coll[1], P.coll_off); bad |= add(P.coll[0], P.coll_off); }
        else bad |= add(P.coll[0], P.coll_off);
    };
    bad |= add(P.pred, base);
    if (P.kind == 0 && coll) add_coll();
    for (int l = P.n_dec - 1; l >= 0; --l) bad |= add(P.dec[l], base);
    if (P.kind == 1 && coll) add_coll();
    if (P.proc_mode == 1) bad |= add(P.proc, base);
    for (int l = P.n_enc - 1; l >= 0; --l) bad |= add(P.enc[l], base);
    T->n[br] = n;
    return bad;
}

// ---- dW / db -----------------------------------------------------------------------------------------------
struct DwJob { const float *A; const float *G; int64_t rows; int K, OUT; int64_t dst; };
// One job per Linear: per branch the encoders, the single processor block, the decoders and the predictor, then the
// collision head.  The largest net build_plan accepts needs 2 * (8 + 1 + 8 + 1) + 2 = 38 (piml_b200/_lib.py
// PINNSF_DW_JOBS mirrors this number for the CPU tests).
constexpr int DW_MAX_JOBS = 38;
static_assert(DW_MAX_JOBS == 2 * (sizeof(FPlan::enc) / sizeof(FLayer) + 1 + sizeof(FPlan::dec) / sizeof(FLayer) + 1) +
                                 sizeof(FPlan::coll) / sizeof(FLayer),
              "DwTab must hold one job per Linear of the largest net build_plan accepts");
struct DwTab { int n; DwJob j[DW_MAX_JOBS]; };
constexpr int DW_ROWS = 32;
constexpr int DW_LD = 132;

// grid = (row splits, Linears).  ws[split][dst + o*K + k] = sum_r G[r][o] A[r][k];  ws[split][dst + OUT*K + o] = sum_r G[r][o]
__global__ void __launch_bounds__(256) pinnsf_dw_kernel(const __grid_constant__ DwTab T, float *__restrict__ ws,
                                                        int64_t t_total) {
    __shared__ __align__(16) float As[DW_ROWS][DW_LD];
    __shared__ __align__(16) float Gs[DW_ROWS][DW_LD];
    const DwJob &J = T.j[blockIdx.y];
    const int tid = threadIdx.x, to = tid & 15, tk = tid >> 4;
    const int K = J.K, OUT = J.OUT;
    const int Kp = (K + 7) & ~7, Op = (OUT + 7) & ~7;
    const int64_t nchunks = (J.rows + DW_ROWS - 1) / DW_ROWS;
    const int64_t c0 = nchunks * blockIdx.x / gridDim.x, c1 = nchunks * (blockIdx.x + 1) / gridDim.x;
    const bool active = to * 8 < OUT && tk * 8 < K;
    float2 acc[8][4];
    float bacc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        bacc[i] = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = make_float2(0.f, 0.f);
    }
    for (int64_t c = c0; c < c1; ++c) {
        const int64_t r0 = c * DW_ROWS;
        const int nr = static_cast<int>(min(static_cast<int64_t>(DW_ROWS), J.rows - r0));
        for (int e = tid; e < DW_ROWS * Kp; e += 256) {
            const int r = e / Kp, kk = e - r * Kp;
            As[r][kk] = (r < nr && kk < K) ? J.A[(r0 + r) * K + kk] : 0.f;
        }
        for (int e = tid; e < DW_ROWS * Op; e += 256) {
            const int r = e / Op, o = e - r * Op;
            Gs[r][o] = (r < nr && o < OUT) ? J.G[(r0 + r) * OUT + o] : 0.f;
        }
        __syncthreads();
        if (active) {
#pragma unroll 4
            for (int r = 0; r < DW_ROWS; ++r) {
                const float4 g0 = *reinterpret_cast<const float4 *>(&Gs[r][to * 8]);
                const float4 g1 = *reinterpret_cast<const float4 *>(&Gs[r][to * 8 + 4]);
                const float4 a0 = *reinterpret_cast<const float4 *>(&As[r][tk * 8]);
                const float4 a1 = *reinterpret_cast<const float4 *>(&As[r][tk * 8 + 4]);
                const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
                const float2 x[4] = {make_float2(a0.x, a0.y), make_float2(a0.z, a0.w), make_float2(a1.x, a1.y),
                                     make_float2(a1.z, a1.w)};
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float2 gg = make_float2(g[i], g[i]);
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = __ffma2_rn(gg, x[j], acc[i][j]);
                    bacc[i] += g[i];
                }
            }
        }
        __syncthreads();
    }
    if (!active) return;
    float *out = ws + static_cast<int64_t>(blockIdx.x) * t_total + J.dst;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int o = to * 8 + i;
        if (o >= OUT) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int kk = tk * 8 + 2 * j;
            if (kk < K) out[static_cast<int64_t>(o) * K + kk] = acc[i][j].x;
            if (kk + 1 < K) out[static_cast<int64_t>(o) * K + kk + 1] = acc[i][j].y;
        }
        if (tk == 0) out[static_cast<int64_t>(OUT) * K + o] = bacc[i];
    }
}

__global__ void pinnsf_dw_reduce_kernel(const float *__restrict__ ws, int nsplit, int64_t t_total,
                                        float *__restrict__ g_params) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= t_total) return;
    float s = 0.f;
    for (int sp = 0; sp < nsplit; ++sp) s += ws[static_cast<int64_t>(sp) * t_total + i];
    g_params[i] = s;
}

// ---- destination term backward (model.py:1205-1210) --------------------------------------------------------------
// acc = ... + (v0 * x / n - v) / tau,  x = self[:, 0:2], v = self[:, 2:4], v0 = self[:, 6];
// group == 0: n = ||x|| per row; group > 0: n_q = ||x[:, q]|| over the `group` agents of a channel (dim=1 quirk).
// n == 0 -> n = 0.1 with no gradient through the norm (torch.norm's subgradient at 0 is 0).
__global__ void pinnsf_finish_bwd_kernel(const float *__restrict__ g_acc, const float *__restrict__ self, int64_t R,
                                         int group, float tau, float *__restrict__ g_self) {
    __shared__ float red[4][128];
    const float itau = 1.f / tau;
    if (group == 0) {
        const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
        if (i >= R) return;
        const float *s = self + i * 7;
        const float x0 = s[0], x1 = s[1], v0 = s[6];
        const float ga0 = g_acc[i * 2], ga1 = g_acc[i * 2 + 1];
        const float gd0 = ga0 * v0 * itau, gd1 = ga1 * v0 * itau;
        const float n = sqrtf(fmaf(x1, x1, x0 * x0));
        float gx0, gx1, d0, d1;
        if (n == 0.f) {
            gx0 = gd0 / 0.1f; gx1 = gd1 / 0.1f; d0 = x0 / 0.1f; d1 = x1 / 0.1f;
        } else {
            const float dot = gd0 * x0 + gd1 * x1;
            const float in = 1.f / n, in3 = in * in * in;
            gx0 = gd0 * in - x0 * dot * in3; gx1 = gd1 * in - x1 * dot * in3;
            d0 = x0 * in; d1 = x1 * in;
        }
        float *g = g_self + i * 7;
        g[0] = gx0; g[1] = gx1; g[2] = -ga0 * itau; g[3] = -ga1 * itau; g[4] = 0.f; g[5] = 0.f;
        g[6] = (ga0 * d0 + ga1 * d1) * itau;
        return;
    }
    const int64_t base = static_cast<int64_t>(blockIdx.x) * group;
    float s0 = 0.f, s1 = 0.f, t0 = 0.f, t1 = 0.f;
    for (int i = threadIdx.x; i < group; i += blockDim.x) {
        const float *s = self + (base + i) * 7;
        const float x0 = s[0], x1 = s[1], v0 = s[6];
        s0 = fmaf(x0, x0, s0); s1 = fmaf(x1, x1, s1);
        t0 = fmaf(g_acc[(base + i) * 2] * v0 * itau, x0, t0);
        t1 = fmaf(g_acc[(base + i) * 2 + 1] * v0 * itau, x1, t1);
    }
    red[0][threadIdx.x] = s0; red[1][threadIdx.x] = s1; red[2][threadIdx.x] = t0; red[3][threadIdx.x] = t1;
    __syncthreads();
    for (int off = blockDim.x / 2; off > 0; off >>= 1) {
        if (threadIdx.x < off)
#pragma unroll
            for (int q = 0; q < 4; ++q) red[q][threadIdx.x] += red[q][threadIdx.x + off];
        __syncthreads();
    }
    const float n0 = sqrtf(red[0][0]), n1 = sqrtf(red[1][0]);
    const float in0 = 1.f / (n0 == 0.f ? 0.1f : n0), in1 = 1.f / (n1 == 0.f ? 0.1f : n1);
    const float c0 = n0 == 0.f ? 0.f : red[2][0] * in0 * in0 * in0, c1 = n1 == 0.f ? 0.f : red[3][0] * in1 * in1 * in1;
    for (int i = threadIdx.x; i < group; i += blockDim.x) {
        const float *s = self + (base + i) * 7;
        const float x0 = s[0], x1 = s[1], v0 = s[6];
        const float ga0 = g_acc[(base + i) * 2], ga1 = g_acc[(base + i) * 2 + 1];
        float *g = g_self + (base + i) * 7;
        g[0] = ga0 * v0 * itau * in0 - x0 * c0;
        g[1] = ga1 * v0 * itau * in1 - x1 * c1;
        g[2] = -ga0 * itau; g[3] = -ga1 * itau; g[4] = 0.f; g[5] = 0.f;
        g[6] = (ga0 * x0 * in0 + ga1 * x1 * in1) * itau;
    }
}

// Row splits of the dW kernel: one per 128 rows up to 64, so that a training batch of 128 samples (1-2k slot rows)
// already spreads every Linear over ~10 CTAs instead of one (295 -> ~40 us), and large batches get 64 x Linears CTAs.
static int dw_splits(int64_t max_rows) {
    int64_t s = (max_rows + 127) / 128;
    return static_cast<int>(s < 1 ? 1 : (s > 64 ? 64 : s));
}

}  // namespace piml

using namespace piml;

extern "C" int64_t piml_pinnsf_packed_bwd_floats(const piml_net_desc *desc) {
    if (!desc) return -1;
    FPlan P;
    PackTab PT;
    if (build_plan(desc, &P, &PT, true)) return -1;
    return P.total;
}

extern "C" int piml_pinnsf_pack_bwd_f32(const piml_net_desc *desc, const float *params_torch, float *packed_bwd,
                                        void *stream) {
    PIML_REQUIRE(desc && params_torch && packed_bwd, "piml_pinnsf_pack_bwd_f32: null pointer");
    FPlan P;
    PackTab PT;
    int rc = build_plan(desc, &P, &PT, true);
    if (rc) return rc;
    PIML_REQUIRE(aligned16(packed_bwd), "piml_pinnsf_pack_bwd_f32: packed_bwd must be 16-byte aligned");
    const int threads = 256;
    pinnsf_pack_kernel<<<static_cast<unsigned>((P.total + threads - 1) / threads), threads, 0,
                         static_cast<cudaStream_t>(stream)>>>(PT, params_torch, packed_bwd, P.total);
    count_launch();
    return check_launch("pinnsf_pack_kernel");
}

extern "C" int64_t piml_pinnsf_backward_workspace_floats(const piml_net_desc *desc, int has_obs, int64_t R, int kp,
                                                         int ko) {
    if (!desc || R < 0 || kp < 1 || ko < 0) return -1;
    FPlan P;
    PackTab PT;
    if (build_plan(desc, &P, &PT)) return -1;
    if (!has_obs || ko == 0) { has_obs = 0; ko = 0; }
    const SPlan G = make_splan(P, has_obs != 0, R, kp, ko, true);
    const int64_t maxrows = R * (kp > ko ? kp : ko);
    return G.total + static_cast<int64_t>(dw_splits(maxrows)) * ((P.t_total + 3) / 4 * 4);
}

extern "C" int piml_pinnsf_backward_f32(const piml_net_desc *desc, const float *packed_bwd, int has_obs, float tau,
                                        const float *ped, const float *obs, const float *self, int64_t R, int kp,
                                        int ko, int norm_group, const float *drop_ped, const float *drop_obs,
                                        const float *stash, const float *g_acc, const float *g_ped_msgs,
                                        const float *g_obs_msgs, const float *g_coll, float *g_params, float *g_ped,
                                        float *g_obs, float *g_self, float *workspace, void *stream) {
    PIML_REQUIRE(desc && packed_bwd && g_params, "piml_pinnsf_backward_f32: null pointer");
    PIML_REQUIRE(R >= 0 && kp >= 1 && ko >= 0 && kp <= FT_TR && ko <= FT_TR, "piml_pinnsf_backward_f32: bad dimensions");
    if (!has_obs || ko == 0) { has_obs = 0; ko = 0; }
    FPlan P, Pt;
    PackTab PT;
    int rc = build_plan(desc, &P, &PT);
    if (rc) return rc;
    rc = build_plan(desc, &Pt, &PT, true);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t t_total = P.t_total, t_pad = (t_total + 3) / 4 * 4;
    if (R == 0) {                      // empty batch: the row buffers may be null (torch's empty tensors are)
        PIML_CUDA(cudaMemsetAsync(g_params, 0, sizeof(float) * t_total, st));
        return PIML_OK;
    }
    PIML_REQUIRE(ped && self && stash && g_acc && workspace, "piml_pinnsf_backward_f32: null pointer");
    PIML_REQUIRE(!has_obs || obs, "piml_pinnsf_backward_f32: has_obs set but obs is null");
    PIML_REQUIRE(aligned16(packed_bwd) && aligned16(workspace),
                 "piml_pinnsf_backward_f32: packed_bwd and workspace must be 16-byte aligned");
    const bool coll = P.n_coll > 0;
    const SPlan S = make_splan(P, has_obs != 0, R, kp, ko, true);
    const SPlan Gp = S;                                            // same shapes
    float *G = workspace;
    float *ws = workspace + Gp.total;
    const int nsplit = dw_splits(R * (kp > ko ? kp : ko));

    // 1. dX chain
    FTab T;
    T.n[1] = 0;
    PIML_REQUIRE(build_chunks_bwd(Pt, 0, coll, &T) == 0 && (!has_obs || build_chunks_bwd(Pt, 1, false, &T) == 0),
                 "piml_pinnsf_backward_f32: network needs more than %d weight chunks per branch", FT_MAXCH);
    BArgs a;
    a.wT = packed_bwd; a.stash = stash; a.G = G; a.drop_ped = drop_ped; a.drop_obs = drop_obs;
    a.g_acc = g_acc; a.g_ped_msgs = g_ped_msgs; a.g_obs_msgs = has_obs ? g_obs_msgs : nullptr; a.g_coll = g_coll;
    a.g_ped = g_ped; a.g_obs = has_obs ? g_obs : nullptr;
    a.R = R; a.kp = kp; a.ko = ko;
    a.ag_ped = FT_TR / kp; a.ag_obs = ko ? FT_TR / ko : 1;
    a.n_ped_tiles = (R + a.ag_ped - 1) / a.ag_ped;
    a.n_obs_tiles = has_obs ? (R + a.ag_obs - 1) / a.ag_obs : 0;
    a.has_coll = coll ? 1 : 0;
    const size_t smem = sizeof(float) * (2 * FT_MAXW * FT_TRP + 2 * FT_KC * FT_MAXW + FT_SMALL * FT_TRP) + 16;
    // per launch: the attribute is per DEVICE, and a process may touch several (it costs well under a microsecond)
    PIML_CUDA(cudaFuncSetAttribute(pinnsf_bwd_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(smem)));
    const int64_t tiles = a.n_ped_tiles + a.n_obs_tiles;
    PIML_REQUIRE(tiles < (1LL << 31), "piml_pinnsf_backward_f32: too many tiles");
    pinnsf_bwd_tile_kernel<<<static_cast<unsigned>(tiles), FT_THREADS, smem, st>>>(Pt, T, a, S, Gp);
    count_launch();
    rc = check_launch("pinnsf_bwd_tile_kernel");
    if (rc) return rc;

    // 2. dW / db of every Linear
    DwTab J;
    J.n = 0;
    auto job = [&](const float *A, int64_t goff, int64_t rows, const FLayer &L, int64_t tbase) -> int {
        PIML_REQUIRE(J.n < DW_MAX_JOBS, "piml_pinnsf_backward_f32: more than %d Linears", DW_MAX_JOBS);
        DwJob &j = J.j[J.n++];
        j.A = A; j.G = G + goff; j.rows = rows; j.K = L.K; j.OUT = L.OUT; j.dst = tbase + L.t_off;
        return PIML_OK;
    };
    for (int br = 0; br < (has_obs ? 2 : 1); ++br) {
        const int64_t rows = R * (br == 0 ? kp : ko);
        const int64_t prow = P.kind == 0 ? rows : R;
        const float *feat = br == 0 ? ped : obs;
        const int64_t tb = P.t_branch_off[br];
        for (int l = 0; l < P.n_enc; ++l)
            rc |= job(l == 0 ? feat : stash + S.enc[br][l - 1], Gp.enc[br][l], rows, P.enc[l], tb);
        const float *proc_out = P.proc_mode == 1 ? stash + S.proc[br] : stash + S.enc[br][P.n_enc - 1];
        if (P.proc_mode == 1) rc |= job(stash + S.enc[br][P.n_enc - 1], Gp.proc[br], rows, P.proc, tb);
        for (int l = 0; l < P.n_dec; ++l) {
            const float *A = l > 0 ? stash + S.dec[br][l - 1] : (P.kind == 0 ? proc_out : stash + S.sum[br]);
            rc |= job(A, Gp.dec[br][l], prow, P.dec[l], tb);
        }
        rc |= job(stash + S.dec[br][P.n_dec - 1], Gp.pred[br], prow, P.pred, tb);
    }
    if (coll) {
        const int64_t rows = R * kp;
        const float *A0 = P.kind == 0 ? stash + S.dec[0][P.n_dec - 1]
                                      : (P.proc_mode == 1 ? stash + S.proc[0] : stash + S.enc[0][P.n_enc - 1]);
        if (P.n_coll == 2) {
            rc |= job(A0, Gp.collh, rows, P.coll[0], P.t_coll_off);
            rc |= job(stash + S.collh, Gp.prob, rows, P.coll[1], P.t_coll_off);
        } else {
            rc |= job(A0, Gp.prob, rows, P.coll[0], P.t_coll_off);
        }
    }
    if (rc) return rc;
    PIML_CUDA(cudaMemsetAsync(ws, 0, sizeof(float) * t_pad * nsplit, st));
    pinnsf_dw_kernel<<<dim3(nsplit, J.n), 256, 0, st>>>(J, ws, t_pad);
    count_launch();
    rc = check_launch("pinnsf_dw_kernel");
    if (rc) return rc;
    pinnsf_dw_reduce_kernel<<<static_cast<unsigned>((t_total + 255) / 256), 256, 0, st>>>(ws, nsplit, t_pad, g_params);
    count_launch();
    rc = check_launch("pinnsf_dw_reduce_kernel");
    if (rc) return rc;

    // 3. destination term
    if (g_self) {
        if (norm_group > 0) {
            PIML_REQUIRE(R % norm_group == 0, "piml_pinnsf_backward_f32: R not a multiple of norm_group");
            pinnsf_finish_bwd_kernel<<<static_cast<unsigned>(R / norm_group), 128, 0, st>>>(g_acc, self, R, norm_group,
                                                                                              tau, g_self);
        } else {
            pinnsf_finish_bwd_kernel<<<static_cast<unsigned>((R + 127) / 128), 128, 0, st>>>(g_acc, self, R, 0, tau,
                                                                                              g_self);
        }
        count_launch();
        rc = check_launch("pinnsf_finish_bwd_kernel");
        if (rc) return rc;
    }
    return PIML_OK;
}
