// mlp.cu -- fused forward of the physics-infused interaction networks for sm_100a.
//
// Replaces MLP / ResBlock / ResDNN (reference src/models/model.py:40-119) and the forwards of PINNSF (:762-792),
// PINNSF_bottleneck (:1104-1135), PINNSF_bottleneck_multitask (:1185-1221) and PINNSF_multitask (:1271-1305).
// The reference runs 9-11 MKL/cuBLAS addmm calls plus elementwise kernels per forward.  Here ONE kernel takes a tile
// of up to 128 neighbour-slot rows (whole agents of one branch: 21 agents x 6 pedestrian slots, or 12 agents x 10
// obstacle slots) through encoder -> processor -> decoder -> predictor (-> collision head):
//   * activations live in shared memory TRANSPOSED ([feature][row]), ping-ponged between two 128x132 buffers;
//   * every Linear is a register-tiled GEMM: 256 threads x (8 rows x 8 outputs), packed FP32 FMAs (FFMA2) with the
//     weight as the broadcast operand, fp32 accumulation (1e-5 parity with the reference rules out TF32);
//   * weights stream from L2 in 32-row chunks by TMA bulk copies (cp.async.bulk, double buffered on mbarriers), the
//     next chunk -- also across layer boundaries -- in flight while the current one is consumed;
//   * weights come pre-permuted (piml_pinnsf_pack_f32) so that each thread's 8 output columns {tc + 16 j} are two
//     conflict-free float4 loads and the transposed stores of a warp hit 32 distinct banks.
// Per-agent message sums go to a small workspace; pinnsf_finish_kernel adds the destination (social-force driving)
// term.  Every agent's sum is produced by exactly one CTA in a fixed order: results are run-to-run deterministic.
//
// Reference quirks reproduced on purpose (SURVEY.md Appendix B): ResDNN with >1 layers is exactly 2*x (B-4);
// zero-padded neighbour slots are NOT masked and contribute f(0) (B-5); the destination norm of a channelled
// (C,N,7) input reduces over the agent axis (B-3) -- handled by dest_colnorm_kernel.
#include <math_constants.h>

#include "common.cuh"

#include "mlp_tile.cuh"

namespace piml {

struct FArgs {
    const float *params; const float *ped; const float *obs; const float *drop_ped; const float *drop_obs;
    int64_t R; int kp, ko, ag_ped, ag_obs; int64_t n_ped_tiles, n_obs_tiles;
    float *sums;                      // (R,4): ped.x ped.y obs.x obs.y
    float *ped_msgs; float *obs_msgs; float *coll;
    float *stash;                     // training mode: activations kept for the backward (layout SPlan), or NULL
};

__global__ void __launch_bounds__(FT_THREADS, 1) pinnsf_tile_kernel(const __grid_constant__ FPlan P,
                                                                    const __grid_constant__ FTab T,
                                                                    const __grid_constant__ FArgs a,
                                                                    const __grid_constant__ SPlan S) {
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
    const float *pbase = a.params + P.branch_off[br];
    const bool want_coll = br == 0 && P.n_coll > 0 && a.coll != nullptr;

    WPipe wp;
    wp.base = a.params; wp.tab = T.c[br]; wp.n = T.n[br]; wp.cons = 0; wp.wbuf = wbuf; wp.bars = bars; wp.phase = 0;
    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
        wp.issue(0);
    }
    // stage the 6-d features transposed: bufA[c][r]
    {
        const float *feat = (br == 0 ? a.ped : a.obs) + row0 * 6;
        for (int e = tid; e < nrows * 6; e += FT_THREADS) bufA[(e % 6) * FT_TRP + (e / 6)] = feat[e];
    }
    __syncthreads();                                               // barrier init + features visible
    float *cur = bufA, *oth = bufB;
    const float *drop = br == 0 ? a.drop_ped : a.drop_obs;
    if (drop) drop += row0 * P.pw;

    for (int l = 0; l < P.n_enc; ++l) {      // MLP: ReLU between layers, Identity at the end (model.py:54-61)
        const bool last = l == P.n_enc - 1;
        const bool fold = last && P.proc_mode == 0;                // ResDNN == 2x (+ dropout)
        dense_any(wp, P.enc[l], pbase, cur, oth, nrows, !last, fold ? 2.f : 1.f, nullptr, fold ? drop : nullptr, P.pw);
        float *t = cur; cur = oth; oth = t;
        if (a.stash) { __syncthreads(); store_tile(cur, a.stash + S.enc[br][l], row0, nrows, P.enc[l].OUT); }
    }
    if (P.proc_mode == 1) {                  // single ResBlock: relu(Wx+b) + x, then dropout (model.py:68-79,118)
        if (a.stash) {                       // training: keep relu(Wx+b) and the block output for the backward
            dense_any(wp, P.proc, pbase, cur, oth, nrows, true, 1.f);
            __syncthreads();
            store_tile(oth, a.stash + S.proc_h[br], row0, nrows, P.pw);
            const int pw = P.pw;
            float *yout = a.stash + S.proc[br];
            tile_pass(pw, nrows, [&](int i, int r) {
                float y = oth[i * FT_TRP + r] + cur[i * FT_TRP + r];
                if (drop) y *= drop[static_cast<int64_t>(r) * pw + i];
                oth[i * FT_TRP + r] = y;
                yout[(row0 + r) * pw + i] = y;
            });
        } else {
            dense_any(wp, P.proc, pbase, cur, oth, nrows, true, 1.f, cur, drop, P.pw);
        }
        float *t = cur; cur = oth; oth = t;
    }
    float *msgs_out = br == 0 ? a.ped_msgs : a.obs_msgs;

    if (P.kind == 0) {
        // per-slot decoder -> predictor; messages are 2-d (model.py:1190-1194)
        for (int l = 0; l < P.n_dec; ++l) {
            dense_any(wp, P.dec[l], pbase, cur, oth, nrows, l < P.n_dec - 1, 1.f);
            float *t = cur; cur = oth; oth = t;
            if (a.stash) { __syncthreads(); store_tile(cur, a.stash + S.dec[br][l], row0, nrows, P.dec[l].OUT); }
        }
        dense_any(wp, P.pred, pbase, cur, small, nrows, false, 1.f);
        if (want_coll) {                     // collision head on the decoder output (model.py:1214-1215)
            const float *cb = a.params + P.coll_off;
            const float *h = cur;
            for (int l = 0; l < P.n_coll; ++l) {
                const bool last = l == P.n_coll - 1;
                dense_any(wp, P.coll[l], cb, h, last ? small + 2 * FT_TRP : oth, nrows, !last, 1.f);
                h = oth;
                if (a.stash && !last) { __syncthreads(); store_tile(oth, a.stash + S.collh, row0, nrows, P.coll[l].OUT); }
            }
        }
        __syncthreads();
        if (want_coll)
            for (int r = tid; r < nrows; r += FT_THREADS) {
                const float pr = 1.f / (1.f + expf(-small[2 * FT_TRP + r]));
                a.coll[row0 + r] = pr;
                if (a.stash) a.stash[S.prob + row0 + r] = pr;
            }
        if (msgs_out)
            for (int e = tid; e < nrows * 2; e += FT_THREADS) msgs_out[row0 * 2 + e] = small[(e & 1) * FT_TRP + (e >> 1)];
        if (tid < 2 * na) {                  // torch.sum(dim=-2) over the k slots (model.py:1194/1202)
            const int ag = tid >> 1, c = tid & 1;
            float s = 0.f;
            for (int j = 0; j < k; ++j) s += small[c * FT_TRP + ag * k + j];
            a.sums[(agent0 + ag) * 4 + br * 2 + c] = s;
        }
    } else {
        // messages are the processor outputs; sum over slots, then decode per agent (model.py:1276-1279)
        __syncthreads();
        if (msgs_out)
            for (int e = tid; e < nrows * P.pw; e += FT_THREADS) {
                const int r = e / P.pw, i = e % P.pw;
                msgs_out[(row0 + r) * P.pw + i] = cur[i * FT_TRP + r];
            }
        if (want_coll) {                     // collision head on the per-slot messages (model.py:1298-1299)
            const float *cb = a.params + P.coll_off;
            const float *h = cur;
            for (int l = 0; l < P.n_coll; ++l) {
                const bool last = l == P.n_coll - 1;
                dense_any(wp, P.coll[l], cb, h, last ? small + 2 * FT_TRP : oth, nrows, !last, 1.f);
                h = oth;
                if (a.stash && !last) { __syncthreads(); store_tile(oth, a.stash + S.collh, row0, nrows, P.coll[l].OUT); }
            }
            __syncthreads();
            for (int r = tid; r < nrows; r += FT_THREADS) {
                const float pr = 1.f / (1.f + expf(-small[2 * FT_TRP + r]));
                a.coll[row0 + r] = pr;
                if (a.stash) a.stash[S.prob + row0 + r] = pr;
            }
        }
        for (int e = tid; e < na * P.pw; e += FT_THREADS) {
            const int i = e / na, ag = e % na;
            float s = 0.f;
            for (int j = 0; j < k; ++j) s += cur[i * FT_TRP + ag * k + j];
            oth[i * FT_TRP + ag] = s;
        }
        { float *t = cur; cur = oth; oth = t; }
        if (a.stash) { __syncthreads(); store_tile(cur, a.stash + S.sum[br], agent0, na, P.pw); }
        for (int l = 0; l < P.n_dec; ++l) {
            dense_any(wp, P.dec[l], pbase, cur, oth, na, l < P.n_dec - 1, 1.f);
            float *t = cur; cur = oth; oth = t;
            if (a.stash) { __syncthreads(); store_tile(cur, a.stash + S.dec[br][l], agent0, na, P.dec[l].OUT); }
        }
        dense_any(wp, P.pred, pbase, cur, small, na, false, 1.f);
        __syncthreads();
        if (tid < 2 * na) {
            const int ag = tid >> 1, c = tid & 1;
            a.sums[(agent0 + ag) * 4 + br * 2 + c] = small[c * FT_TRP + ag];
        }
    }
}

// acc = sum_ped + sum_obs + (v0 * dest/||dest|| - v) / tau      (model.py:1205-1212)
__global__ void pinnsf_finish_kernel(const float *__restrict__ sums, const float *__restrict__ self,
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
    float m = sums[ag * 4 + c];
    if (has_obs) m = __fadd_rn(m, sums[ag * 4 + 2 + c]);
    acc[i] = __fadd_rn(m, dterm);
}

// column norms over the agent axis for channelled (C,N,7) inputs: dnorm[(c*N+n)*2 + q] = ||self[c,:,q]||_2
__global__ void dest_colnorm_kernel(const float *__restrict__ self, int group, float *__restrict__ dnorm) {
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
        if (threadIdx.x < off) {
            red[0][threadIdx.x] += red[0][threadIdx.x + off];
            red[1][threadIdx.x] += red[1][threadIdx.x + off];
        }
        __syncthreads();
    }
    const float n0 = sqrtf(red[0][0]), n1 = sqrtf(red[1][0]);
    for (int i = threadIdx.x; i < group; i += blockDim.x) {
        dnorm[(base + i) * 2] = n0;
        dnorm[(base + i) * 2 + 1] = n1;
    }
}

// chunk consumption order of one branch -- must mirror pinnsf_tile_kernel exactly
static int build_chunks(const FPlan &P, int br, bool want_coll, FTab *T) {
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
    int bad = 0;
    for (int l = 0; l < P.n_enc; ++l) bad |= add(P.enc[l], base);
    if (P.proc_mode == 1) bad |= add(P.proc, base);
    const bool coll = want_coll && br == 0 && P.n_coll > 0;
    if (P.kind == 0) {
        for (int l = 0; l < P.n_dec; ++l) bad |= add(P.dec[l], base);
        bad |= add(P.pred, base);
        if (coll) for (int l = 0; l < P.n_coll; ++l) bad |= add(P.coll[l], P.coll_off);
    } else {
        if (coll) for (int l = 0; l < P.n_coll; ++l) bad |= add(P.coll[l], P.coll_off);
        for (int l = 0; l < P.n_dec; ++l) bad |= add(P.dec[l], base);
        bad |= add(P.pred, base);
    }
    T->n[br] = n;
    return bad;
}

}  // namespace piml

using namespace piml;

extern "C" int64_t piml_pinnsf_packed_floats(const piml_net_desc *desc) {
    if (!desc) return -1;
    FPlan P;
    PackTab PT;
    if (build_plan(desc, &P, &PT)) return -1;
    return P.total;
}

extern "C" int piml_pinnsf_pack_f32(const piml_net_desc *desc, const float *params_torch, float *packed, void *stream) {
    PIML_REQUIRE(desc && params_torch && packed, "piml_pinnsf_pack_f32: null pointer");
    FPlan P;
    PackTab PT;
    int rc = build_plan(desc, &P, &PT);
    if (rc) return rc;
    PIML_REQUIRE(aligned16(packed), "piml_pinnsf_pack_f32: packed must be 16-byte aligned");
    const int threads = 256;
    pinnsf_pack_kernel<<<static_cast<unsigned>((P.total + threads - 1) / threads), threads, 0,
                         static_cast<cudaStream_t>(stream)>>>(PT, params_torch, packed, P.total);
    count_launch();
    return check_launch("pinnsf_pack_kernel");
}

static int pinnsf_forward_impl(const piml_net_desc *desc, const float *params, int has_obs, float tau,
                               const float *ped, const float *obs, const float *self, int64_t R, int kp, int ko,
                               int norm_group, const float *drop_ped, const float *drop_obs, float *acc,
                               float *ped_msgs, float *obs_msgs, float *coll, float *stash, void *stream) {
    PIML_REQUIRE(desc && params, "piml_pinnsf_forward_f32: null pointer");
    PIML_REQUIRE(R >= 0 && kp >= 1 && ko >= 0, "piml_pinnsf_forward_f32: bad dimensions R=%lld kp=%d ko=%d",
                 static_cast<long long>(R), kp, ko);
    PIML_REQUIRE(kp <= FT_TR && ko <= FT_TR, "piml_pinnsf_forward_f32: more than %d slots per agent", FT_TR);
    PIML_REQUIRE(aligned16(params), "piml_pinnsf_forward_f32: params must be 16-byte aligned (piml_pinnsf_pack_f32)");
    if (!has_obs || ko == 0) { has_obs = 0; ko = 0; }
    FPlan P;
    PackTab PT;
    int rc = build_plan(desc, &P, &PT);
    if (rc) return rc;
    if (R == 0) return PIML_OK;        // empty batch: the row buffers may be null (torch's empty tensors are)
    PIML_REQUIRE(ped && self && acc, "piml_pinnsf_forward_f32: null pointer");
    PIML_REQUIRE(!has_obs || obs, "piml_pinnsf_forward_f32: has_obs set but obs is null");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const SPlan S = make_splan(P, has_obs != 0, R, kp, ko, coll != nullptr);

    FTab T;
    T.n[1] = 0;
    PIML_REQUIRE(build_chunks(P, 0, coll != nullptr, &T) == 0 && (!has_obs || build_chunks(P, 1, false, &T) == 0),
                 "piml_pinnsf_forward_f32: network needs more than %d weight chunks per branch", FT_MAXCH);

    float *scratch = nullptr;
    rc = scratch_get(st, R * 4 + (norm_group > 0 ? R * 2 : 0), &scratch);
    if (rc) return rc;
    float *sums = scratch;
    const float *dnorm = nullptr;
    if (norm_group > 0) {
        PIML_REQUIRE(R % norm_group == 0, "piml_pinnsf_forward_f32: R=%lld not a multiple of norm_group=%d",
                     static_cast<long long>(R), norm_group);
        float *dn = scratch + R * 4;
        dest_colnorm_kernel<<<static_cast<unsigned>(R / norm_group), 128, 0, st>>>(self, norm_group, dn);
        count_launch();
        rc = check_launch("dest_colnorm_kernel");
        if (rc) return rc;
        dnorm = dn;
    }

    FArgs a;
    a.params = params; a.ped = ped; a.obs = obs; a.drop_ped = drop_ped; a.drop_obs = drop_obs;
    a.R = R; a.kp = kp; a.ko = ko;
    a.ag_ped = FT_TR / kp; a.ag_obs = ko ? FT_TR / ko : 1;
    a.n_ped_tiles = (R + a.ag_ped - 1) / a.ag_ped;
    a.n_obs_tiles = has_obs ? (R + a.ag_obs - 1) / a.ag_obs : 0;
    a.sums = sums; a.ped_msgs = ped_msgs; a.obs_msgs = has_obs ? obs_msgs : nullptr; a.coll = coll;
    a.stash = stash;
    const size_t smem = sizeof(float) * (2 * FT_MAXW * FT_TRP + 2 * FT_KC * FT_MAXW + FT_SMALL * FT_TRP) + 16;
    // per launch: the attribute is per DEVICE, and a process may touch several (it costs well under a microsecond)
    PIML_CUDA(cudaFuncSetAttribute(pinnsf_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(smem)));
    const int64_t tiles = a.n_ped_tiles + a.n_obs_tiles;
    PIML_REQUIRE(tiles < (1LL << 31), "piml_pinnsf_forward_f32: too many tiles");
    pinnsf_tile_kernel<<<static_cast<unsigned>(tiles), FT_THREADS, smem, st>>>(P, T, a, S);
    count_launch();
    rc = check_launch("pinnsf_tile_kernel");
    if (rc) return rc;
    const int threads = 256;
    pinnsf_finish_kernel<<<static_cast<unsigned>((2 * R + threads - 1) / threads), threads, 0, st>>>(
        sums, self, dnorm, R, has_obs, tau, acc);
    count_launch();
    return check_launch("pinnsf_finish_kernel");
}

extern "C" int piml_pinnsf_forward_f32(const piml_net_desc *desc, const float *params, int has_obs, float tau,
                                       const float *ped, const float *obs, const float *self, int64_t R, int kp,
                                       int ko, int norm_group, const float *drop_ped, const float *drop_obs,
                                       float *acc, float *ped_msgs, float *obs_msgs, float *coll, void *stream) {
    return pinnsf_forward_impl(desc, params, has_obs, tau, ped, obs, self, R, kp, ko, norm_group, drop_ped, drop_obs,
                               acc, ped_msgs, obs_msgs, coll, nullptr, stream);
}

extern "C" int64_t piml_pinnsf_stash_floats(const piml_net_desc *desc, int has_obs, int64_t R, int kp, int ko) {
    if (!desc || R < 0 || kp < 1 || ko < 0) return -1;
    FPlan P;
    PackTab PT;
    if (build_plan(desc, &P, &PT)) return -1;
    if (!has_obs || ko == 0) { has_obs = 0; ko = 0; }
    return make_splan(P, has_obs != 0, R, kp, ko, true).total;
}

extern "C" int piml_pinnsf_forward_train_f32(const piml_net_desc *desc, const float *params, int has_obs, float tau,
                                             const float *ped, const float *obs, const float *self, int64_t R, int kp,
                                             int ko, int norm_group, const float *drop_ped, const float *drop_obs,
                                             float *acc, float *ped_msgs, float *obs_msgs, float *coll, float *stash,
                                             void *stream) {
    PIML_REQUIRE(stash || R == 0, "piml_pinnsf_forward_train_f32: stash is null");
    PIML_REQUIRE(!desc || desc->n_coll == 0 || coll || R == 0, "piml_pinnsf_forward_train_f32: coll output is required");
    return pinnsf_forward_impl(desc, params, has_obs, tau, ped, obs, self, R, kp, ko, norm_group, drop_ped, drop_obs,
                               acc, ped_msgs, obs_msgs, coll, stash, stream);
}
