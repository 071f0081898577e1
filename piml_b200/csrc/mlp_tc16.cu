// mlp_tc16.cu -- interaction-network forward on the tensor cores, 16-bit path: tcgen05.mma kind::f16 with every operand
// split into fp16 hi + lo (x_lo w_hi + x_hi w_lo + x_hi w_hi, fp32 accumulation in TMEM), TWO tiles in flight per SM
// and the branch's weights resident in shared memory.  sm_100a.
//
// Same mathematics as pinnsf_tc_kernel (mlp_tc.cu) / pinnsf_tile_kernel (mlp.cu): reference src/models/model.py:40-119,
// :1104-1135 (pinnsf_bottleneck), :1185-1212 (pinnsf_bm): per slot row enc -> 2x -> dec -> pred, zero-padded slots NOT
// masked.  Why a second tensor-core kernel (profiles/r01d_ncu_pinnsf_tc_kernel.txt: tensor pipe 29 % busy, the MMA
// thread waits 8k of 26k cycles per tile for the epilogue, one tile in flight): with tf32 operands a tile needs
// A_hi | A_lo | D = 384 TMEM columns, so two tiles do not fit the 512 columns of an SM.  fp16 has the same 11-bit
// significand as tf32 but packs two K elements per 32-bit column: a tile is D (128) + A_hi (64) + A_lo (64) = 256 columns,
// two tiles fit, K = 16 per instruction halves the MMA count (171 -> 87 per tile) and the whole branch's weight images
// are 184 KB -- they stay in shared memory instead of streaming through a ring for every tile.
//
// fp16's narrow exponent is handled by exact power-of-two scaling, so the result does not depend on the magnitude of
// weights or activations:  * per layer (pack time): W * 2^e_l with max|W| in [2^13, 2^14);
//                          * per tile row and layer (epilogue): y * 2^s with max|y_row| in [2^14, 2^15);
// both are undone in the next epilogue (y = D * 2^-s * 2^-e_l + b).  The split drops lo*lo = O(2^-22): measured
// 6.8e-7 of fp64 for a 128 x 128 x 128 layer (3xTF32: 1.0e-6).
//
// Per set (SETS, piml_pinnsf_forward_tc_sets_f32): S networks of one description, each with its own rows; CTA
// blockIdx.x serves set blockIdx.x / ctas_per_set and splits its ctas_per_set CTAs between the set's two branches as
// the single-network kernel splits the grid, so every CTA still keeps ONE branch's weights resident.  More sets than
// SMs run as several waves.  A row's result depends only on the row and its set's weights (per-row scaling, in-tile
// slot sums), so set s equals piml_pinnsf_forward_tc_f32 on set s alone, bit for bit.
//
// Per CTA (persistent, one per SM, ONE branch per CTA, 576 threads):
//   warp 0   : loads the branch's weight images (hi + lo per layer, UMMA K-major core matrices written by
//              piml_pinnsf_pack_tc_f32) with cp.async.bulk, one mbarrier per layer, once;
//   warp 1   : MMA issuer -- one thread; alternates between the two tile slots: while slot X's accumulator is in the
//              epilogue, slot Y's layer runs on the tensor pipe;
//   warps 2-9: epilogue of slot 0, warps 10-17: epilogue of slot 1 -- thread = (tile row = TMEM lane, one half of the
//              layer's columns, kept in registers): tcgen05.ld D -> scale, bias, ReLU -> row maximum (exchanged between
//              the two halves through shared memory) -> scale, split into fp16 hi / lo pairs, tcgen05.st as the NEXT
//              layer's A operand; the 2-wide predictor and the slot sums run on the CUDA cores in fp32.
// TMEM columns of slot s: D [256 s, +128), A_hi [256 s + 128, +64), A_lo [256 s + 192, +64).
#include "common.cuh"
#include "tc.cuh"
#include "mlp_tc16.cuh"

namespace piml {

__device__ __forceinline__ void t16_wait(uint64_t *bar, uint32_t parity) {
    if (!mbar_wait_bounded(bar, parity, 1u << 28)) __trap();       // a protocol bug traps instead of hanging the GPU
}
__device__ __forceinline__ void slot_barrier(int slot) {           // the 256 epilogue threads of one tile slot
    asm volatile("bar.sync %0, 256;" ::"r"(1 + slot) : "memory");
}

// 2^s with max * 2^s in [2^14, 2^15) and its inverse (both exact); max == 0 / subnormal -> 1.
__device__ __forceinline__ void row_scale(float mx, float &s, float &inv_s) {
    int E = static_cast<int>((__float_as_uint(mx) >> 23) & 0xffu);
    if (E == 0) { s = 1.f; inv_s = 1.f; return; }
    E = E < 15 ? 15 : (E > 254 ? 254 : E);
    s = __uint_as_float(static_cast<uint32_t>(268 - E) << 23);
    inv_s = __uint_as_float(static_cast<uint32_t>(E - 14) << 23);
}

template <bool COMPACT, bool SETS>
__global__ void __launch_bounds__(T16_THREADS, 1) pinnsf_tc16_kernel(const __grid_constant__ Tc16Plan P,
                                                                     const __grid_constant__ Tc16Args a) {
    extern __shared__ __align__(128) unsigned char t16_smem[];
    unsigned char *wimg = t16_smem;                                               // the branch's weight images
    float *biasb = reinterpret_cast<float *>(wimg + P.w_bytes);                   // [bias_floats]
    float *small = biasb + P.bias_floats;       // [2 slots][1024]: row maxima [2 parities][2 halves][128] | predictor scratch [512]
    uint64_t *bars = reinterpret_cast<uint64_t *>(small + 2048);
    uint64_t *w_ready = bars, *a_ready = bars + T16_MAXL, *d_ready = a_ready + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(d_ready + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (warp == 0) tc::tmem_alloc(tmem_slot, 512);
    if (tid == 32) {
        for (int l = 0; l < P.nl; ++l) mbar_init(&w_ready[l], 1);
        for (int s = 0; s < 2; ++s) { mbar_init(&a_ready[s], 256); mbar_init(&d_ready[s], 1); }
        mbar_fence_init();
    }
    // tiles of both branches (compact mode: the listed non-zero rows + ONE zero row per branch), CTAs split in proportion
    // 32-bit bookkeeping throughout (row counts are < 2^31 by the callers' checks): the epilogue lives at a 96-register ceiling
    const int cnt_ped = COMPACT ? a.counts[0] + 1 : 0, cnt_obs = (COMPACT && a.has_obs) ? a.counts[1] + 1 : 0;
    const int nP = COMPACT ? (cnt_ped + 127) / 128 : static_cast<int>(a.n_ped_tiles);
    const int nO = COMPACT ? (cnt_obs + 127) / 128 : static_cast<int>(a.n_obs_tiles);
    // SETS: this CTA's set and its place among the set's CTAs (a.R, tile counts and the split are per set)
    const int G = SETS ? a.ctas_per_set : static_cast<int>(gridDim.x);
    const int set = SETS ? static_cast<int>(blockIdx.x) / a.ctas_per_set : 0;
    const int cta = SETS ? static_cast<int>(blockIdx.x) - set * a.ctas_per_set : static_cast<int>(blockIdx.x);
    // CTAs per branch (one branch per CTA: its weights stay resident).  The kernel ends with its slowest CTA, so the
    // split minimises the larger per-CTA tile count: start from the proportional share and give the obstacle branch
    // CTAs until it is no longer the straggler (rounding to nearest left 43 obstacle tiles on ONE CTA next to 32 per
    // pedestrian CTA at N = 100k: the kernel took 539k cycles where the pedestrian CTAs needed 390k).
    int gO = 0;
    if (nO > 0) {
        if (nP == 0) gO = G;
        else {
            gO = static_cast<int>((static_cast<int64_t>(G) * nO) / (nP + nO));
            gO = gO < 1 ? 1 : (gO > G - 1 ? G - 1 : gO);
            while (gO < G - 1 && (nO + gO - 1) / gO > (nP + (G - gO) - 1) / (G - gO)) ++gO;
        }
    }
    const int gP = G - gO;
    const int br = cta < gP ? 0 : 1;
    const int first = br == 0 ? cta : cta - gP;
    const int stride = br == 0 ? gP : gO;
    const int ntiles_br = br == 0 ? nP : nO;
    const int my_tiles = first < ntiles_br ? (ntiles_br - first + stride - 1) / stride : 0;

    const float *branch = a.params + (SETS ? set * a.set_stride : 0) + P.base + static_cast<int64_t>(br) * P.branch_floats;
    for (int e = tid; e < P.bias_floats; e += T16_THREADS) biasb[e] = branch[P.w_bytes / 4 + e];
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tbase = *tmem_slot;

    if (warp == 0) {
        // ===== weight loader: the whole branch, once =====
        if (lane == 0 && my_tiles > 0) {
            const unsigned char *src = reinterpret_cast<const unsigned char *>(branch);
            for (int l = 0; l < P.nl; ++l) {
                const uint32_t bytes = static_cast<uint32_t>(P.L[l].bytes);
                mbar_expect_tx(&w_ready[l], bytes);
                for (uint32_t o = 0; o < bytes; o += 16384u)
                    tma_bulk_g2s(wimg + P.L[l].w_off + o, src + P.L[l].w_off + o, min(16384u, bytes - o), &w_ready[l]);
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: round robin over the two slots =====
        // The WHOLE warp runs this loop on warp-uniform values (broadcast through shfl so that ptxas knows it) and one
        // elected lane issues: descriptors then live in uniform registers and an MMA costs one instruction, not a
        // 10-instruction R2UR waterfall (see tc::elect_one).
        const uint32_t tb = __shfl_sync(0xffffffffu, tbase, 0);
        const int mt = __shfl_sync(0xffffffffu, static_cast<int>(my_tiles), 0);
        const uint32_t wbase = __shfl_sync(0xffffffffu, tc::smem_addr(wimg), 0);
        int done[2] = {0, 0};                                      // tiles finished per slot
        int layer[2] = {0, 0};
        uint32_t aph = 0, wseen = 0;
        const int n_slot[2] = {(mt + 1) / 2, mt / 2};
        for (;;) {
            bool any = false;
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                if (done[s] >= n_slot[s]) continue;
                any = true;
                const int li = layer[s];
                const Tc16Layer &Ly = P.L[li];
                t16_wait(&a_ready[s], (aph >> s) & 1u);            // A of (this slot's tile, layer li) is in TMEM
                aph ^= (1u << s);
                if (!((wseen >> li) & 1u)) { t16_wait(&w_ready[li], 0); wseen |= (1u << li); }
                tc::fence_after_sync();
                const uint32_t dcol = tb + s * T16_SLOT_COLS + T16_COL_D;
                uint32_t ah = tb + s * T16_SLOT_COLS + T16_COL_AH, al = tb + s * T16_SLOT_COLS + T16_COL_AL;
                const uint32_t idesc = tc::idesc_f16(Ly.N);
                const uint32_t lbo = Ly.N * 16, sbo = 128;
                const uint32_t hi_addr = wbase + Ly.w_off;
                uint64_t bh = tc::smem_desc(hi_addr, lbo, sbo);
                uint64_t bl = tc::smem_desc(hi_addr + Ly.Kp * Ly.N * 2, lbo, sbo);
                const uint64_t dstep = (2 * lbo) >> 4;             // start-address field per K = 16 step
                const int nks = Ly.Kp / 16;
                if (tc::elect_one()) {
                    bool acc = false;
#pragma unroll 2
                    for (int ks = 0; ks < nks; ++ks, bh += dstep, bl += dstep, ah += 8, al += 8) {
                        tc::mma_f16_ts(dcol, al, bh, idesc, acc);        // x_lo w_hi
                        tc::mma_f16_ts(dcol, ah, bl, idesc, true);       // x_hi w_lo
                        tc::mma_f16_ts(dcol, ah, bh, idesc, true);       // x_hi w_hi
                        acc = true;
                    }
                    tc::commit(&d_ready[s]);                       // accumulator of this (slot, layer) complete
                }
                __syncwarp();
                if (++layer[s] == P.nl) { layer[s] = 0; ++done[s]; }
            }
            if (!any) break;
        }
    } else {
        // ===== epilogue warps: 8 per slot; thread = (tile row, column half) =====
        const int slot = (warp - 2) >> 3;
        const int q4 = warp & 3;                                   // TMEM lane quarter this warp may access
        const int half = ((warp - 2) & 7) >> 2;                    // which half of a layer's columns
        const int m = q4 * 32 + lane;                              // tile row == TMEM lane
        const uint32_t tl = tbase + (static_cast<uint32_t>(q4 * 32) << 16) + slot * T16_SLOT_COLS;
        const int k = br == 0 ? a.kp : a.ko;
        const int AG = br == 0 ? a.ag_ped : a.ag_obs;
        const int cnt = br == 0 ? cnt_ped : cnt_obs;
        const int *list = br == 0 ? a.list_ped : a.list_obs;
        const float *feat = (br == 0 ? a.ped : a.obs) + (SETS ? static_cast<int64_t>(set) * a.R * k * 6 : 0);
        float *smax = small + slot * 1024;                         // [2 parities][2 halves][128] row maxima
        float *sm2 = smax + 512;                                   // [2 halves][128][2] predictor partials / slot sums
        uint32_t dph = 0;
        struct RowFeat { int crow; float f[6]; bool live; };
        auto load_row = [&](int j) {                           // j: index into this CTA's tile sequence
            RowFeat rf;
            rf.crow = -1; rf.live = false;
#pragma unroll
            for (int q = 0; q < 6; ++q) rf.f[q] = 0.f;
            if (j >= my_tiles) return rf;
            const int tloc = first + j * stride;
            int64_t src;
            if (COMPACT) {
                const int nrows = min(128, cnt - tloc * 128);
                if (m < nrows && tloc * 128 + m < cnt - 1)                // no list (fused NN step): rows are stored compactly
                    rf.crow = list ? list[tloc * 128 + m] : static_cast<int>(tloc * 128 + m);
                rf.live = rf.crow >= 0;
                src = rf.crow;
            } else {
                const int64_t agent0 = static_cast<int64_t>(tloc) * AG;
                const int na = static_cast<int>(min(static_cast<int64_t>(AG), a.R - agent0));
                rf.live = m < na * k;
                src = agent0 * k + m;
            }
            if (rf.live) {
                const float2 *f2 = reinterpret_cast<const float2 *>(feat + src * 6);
                const float2 x0 = f2[0], x1 = f2[1], x2 = f2[2];
                rf.f[0] = x0.x; rf.f[1] = x0.y; rf.f[2] = x1.x; rf.f[3] = x1.y; rf.f[4] = x2.x; rf.f[5] = x2.y;
            }
            return rf;
        };
        // the 6-d features of a row as the first A operand of its tile: K padded to 16 with zeros, row-scaled
        auto write_features = [&](const RowFeat &rf, float &inv_s_out) {
            float mx = 0.f;
#pragma unroll
            for (int q = 0; q < 6; ++q) mx = fmaxf(mx, fabsf(rf.f[q]));
            float s;
            row_scale(mx, s, inv_s_out);
            if (half == 0) {
                uint32_t hi[8], lo[8];
#pragma unroll
                for (int q = 0; q < 3; ++q) tc::split_f16x2(rf.f[2 * q] * s, rf.f[2 * q + 1] * s, hi[q], lo[q]);
#pragma unroll
                for (int q = 3; q < 8; ++q) { hi[q] = 0u; lo[q] = 0u; }
                tc::st8(tl + T16_COL_AH, hi);
                tc::st8(tl + T16_COL_AL, lo);
                tc::wait_st();
                tc::fence_before_sync();
            }
            tc::mbar_arrive(&a_ready[slot]);
        };
        // Software pipeline across tiles: the operand of tile j + 2 (this slot's next tile) is written as soon as the
        // LAST accumulator of tile j has been read out, so its first layer runs on the tensor pipe while tile j's
        // predictor, exchange and stores are still in progress.  (Its rows are loaded right there: holding them in
        // registers across the tile cost 8 of the 96 registers the epilogue has, i.e. spills.)
        float inv_s = 1.f;
        int crow = -1;
        {
            const RowFeat first_rows = load_row(slot);
            crow = first_rows.crow;
            if (slot < my_tiles) write_features(first_rows, inv_s);
        }
        for (int j = slot; j < my_tiles; j += 2) {
            const int tloc = first + j * stride;
            const int64_t agent0 = static_cast<int64_t>(tloc) * AG;
            const int na = COMPACT ? 0 : static_cast<int>(min(static_cast<int64_t>(AG), a.R - agent0));
            const int nrows = COMPACT ? min(128, cnt - tloc * 128) : na * k;
            const int64_t row0 = agent0 * k;
            float inv_s_next = 1.f;
            int crow_next = -1;
            float m0 = 0.f, m1 = 0.f;
            for (int li = 0; li < P.nl; ++li) {
                const Tc16Layer &Ly = P.L[li];
                const bool last = li == P.nl - 1;
                const int hc = Ly.N >> 1;                          // columns of this thread: [half * hc, +hc), 16 at a time
                const int nchunk = hc >> 4;
                t16_wait(&d_ready[slot], dph);
                dph ^= 1u;
                tc::fence_after_sync();
                const float *bias = biasb + Ly.bias_off + half * hc;
                const float sc = inv_s * biasb[P.winv_off + li];   // undo the input's row scale and the layer's weight scale
                // all of this thread's columns in one go: the loads overlap, one wait
                uint32_t r[64];
                {
                    uint32_t (&r0)[32] = *reinterpret_cast<uint32_t (*)[32]>(&r[0]);
                    uint32_t (&r1)[32] = *reinterpret_cast<uint32_t (*)[32]>(&r[32]);
                    uint32_t (&h0)[16] = *reinterpret_cast<uint32_t (*)[16]>(&r[0]);
                    if (nchunk == 4) { tc::ld32(tl + T16_COL_D + half * hc, r0); tc::ld32(tl + T16_COL_D + half * hc + 32, r1); }
                    else if (nchunk == 2) tc::ld32(tl + T16_COL_D + half * hc, r0);
                    else tc::ld16(tl + T16_COL_D + half * hc, h0);
                    tc::wait_ld();
                }
                if (last) {                                        // D and A of this slot are free: next tile's operand
                    const RowFeat nxt = load_row(j + 2);           // (loaded here: 8 registers less across the tile)
                    crow_next = nxt.crow;
                    if (j + 2 < my_tiles) write_features(nxt, inv_s_next);
                }
                float *v = reinterpret_cast<float *>(r);
                float mx = 0.f, mxb4[4] = {0.f, 0.f, 0.f, 0.f};   // four independent maximum chains (ILP), merged below
                const float2 sc2 = make_float2(sc, sc);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (c < nchunk) {
#pragma unroll
                        for (int q4b = 0; q4b < 4; ++q4b) {        // packed FP32 (FFMA2): two columns per instruction
                            const float4 b4 = *reinterpret_cast<const float4 *>(bias + c * 16 + q4b * 4);
                            const int e = c * 16 + q4b * 4;
                            float2 y01 = __ffma2_rn(make_float2(v[e], v[e + 1]), sc2, make_float2(b4.x, b4.y));
                            float2 y23 = __ffma2_rn(make_float2(v[e + 2], v[e + 3]), sc2, make_float2(b4.z, b4.w));
                            if (Ly.relu) {
                                y01.x = fmaxf(y01.x, 0.f); y01.y = fmaxf(y01.y, 0.f);
                                y23.x = fmaxf(y23.x, 0.f); y23.y = fmaxf(y23.y, 0.f);
                            }
                            v[e] = y01.x; v[e + 1] = y01.y; v[e + 2] = y23.x; v[e + 3] = y23.y;
                            mxb4[q4b] = fmaxf(fmaxf(mxb4[q4b], fmaxf(fabsf(y01.x), fabsf(y01.y))), fmaxf(fabsf(y23.x), fabsf(y23.y)));
                        }
                    }
                }
                mx = fmaxf(fmaxf(mxb4[0], mxb4[1]), fmaxf(mxb4[2], mxb4[3]));
                if (last) {                                        // predictor Linear(dw, 2) on the CUDA cores
                    const float *w0 = biasb + P.predw_off + half * hc, *w1 = w0 + P.dw;
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        if (c < nchunk) {
#pragma unroll
                            for (int q = 0; q < 16; ++q) {
                                m0 = fmaf(v[c * 16 + q], w0[c * 16 + q], m0);
                                m1 = fmaf(v[c * 16 + q], w1[c * 16 + q], m1);
                            }
                        }
                    break;
                }
                float *mxb = smax + (li & 1) * 256;                // double buffered: one barrier per layer is enough
                mxb[half * 128 + m] = mx;                          // row maximum over both column halves
                slot_barrier(slot);
                mx = fmaxf(mx, mxb[(half ^ 1) * 128 + m]);
                float s;
                row_scale(mx, s, inv_s);
                // Split relative to the ROW: after scaling, |x| < 2^15; hi = x rounded to a multiple of 16 (the fp16
                // spacing of [2^14, 2^15): exact in fp16, obtained with the add-magic-subtract trick on the packed FP32
                // pipe), lo = x - hi in [-8, 8] rounded to fp16: |x - hi - lo| <= 2^-9 = 2^-23 of the row maximum.
                const float2 s2 = make_float2(s, s), M2 = make_float2(201326592.f, 201326592.f), nM2 = make_float2(-201326592.f, -201326592.f);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (c < nchunk) {                              // scale, split, store as the next layer's A operand
                        uint32_t hi[8], lo[8];
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float2 x = __fmul2_rn(make_float2(v[c * 16 + 2 * q], v[c * 16 + 2 * q + 1]), s2);
                            const float2 h = __fadd2_rn(__fadd2_rn(x, M2), nM2);
                            const float2 l = __fadd2_rn(x, make_float2(-h.x, -h.y));
                            asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hi[q]) : "f"(h.y), "f"(h.x));
                            asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(lo[q]) : "f"(l.y), "f"(l.x));
                        }
                        tc::st8(tl + T16_COL_AH + ((half * hc + c * 16) >> 1), hi);
                        tc::st8(tl + T16_COL_AL + ((half * hc + c * 16) >> 1), lo);
                    }
                }
                tc::wait_st();
                tc::fence_before_sync();
                tc::mbar_arrive(&a_ready[slot]);                   // the next layer of this slot may start
            }
            // combine the two column halves of the predictor: half 1 hands its partial sums over and moves on
            // (bar.arrive), only half 0 waits (the next write of sm2 is several slot barriers away)
            if (half == 1) {
                sm2[m * 2] = m0; sm2[m * 2 + 1] = m1;
                asm volatile("bar.arrive %0, 256;" ::"r"(3 + slot) : "memory");
            } else {
                asm volatile("bar.sync %0, 256;" ::"r"(3 + slot) : "memory");
                m0 = m0 + sm2[m * 2] + biasb[P.predb_off];
                m1 = m1 + sm2[m * 2 + 1] + biasb[P.predb_off + 1];
            }
            if (COMPACT) {
                if (half == 0 && m < nrows) {                      // slot sums are formed by the finish kernel
                    float *dst = crow >= 0 ? (br == 0 ? a.cmsg_ped : a.cmsg_obs) + static_cast<int64_t>(crow) * 2 : a.f0 + br * 2;
                    dst[0] = m0; dst[1] = m1;
                }
            } else {
                float *msgs_out = SETS ? nullptr : (br == 0 ? a.ped_msgs : a.obs_msgs);   // SETS: no messages
                if (half == 0 && msgs_out && m < nrows) { msgs_out[(row0 + m) * 2] = m0; msgs_out[(row0 + m) * 2 + 1] = m1; }
                slot_barrier(slot);                                // every partial read before the totals overwrite
                if (half == 0) { sm2[m * 2] = m0; sm2[m * 2 + 1] = m1; }
                slot_barrier(slot);
                if (half == 0)
                    for (int e = m; e < 2 * na; e += 128) {        // torch.sum(dim=-2) over the k slots (model.py:1194);
                        const int ag = e >> 1, c = e & 1;          // k = 1: 128 agents per tile, two sums per thread
                        float sum = 0.f;
                        for (int jj = 0; jj < k; ++jj) sum += sm2[(ag * k + jj) * 2 + c];
                        a.sums[((SETS ? static_cast<int64_t>(set) * a.R : 0) + agent0 + ag) * 4 + br * 2 + c] = sum;
                    }
                slot_barrier(slot);                                // sm2 is free for this slot's next tile
            }
            inv_s = inv_s_next; crow = crow_next;
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tbase, 512);
}

// ---- plan ------------------------------------------------------------------------------------------------------------
// weight images | bias block | row maxima and predictor scratch (2 slots x 1024 floats) | mbarriers | TMEM address
size_t tc16_smem_bytes(const Tc16Plan &P) {
    return static_cast<size_t>(P.w_bytes) + sizeof(float) * (P.bias_floats + 2048) + 8 * (T16_MAXL + 4) + 16;
}

// Layers as the tf32 plan lists them (K, N, relu, ResDNN 2x fold): enc..., dec...; K padded to 16.
int tc16_build_plan(const piml_net_desc *d, int64_t base_floats, Tc16Plan *P) {
    if (d->kind != 0 || d->proc_mode != 0 || d->enc_dims[0] != 6) return 1;       // per-slot-decoder networks only
    if (d->n_enc < 1 || d->n_dec < 1 || d->n_enc + d->n_dec > T16_MAXL) return 1;
    P->nl = d->n_enc + d->n_dec;
    P->dw = d->dec_dims[d->n_dec];
    int woff = 0, boff = 0, li = 0;
    auto layer = [&](int K, int N, int relu) -> int {
        if ((N != 32 && N != 64 && N != 128) || K > 128 || (K % 16 != 0 && li != 0)) return 1;
        Tc16Layer &L = P->L[li++];
        L.K = K; L.Kp = (K + 15) & ~15; L.N = N; L.relu = relu; L.bias_off = boff; L.w_off = woff;
        L.bytes = 2 * L.Kp * N * 2;
        woff += L.bytes;
        boff += N;
        return 0;
    };
    for (int l = 0; l < d->n_enc; ++l)
        if (layer(d->enc_dims[l], d->enc_dims[l + 1], l == d->n_enc - 1 ? 0 : 1)) return 1;
    for (int l = 0; l < d->n_dec; ++l)
        if (layer(d->dec_dims[l], d->dec_dims[l + 1], l < d->n_dec - 1 ? 1 : 0)) return 1;
    P->w_bytes = woff;                                             // every layer image is a multiple of 1 KB
    P->predw_off = boff; boff += 2 * P->dw;
    P->predb_off = boff; boff += 2;
    P->winv_off = boff; boff += P->nl;
    P->bias_floats = (boff + 3) & ~3;
    P->branch_floats = P->w_bytes / 4 + P->bias_floats;
    P->base = (base_floats + 31) & ~static_cast<int64_t>(31);      // 128-byte aligned behind the tf32 image
    // the branch must stay resident in shared memory.  220 KB - 128 B: the kernel's shared memory used to include 128 B
    // of cycle counters; the limit moved down with them, so that every network keeps the kernel it ran on
    if (tc16_smem_bytes(*P) > 220 * 1024 - 128) return 1;
    return 0;
}

// ---- packing -----------------------------------------------------------------------------------------------------------
// one CTA per (branch, layer): exponent of max |W * fold|, stored as the inverse weight scale 2^-e in the bias block
__global__ void tc16_wmax_kernel(const __grid_constant__ Tc16Plan P, const __grid_constant__ Tc16Src S,
                                 const float *__restrict__ src, float *__restrict__ dst) {
    __shared__ float red[256];
    const int br = blockIdx.x / P.nl, l = blockIdx.x % P.nl;
    const Tc16Layer &L = P.L[l];
    const float *w = src + S.src_w[br * P.nl + l];
    float mx = 0.f;
    for (int e = threadIdx.x; e < L.K * L.N; e += blockDim.x) mx = fmaxf(mx, fabsf(w[e] * S.scale[l]));
    red[threadIdx.x] = mx;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if (threadIdx.x < off) red[threadIdx.x] = fmaxf(red[threadIdx.x], red[threadIdx.x + off]);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        int E = static_cast<int>((__float_as_uint(red[0]) >> 23) & 0xffu);
        float winv = 1.f;
        if (E != 0 && E != 255) {                                  // max * 2^e in [2^13, 2^14): e = 13 - (E - 127)
            E = E < 20 ? 20 : (E > 240 ? 240 : E);
            winv = __uint_as_float(static_cast<uint32_t>(E - 13) << 23);      // 2^-(e) = 2^(E - 127 - 13)
        }
        dst[P.base + static_cast<int64_t>(br) * P.branch_floats + P.w_bytes / 4 + P.winv_off + l] = winv;
    }
}

// one thread per 16-bit element of the weight images / per float of the bias block
__global__ void pinnsf_pack_tc16_kernel(const __grid_constant__ Tc16Plan P, const __grid_constant__ Tc16Src S,
                                        const float *__restrict__ src, float *__restrict__ dst) {
    const int64_t halfs = P.w_bytes / 2;
    const int64_t per_branch = halfs + P.bias_floats;
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= 2 * per_branch) return;
    const int br = static_cast<int>(i / per_branch);
    const int64_t off = i - br * per_branch;
    float *bdst = dst + P.base + static_cast<int64_t>(br) * P.branch_floats;
    float *bias_dst = bdst + P.w_bytes / 4;
    if (off < halfs) {
        int l = 0;
        while (l + 1 < P.nl && off * 2 >= P.L[l + 1].w_off) ++l;
        const Tc16Layer &L = P.L[l];
        const int64_t e = off - L.w_off / 2;
        const int half = static_cast<int>(e / (L.Kp * L.N));
        const int r = static_cast<int>(e - static_cast<int64_t>(half) * L.Kp * L.N);
        const int cell = r / (L.N * 8), n = (r / 8) % L.N, kk = r & 7;
        const int kx = cell * 8 + kk;
        const float wscale = 1.0f / bias_dst[P.winv_off + l];      // written by tc16_wmax_kernel (stream order)
        const float w = kx < L.K ? src[S.src_w[br * P.nl + l] + static_cast<int64_t>(n) * L.K + kx] * S.scale[l] * wscale : 0.f;
        uint16_t hi, lo;
        tc::split_f16(w, hi, lo);
        reinterpret_cast<uint16_t *>(bdst)[off] = half == 0 ? hi : lo;
    } else {
        const int b = static_cast<int>(off - halfs);
        if (b >= P.winv_off) {                                     // winv: written by tc16_wmax_kernel; padding: zero
            if (b >= P.winv_off + P.nl) bias_dst[b] = 0.f;
            return;
        }
        float v;
        if (b >= P.predb_off) v = src[S.pred_src[br] + 2LL * P.dw + (b - P.predb_off)];
        else if (b >= P.predw_off) v = src[S.pred_src[br] + (b - P.predw_off)];
        else {
            int l = 0;
            while (l + 1 < P.nl && b >= P.L[l + 1].bias_off) ++l;
            v = src[S.src_b[br * P.nl + l] + (b - P.L[l].bias_off)] * S.scale[l];
        }
        bias_dst[b] = v;
    }
}

int tc16_pack(const Tc16Plan &P, const Tc16Src &S, const float *params_torch, float *packed, cudaStream_t st) {
    tc16_wmax_kernel<<<2 * P.nl, 256, 0, st>>>(P, S, params_torch, packed);
    count_launch();
    int rc = check_launch("tc16_wmax_kernel");
    if (rc) return rc;
    const int64_t n = 2 * (static_cast<int64_t>(P.w_bytes) / 2 + P.bias_floats);
    pinnsf_pack_tc16_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(P, S, params_torch, packed);
    count_launch();
    return check_launch("pinnsf_pack_tc16_kernel");
}

int tc16_launch(const Tc16Plan &P, const Tc16Args &a, int64_t tiles_bound, cudaStream_t st) {
    const size_t smem = tc16_smem_bytes(P);
    const int grid = static_cast<int>(tiles_bound < sm_count() ? tiles_bound : sm_count());
    // (compact and dense are separate instantiations: at the epilogue's 96-register ceiling every dead path costs spills)
    const auto kernel = a.compact ? pinnsf_tc16_kernel<true, false> : pinnsf_tc16_kernel<false, false>;
    PIML_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    kernel<<<grid, T16_THREADS, smem, st>>>(P, a);
    count_launch();
    return check_launch("pinnsf_tc16_kernel");
}

// S sets of a.R rows each, dense mode: a.ctas_per_set CTAs per set (at least one per branch with tiles, at most one
// per tile), as many as fill the SMs; more sets than SMs make several waves of a.ctas_per_set CTAs per set.
int tc16_launch_sets(const Tc16Plan &P, Tc16Args a, int S, cudaStream_t st) {
    const int64_t tiles = a.n_ped_tiles + a.n_obs_tiles;
    const int64_t fill = sm_count() / S, least = a.n_obs_tiles > 0 ? 2 : 1;
    a.ctas_per_set = static_cast<int>(fill < least ? least : (fill > tiles ? tiles : fill));
    const size_t smem = tc16_smem_bytes(P);
    PIML_CUDA(cudaFuncSetAttribute(pinnsf_tc16_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(smem)));
    pinnsf_tc16_kernel<false, true><<<static_cast<unsigned>(static_cast<int64_t>(S) * a.ctas_per_set), T16_THREADS,
                                      smem, st>>>(P, a);
    count_launch();
    return check_launch("pinnsf_tc16_kernel");
}

}  // namespace piml
