// mlapm.cu -- all-pairs MLAPM force for sm_100a.
//
// The whole-crowd production path (mlapm_sym_list_kernel) evaluates every unordered pair once and skips the pairs
// farther apart than the radius where the fp32 weight is exactly 0 (a spatial sort, boxes per block and a work list
// built on the device); the dense kernels below evaluate every pair (row ranges, small crowds, validation).
//
// Replaces MLAPM.step (reference src/models/mlapm.py:10-58) and the loop body of src/main_mlapm.py:19-34.
// The reference materialises (N,N,2)x4 + (N,N,2,2) + (N,N)x6 temporaries (~100 B per ordered pair); here each thread
// keeps R rows in registers and streams the columns through shared memory (TMA bulk copies of position / velocity
// tiles, double buffered), so DRAM traffic is O(N) and the kernel is bound by the FP32 and MUFU pipes.
//
// Grid: (row blocks of 128*R rows) x (column splits).  Each CTA writes its partial row sums to workspace[split][row];
// a finalize kernel adds the splits in a fixed order (deterministic), applies the destination term and the Euler
// update.  The field-of-view gate `v_n . (p_m - p_n) > 0` uses the reference's exact fp32 form
// fmaf(v1, r1, v0*r0) (einsum -> bmm, SURVEY.md A.1); the force magnitude only has to hold 1e-5 relative, which
// both math variants below do:
//   EXACT: IEEE div / sqrt / expf in the reference's operation order (validation variant)
//   fast : rsqrt.approx + ex2.approx, shared 1/r, constant-angle rotation folded into two FMAs (production)
#include <math_constants.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "common.cuh"

namespace piml {

constexpr int ML_THREADS = 128;
constexpr int ML_TILE = 512;          // columns per shared-memory stage: 4 KB positions + 4 KB velocities

struct MlConst {
    int version;
    float A, B, C, D;                  // reference constants
    float Bl, Cl, Dl;                  // pre-multiplied by log2(e) for ex2
    float cos_t, sin_t;                // cos/sin of theta (fp32 angle as the reference builds it)
    float inv_tau, tau;
};

// The kernels' constants from the reference's six (host: mlapm_consts; device: one set per scene of
// mlapm_scenes_kernel).  One derivation, so a scene's constants do not depend on where they were formed.
__host__ __device__ __forceinline__ MlConst mlapm_derive(int version, float tau, float A, float B, float C, float D,
                                                         float theta_deg) {
    MlConst k;
    k.version = version;
    k.A = A; k.B = B; k.C = C; k.D = D;
    const double log2e = 1.4426950408889634;
    k.Bl = static_cast<float>(B * log2e); k.Cl = static_cast<float>(C * log2e);
    k.Dl = static_cast<float>(D * log2e);
    // theta tensor as the reference builds it in fp32: ((+-1 * theta) / 180) * pi   (mlapm.py:33)
    const float th = (theta_deg / 180.0f) * 3.14159274101257324f;
    k.cos_t = static_cast<float>(cos(static_cast<double>(th)));
    k.sin_t = static_cast<float>(sin(static_cast<double>(th)));
    k.tau = tau; k.inv_tau = 1.0f / tau;
    return k;
}

// The rest of the loop body main_mlapm.py:19-34 for one agent, shared by every kernel that finishes a step.  Split so
// that a kernel forms the destination term before it gathers the pair sum (sx, sy), and the new position and the
// arrival test only where they are stored (the finalize kernels keep their register counts):
//   fd = (desired_speed * ed - v) / tau                                (mlapm.py:21-22)
//   force = fd - (sx, sy) (mlapm.py:29/39);  action = v + force*dt     (mlapm.py:57)
//   p' = p + action*dt;  arrived = |p' - dest| < radius                (main_mlapm.py:26,34)
// ed = F.normalize(destination - position)                             (mlapm.py:21)
__device__ __forceinline__ float2 mlapm_dest_dir(float2 p, float2 d) {
    const float dx = __fsub_rn(d.x, p.x), dy = __fsub_rn(d.y, p.y);
    const float dn = fmaxf(norm2_rn(dx, dy), 1e-12f);
    return make_float2(__fdiv_rn(dx, dn), __fdiv_rn(dy, dn));
}
__device__ __forceinline__ float2 mlapm_dest_term(float2 p, float2 v, float2 d, float dsx, float dsy, float tau) {
    const float2 e = mlapm_dest_dir(p, d);
    return make_float2(__fdiv_rn(__fsub_rn(__fmul_rn(dsx, e.x), v.x), tau),
                       __fdiv_rn(__fsub_rn(__fmul_rn(dsy, e.y), v.y), tau));
}
__device__ __forceinline__ float2 mlapm_action(float2 v, float2 fd, float sx, float sy, float dt) {
    const float fx = __fsub_rn(fd.x, sx), fy = __fsub_rn(fd.y, sy);
    return make_float2(__fadd_rn(v.x, __fmul_rn(fx, dt)), __fadd_rn(v.y, __fmul_rn(fy, dt)));
}
__device__ __forceinline__ float2 mlapm_move(float2 p, float2 a, float dt) {
    return make_float2(__fadd_rn(p.x, __fmul_rn(a.x, dt)), __fadd_rn(p.y, __fmul_rn(a.y, dt)));
}
__device__ __forceinline__ bool mlapm_arrived(float2 q, float2 d, float radius) {
    return norm2_rn(__fsub_rn(q.x, d.x), __fsub_rn(q.y, d.y)) < radius;
}

__device__ __forceinline__ float ex2_approx(float x) {            // one MUFU.EX2
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rsqrt_approx(float x) {          // one MUFU.RSQ
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Stage one tile of positions and velocities (n float2 each) on ONE mbarrier phase.  All threads call it.
__device__ __forceinline__ bool stage_tile_pv(float2 *dp, float2 *dv, const float2 *gp, const float2 *gv, int n,
                                              uint64_t *bar) {
    const bool tma = ((reinterpret_cast<uintptr_t>(gp) | reinterpret_cast<uintptr_t>(gv)) & 15u) == 0 && n >= 2;
    if (tma) {
        if (threadIdx.x == 0) {
            const uint32_t bytes = static_cast<uint32_t>(n & ~1) * 8u;
            mbar_expect_tx(bar, 2u * bytes);
            tma_bulk_g2s(dp, gp, bytes, bar);
            tma_bulk_g2s(dv, gv, bytes, bar);
            if (n & 1) { dp[n - 1] = gp[n - 1]; dv[n - 1] = gv[n - 1]; }
        }
    } else {
        for (int i = threadIdx.x; i < n; i += blockDim.x) { dp[i] = gp[i]; dv[i] = gv[i]; }
    }
    return tma;
}

// One ordered pair, production math.  ~37 issue slots for version GC.
template <int VERSION>
__device__ __forceinline__ void pair_fast(float px, float py, float vx, float vy, float ex, float ey, float2 pm,
                                          float2 vm, const MlConst &k, float &fx, float &fy) {
    const float rx = __fsub_rn(pm.x, px);
    const float ry = __fsub_rn(pm.y, py);
    const float gate = (__fmaf_rn(vy, ry, __fmul_rn(vx, rx)) > 0.f) ? k.A : 0.f;     // exact FoV gate (mlapm.py:27)
    const float r2 = fmaf(ry, ry, rx * rx);
    const float inv_r = rsqrt_approx(fmaxf(r2, 1e-30f));
    const float r = r2 * inv_r;
    if (VERSION == 0) {
        const float w = gate * ex2_approx(k.Bl * r) * inv_r;          // view*A*exp(B r) * vr/|vr|   (mlapm.py:29)
        fx = fmaf(w, rx, fx);
        fy = fmaf(w, ry, fy);
    } else {
        const float ux = vm.x - vx, uy = vm.y - vy;
        const float u2 = fmaf(uy, uy, ux * ux);
        const float dot = fmaf(ry, uy, rx * ux);
        const float cosv = dot * inv_r * rsqrt_approx(fmaxf(u2, 1e-30f));   // cosine_similarity(vr, vv)  (mlapm.py:32)
        const float cross = fmaf(rx, ey, -(ry * ex));                 // sign picks +-theta           (mlapm.py:33-34)
        const float s = (cross > 0.f) ? -k.sin_t : k.sin_t;
        const float dx = fmaf(k.cos_t, rx, -(s * ry));                // R(theta) * vr                (mlapm.py:35-38)
        const float dy = fmaf(s, rx, k.cos_t * ry);
        const float arg = fmaf(fmaf(k.Dl, r, k.Cl), cosv, k.Bl * r);  // (B r + C cos + D r cos) * log2 e
        const float w = gate * ex2_approx(arg) * inv_r;
        fx = fmaf(w, dx, fx);
        fy = fmaf(w, dy, fy);
    }
}

// One ordered pair in the reference's own operation order with IEEE arithmetic (validation variant).
template <int VERSION>
__device__ __forceinline__ void pair_exact(float px, float py, float vx, float vy, float ex, float ey, float2 pm,
                                           float2 vm, const MlConst &k, float &fx, float &fy) {
    const float rx = __fsub_rn(pm.x, px);
    const float ry = __fsub_rn(pm.y, py);
    const float r = norm2_rn(rx, ry);
    const float gate = (__fmaf_rn(vy, ry, __fmul_rn(vx, rx)) > 0.f) ? 1.f : 0.f;
    const float nr = fmaxf(r, 1e-12f);
    const float nx = __fdiv_rn(rx, nr), ny = __fdiv_rn(ry, nr);
    const float ga = __fmul_rn(gate, k.A);
    if (VERSION == 0) {
        const float e = expf(__fmul_rn(k.B, r));
        fx = __fadd_rn(fx, __fmul_rn(__fmul_rn(ga, e), nx));
        fy = __fadd_rn(fy, __fmul_rn(__fmul_rn(ga, e), ny));
    } else {
        const float ux = __fsub_rn(vm.x, vx), uy = __fsub_rn(vm.y, vy);
        const float cr = fmaxf(r, 1e-8f), cu = fmaxf(norm2_rn(ux, uy), 1e-8f);
        const float cosv = __fadd_rn(__fmul_rn(__fdiv_rn(rx, cr), __fdiv_rn(ux, cu)),
                                     __fmul_rn(__fdiv_rn(ry, cr), __fdiv_rn(uy, cu)));
        const float cross = __fsub_rn(__fmul_rn(rx, ey), __fmul_rn(ry, ex));
        const float s = (cross > 0.f) ? -k.sin_t : k.sin_t;
        const float dx = __fadd_rn(__fmul_rn(k.cos_t, nx), __fmul_rn(-s, ny));
        const float dy = __fadd_rn(__fmul_rn(s, nx), __fmul_rn(k.cos_t, ny));
        const float arg = __fadd_rn(__fadd_rn(__fmul_rn(k.B, r), __fmul_rn(k.C, cosv)),
                                    __fmul_rn(__fmul_rn(k.D, r), cosv));
        const float e = expf(arg);
        fx = __fadd_rn(fx, __fmul_rn(__fmul_rn(ga, e), dx));
        fy = __fadd_rn(fy, __fmul_rn(__fmul_rn(ga, e), dy));
    }
}

// partial[split][row - row0] = sum over this split's columns of  view*A*exp(..)*direc
template <int VERSION, int R, bool EXACT>
__global__ void __launch_bounds__(ML_THREADS) mlapm_pairs_kernel(const float2 *__restrict__ pos,
                                                                 const float2 *__restrict__ vel,
                                                                 const float2 *__restrict__ dest, int N, int row0,
                                                                 int row1, int cols_per_split, MlConst k,
                                                                 float2 *__restrict__ partial) {
    __shared__ __align__(16) float2 sp[2][ML_TILE];
    __shared__ __align__(16) float2 sv[2][ML_TILE];
    __shared__ __align__(8) uint64_t bars[2];
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
    }
    __syncthreads();

    const int nrows = row1 - row0;
    const int rbase = blockIdx.x * (ML_THREADS * R);
    float px[R], py[R], vx[R], vy[R], ex[R], ey[R], fx[R], fy[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
        int rl = rbase + i * ML_THREADS + threadIdx.x;
        rl = rl < nrows ? rl : nrows - 1;
        const int n = row0 + rl;
        const float2 p = pos[n], v = vel[n], e = mlapm_dest_dir(p, dest[n]);
        px[i] = p.x; py[i] = p.y; vx[i] = v.x; vy[i] = v.y;
        ex[i] = e.x; ey[i] = e.y;
        fx[i] = 0.f; fy[i] = 0.f;
    }

    const int c0 = blockIdx.y * cols_per_split;
    const int c1 = min(N, c0 + cols_per_split);
    const int ncols = c1 - c0;
    const int ntiles = (ncols + ML_TILE - 1) / ML_TILE;
    uint32_t phase_bits = 0;
    bool waits[2] = {false, false};
    if (ntiles > 0) {
        const int tn = min(ncols, ML_TILE);
        waits[0] = stage_tile_pv(sp[0], sv[0], pos + c0, vel + c0, tn, &bars[0]);
    }
    __syncthreads();
    for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        if (t + 1 < ntiles) {
            const int m1 = c0 + (t + 1) * ML_TILE;
            const int tn1 = min(c1 - m1, ML_TILE);
            waits[buf ^ 1] = stage_tile_pv(sp[buf ^ 1], sv[buf ^ 1], pos + m1, vel + m1, tn1, &bars[buf ^ 1]);
        }
        if (waits[buf]) {
            mbar_wait(&bars[buf], (phase_bits >> buf) & 1u);
            phase_bits ^= (1u << buf);
        }
        const int tn = min(c1 - (c0 + t * ML_TILE), ML_TILE);
        const float2 *tp = sp[buf];
        const float2 *tv = sv[buf];
#pragma unroll 2
        for (int j = 0; j < tn; ++j) {
            const float2 pm = tp[j];
            const float2 vm = tv[j];
#pragma unroll
            for (int i = 0; i < R; ++i) {
                if (EXACT) pair_exact<VERSION>(px[i], py[i], vx[i], vy[i], ex[i], ey[i], pm, vm, k, fx[i], fy[i]);
                else pair_fast<VERSION>(px[i], py[i], vx[i], vy[i], ex[i], ey[i], pm, vm, k, fx[i], fy[i]);
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < R; ++i) {
        const int rl = rbase + i * ML_THREADS + threadIdx.x;
        if (rl < nrows) partial[static_cast<int64_t>(blockIdx.y) * nrows + rl] = make_float2(fx[i], fy[i]);
    }
}

// force = (v0*ed - v)/tau - sum_splits partial ; action = v + force*dt ; optional p' = p + action*dt and arrival.
__global__ void mlapm_finalize_kernel(const float2 *__restrict__ pos, const float2 *__restrict__ vel,
                                      const float *__restrict__ ds, int ds_dim, const float2 *__restrict__ dest,
                                      int row0, int row1, int nsplit, const float2 *__restrict__ partial, float tau,
                                      float dt, float radius, float2 *__restrict__ action,
                                      float2 *__restrict__ pos_new, uint8_t *__restrict__ arrived) {
    const int rl = blockIdx.x * blockDim.x + threadIdx.x;
    const int nrows = row1 - row0;
    if (rl >= nrows) return;
    const int n = row0 + rl;
    const float2 p = pos[n], v = vel[n], d = dest[n];
    const float dsx = ds[static_cast<int64_t>(n) * ds_dim];
    const float dsy = ds[static_cast<int64_t>(n) * ds_dim + (ds_dim > 1 ? 1 : 0)];
    const float2 fd = mlapm_dest_term(p, v, d, dsx, dsy, tau);
    float sx = 0.f, sy = 0.f;
    for (int s = 0; s < nsplit; ++s) {
        const float2 q = partial[static_cast<int64_t>(s) * nrows + rl];
        sx = __fadd_rn(sx, q.x); sy = __fadd_rn(sy, q.y);
    }
    const float2 a = mlapm_action(v, fd, sx, sy, dt);
    action[rl] = a;
    if (pos_new || arrived) {
        const float2 q = mlapm_move(p, a, dt);
        if (pos_new) pos_new[rl] = q;
        if (arrived) arrived[rl] = mlapm_arrived(q, d, radius) ? 1 : 0;
    }
}


// =====================================================================================================================
// Production pair kernel (v2): packed FP32 (Blackwell FFMA2/FMUL2/FADD2, two rows per instruction), SoA-duplicated
// column tiles staged by ONE TMA bulk copy per stage, rotation and amplitude hoisted out of the pair loop.
//
//   sum_m view*A*exp(..)*R(theta_nm) r^  =  A * [ cos_t*Sx - sin_t*Ty' ,  sin_t*Tx' + cos_t*Sy ]
//     Sx = sum w rx,  Sy = sum w ry,  Ty' = sum (w sigma) ry,  Tx' = sum (w sigma) rx,
//     w = view * exp(..)/r,  sigma = -1 if (vr x e) > 0 else +1                        (mlapm.py:33-39)
//
// Per ordered pair: 26 packed-FP32 instructions per TWO pairs + 3 MUFU + 2 ALU-pipe selects per pair, i.e. 19 issue
// slots per pair (v1: 37), FP32 pipe 26 and MUFU pipe 24 cycles per 32 pairs per SM sub-partition.
// The two discontinuous gates use the reference's exact fp32 arithmetic: view = fmaf(vy,ry,vx*rx) > 0 (einsum/bmm),
// cross = fl(fl(rx*ey) - fl(ry*ex)) un-fused, whose sign is the order of the two rounded products (equal products ->
// sigma = +1, the reference's masked_fill_(theta == 0, +theta)).
// =====================================================================================================================
constexpr int M2_THREADS = 128;
constexpr int M2_TILE = 512;                      // columns per stage: 512 * 16 B = 8 KB
constexpr int M2_COLF = 4;                        // floats per column record {px,py,vx,vy}; the packed instructions
                                                  // read them as scalar-broadcast operands (SASS `Rn.F32`)

__device__ __forceinline__ float2 splat(float x) { return make_float2(x, x); }

// col8[j] = {px,py,vx,vy} for j < N, padded up to Npad with copies of the last agent (never evaluated:
// the pair loop stops at N; the padding only keeps the fixed-size TMA bulk copies in bounds).
__global__ void mlapm_prep_kernel(const float2 *__restrict__ pos, const float2 *__restrict__ vel, int N, int Npad,
                                  float4 *__restrict__ col8) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= Npad) return;
    const int s = j < N ? j : N - 1;
    const float2 p = pos[s], v = vel[s];
    col8[j] = make_float4(p.x, p.y, v.x, v.y);
}

struct M2Const {
    float Bl, Cl, Dl;                  // B, C, D times log2(e)
};

// Two rows (packed lanes) against one column.
template <int VERSION>
__device__ __forceinline__ void pair2(const float2 npx, const float2 npy, const float2 vx, const float2 vy,
                                      const float2 nvx, const float2 nvy, const float2 ex, const float2 ey,
                                      const float4 cp, const float2 Bl, const float2 Cl,
                                      const float2 Dl, float2 &Sx, float2 &Sy, float2 &Tx, float2 &Ty) {
    const float2 eps = splat(1e-30f);
    const float2 rx = __fadd2_rn(make_float2(cp.x, cp.x), npx);            // vr = p_m - p_n          (mlapm.py:25)
    const float2 ry = __fadd2_rn(make_float2(cp.y, cp.y), npy);
    const float2 g = __ffma2_rn(vy, ry, __fmul2_rn(vx, rx));               // einsum('nk,nmk->nm')    (mlapm.py:27)
    const float2 r2 = __ffma2_rn(ry, ry, __ffma2_rn(rx, rx, eps));
    const float2 ir = make_float2(rsqrt_approx(r2.x), rsqrt_approx(r2.y));
    const float2 r = __fmul2_rn(r2, ir);
    float2 w;
    if (VERSION == 0) {
        const float2 arg = __fmul2_rn(Bl, r);
        w = __fmul2_rn(make_float2(ex2_approx(arg.x), ex2_approx(arg.y)), ir);
        w.x = g.x > 0.f ? w.x : 0.f;
        w.y = g.y > 0.f ? w.y : 0.f;
        Sx = __ffma2_rn(w, rx, Sx);
        Sy = __ffma2_rn(w, ry, Sy);
    } else {
        const float2 ux = __fadd2_rn(make_float2(cp.z, cp.z), nvx);        // vv = v_m - v_n          (mlapm.py:31)
        const float2 uy = __fadd2_rn(make_float2(cp.w, cp.w), nvy);
        const float2 u2 = __ffma2_rn(uy, uy, __ffma2_rn(ux, ux, eps));
        const float2 iu = make_float2(rsqrt_approx(u2.x), rsqrt_approx(u2.y));
        const float2 dot = __ffma2_rn(ry, uy, __fmul2_rn(rx, ux));
        // cosine_similarity cs = dot*ir*iu (mlapm.py:32); B r + (C + D r) cs = B r + (dot*iu) (C/r + D): one
        // packed instruction fewer than forming cs (r*ir == 1 to 2^-22, far inside the 1e-5 gate)
        const float2 q = __fmul2_rn(dot, iu);
        // vr x e = fl(rx*ey) - fl(ry*ex) un-fused: its sign is the order of the two rounded products    (mlapm.py:33)
        const float2 m1 = __fmul2_rn(rx, ey), m2 = __fmul2_rn(ry, ex);
        const float2 arg = __ffma2_rn(q, __ffma2_rn(Cl, ir, Dl), __fmul2_rn(Bl, r));
        w = __fmul2_rn(make_float2(ex2_approx(arg.x), ex2_approx(arg.y)), ir);
        w.x = g.x > 0.f ? w.x : 0.f;                                       // view gate
        w.y = g.y > 0.f ? w.y : 0.f;
        float2 ws;                                                         // w * sigma; cross == 0 -> +theta  (:34)
        ws.x = m1.x > m2.x ? -w.x : w.x;
        ws.y = m1.y > m2.y ? -w.y : w.y;
        Sx = __ffma2_rn(w, rx, Sx);
        Sy = __ffma2_rn(w, ry, Sy);
        Tx = __ffma2_rn(ws, rx, Tx);
        Ty = __ffma2_rn(ws, ry, Ty);
    }
}

// partial[split][row - row0] = (Sx, Sy, Tx', Ty') over this split's columns.  Each thread owns 2*RP rows.
template <int VERSION, int RP>
__global__ void __launch_bounds__(M2_THREADS) mlapm_pairs2_kernel(const float2 *__restrict__ pos,
                                                                  const float2 *__restrict__ vel,
                                                                  const float2 *__restrict__ dest,
                                                                  const float4 *__restrict__ col8, int N, int row0,
                                                                  int row1, int cols_per_split, M2Const k,
                                                                  float4 *__restrict__ partial) {
    __shared__ __align__(128) float4 tile[2][M2_TILE];
    __shared__ __align__(8) uint64_t bars[2];
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
    }
    __syncthreads();

    const int nrows = row1 - row0;
    const int rbase = blockIdx.x * (M2_THREADS * 2 * RP);
    float2 npx[RP], npy[RP], vx[RP], vy[RP], nvx[RP], nvy[RP], ex[RP], ey[RP], Sx[RP], Sy[RP], Tx[RP], Ty[RP];
#pragma unroll
    for (int i = 0; i < RP; ++i) {
        float t[2][6];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            int rl = rbase + (2 * i + h) * M2_THREADS + threadIdx.x;
            rl = rl < nrows ? rl : nrows - 1;
            const int n = row0 + rl;
            const float2 p = pos[n], v = vel[n], e = mlapm_dest_dir(p, dest[n]);
            t[h][0] = p.x; t[h][1] = p.y; t[h][2] = v.x; t[h][3] = v.y;
            t[h][4] = e.x; t[h][5] = e.y;
        }
        npx[i] = make_float2(-t[0][0], -t[1][0]); npy[i] = make_float2(-t[0][1], -t[1][1]);
        vx[i] = make_float2(t[0][2], t[1][2]); vy[i] = make_float2(t[0][3], t[1][3]);
        nvx[i] = make_float2(-t[0][2], -t[1][2]); nvy[i] = make_float2(-t[0][3], -t[1][3]);
        ex[i] = make_float2(t[0][4], t[1][4]); ey[i] = make_float2(t[0][5], t[1][5]);
        Sx[i] = Sy[i] = Tx[i] = Ty[i] = make_float2(0.f, 0.f);
    }
    const float2 Bl = splat(k.Bl), Cl = splat(k.Cl), Dl = splat(k.Dl);

    const int c0 = blockIdx.y * cols_per_split;                 // multiple of M2_TILE
    const int c1 = min(N, c0 + cols_per_split);
    const int ntiles = (c1 - c0 + M2_TILE - 1) / M2_TILE;
    constexpr uint32_t TILE_BYTES = M2_TILE * M2_COLF * sizeof(float);
    if (threadIdx.x == 0 && ntiles > 0) {
        mbar_expect_tx(&bars[0], TILE_BYTES);
        tma_bulk_g2s(tile[0], col8 + static_cast<int64_t>(c0), TILE_BYTES, &bars[0]);
    }
    uint32_t phase_bits = 0;
    for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        if (threadIdx.x == 0 && t + 1 < ntiles) {               // tile[buf^1] was released by the barrier below
            mbar_expect_tx(&bars[buf ^ 1], TILE_BYTES);
            tma_bulk_g2s(tile[buf ^ 1], col8 + static_cast<int64_t>(c0 + (t + 1) * M2_TILE), TILE_BYTES,
                         &bars[buf ^ 1]);
        }
        mbar_wait(&bars[buf], (phase_bits >> buf) & 1u);
        phase_bits ^= (1u << buf);
        const int tn = min(c1 - (c0 + t * M2_TILE), M2_TILE);
        const float4 *tl = tile[buf];
#pragma unroll 4
        for (int j = 0; j < tn; ++j) {
            const float4 cp = tl[j];
#pragma unroll
            for (int i = 0; i < RP; ++i)
                pair2<VERSION>(npx[i], npy[i], vx[i], vy[i], nvx[i], nvy[i], ex[i], ey[i], cp, Bl, Cl, Dl, Sx[i],
                               Sy[i], Tx[i], Ty[i]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < RP; ++i) {
        const int ra = rbase + (2 * i) * M2_THREADS + threadIdx.x;
        const int rb = ra + M2_THREADS;
        float4 *out = partial + static_cast<int64_t>(blockIdx.y) * nrows;
        if (ra < nrows) out[ra] = make_float4(Sx[i].x, Sy[i].x, Tx[i].x, Ty[i].x);
        if (rb < nrows) out[rb] = make_float4(Sx[i].y, Sy[i].y, Tx[i].y, Ty[i].y);
    }
}

// =====================================================================================================================
// Symmetric pair kernel (v3): every UNORDERED pair {n,m} is evaluated once and feeds both rows.
//
// Everything smooth in the GC formula is symmetric under n <-> m: vr -> -vr, vv -> -vv, so r, |vv|, cos(vr,vv) and
// the exponent B r + C cos + D r cos are the same numbers for (n,m) and (m,n); only the two discontinuous gates (the
// view test of the row's own velocity and the sign of vr x e of the row's own destination direction) and the
// accumulation differ.  The 16 packed instructions + 3 MUFU of the shared part are therefore spent once per unordered
// pair, and each direction adds 8 packed instructions (gate products, cross products, 4 accumulations):
// 32 packed instructions + 6 MUFU per 128 ordered pairs instead of 48 + 12.  The gates keep the reference's exact
// fp32 arithmetic in BOTH directions because fp32 subtraction, multiplication and fma are odd-symmetric:
//   vr[m,n] = fl(p_n - p_m) = -fl(p_m - p_n),  v_m . vr[m,n] = -fmaf(v_my, ry, fl(v_mx rx))  ->  view' = (gc < 0),
//   vr[m,n] x e_m = fl(fl(ry e_mx) - fl(rx e_my))                                          ->  sigma' = -1 iff m2c > m1c.
//
// Schedule: agents are cut into blocks of 512; block pair (I, J = I + d mod T) is evaluated by the CTA of row block I
// for d = 0 .. floor(T/2) (a circulant schedule: every unordered block pair exactly once, every row block the same
// amount of work; for even T the pairs at d = T/2 belong to I < T/2).  d = 0 is the diagonal block, evaluated one
// direction at a time like v2.  A thread keeps 8 rows (4 packed lane pairs) in registers and streams J's columns from
// shared memory (TMA bulk copies, double buffered), so the row direction accumulates in registers as before.  The
// column direction needs, per column, the sum over all 512 rows of the CTA: the two packed lanes are added, each lane
// parks its 4 sums for a batch of 8 columns in a per-warp shared-memory scratch, the warp transposes (lane -> column
// lane/4, every 4th entry) and finishes with two shuffle stages; the warps' column sums are added in a fixed order and
// go into int64 fixed-point accumulators per agent (ms_add_columns) -- deterministic.  Cost of the reduction per column
// and warp: 9 FADD + 1 SHFL + 2 x 128-bit shared accesses against 64 packed instructions of pair work.
// The finalize kernel subtracts the column-direction sums (vr' = -vr) from the row-direction sums.
// =====================================================================================================================
constexpr int MS_BLOCK = 512;                     // agents per block of the schedule = rows per CTA
constexpr int MS_CT = 128;                        // columns per shared-memory stage (4 KB)
constexpr int MS_BATCH = 8;                       // columns per warp-level reduction
constexpr int MS_RED_STRIDE = 36;                 // float4 per column of the scratch: 32 lanes + 64 B skew (no conflicts)
constexpr int MS_RECF = 8;                        // floats per agent record {px,py,vx,vy, ex,ey,0,0}
constexpr float MS_FAR = 1.0e18f;                 // padding agents sit here: exp(B r) == 0 exactly, nothing overflows
static_assert(MS_BLOCK % MS_CT == 0 && MS_CT % MS_BATCH == 0 && (MS_BATCH == 8 || MS_BATCH == 4), "bad stage shape");

template <int THREADS>
struct MsSmem {
    float4 tile[2][MS_CT * 2];
    float4 red[THREADS / 32][MS_BATCH * MS_RED_STRIDE];
    float4 colacc[THREADS / 32][MS_CT];
    uint64_t bars[2];
};

// Slot j of the symmetric kernels' inputs for this step: zeroed fixed-point accumulators, a cleared NaN flag (bad may
// be null) and the record rec[j] = {px,py,vx,vy},{ex,ey,0,0} of agent n; returns its {px,py,vx,vy}.  agent == false: a
// padding slot, an agent far away whose weight underflows to exactly 0 in both directions, so block tails need no masks.
__device__ __forceinline__ float4 ms_prep_slot(int j, bool agent, int n, const float2 *__restrict__ pos,
                                               const float2 *__restrict__ vel, const float2 *__restrict__ dest,
                                               float4 *__restrict__ rec, ulonglong2 *__restrict__ acc,
                                               unsigned *__restrict__ bad) {
    acc[2 * j] = make_ulonglong2(0ull, 0ull);
    acc[2 * j + 1] = make_ulonglong2(0ull, 0ull);
    if (bad) bad[j] = 0u;
    if (!agent) {
        const float4 far = make_float4(MS_FAR, MS_FAR, 0.f, 0.f);
        rec[2 * j] = far;
        rec[2 * j + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
        return far;
    }
    const float2 p = pos[n], v = vel[n], d = dest[n];
    const float4 pv = make_float4(p.x, p.y, v.x, v.y);
    rec[2 * j] = pv;
    const float2 e = mlapm_dest_dir(p, d);
    rec[2 * j + 1] = make_float4(e.x, e.y, 0.f, 0.f);
    return pv;
}

// The slots of the dense symmetric evaluation: agent j in slot j, padding from N up to Npad.
__global__ void mlapm_prep_sym_kernel(const float2 *__restrict__ pos, const float2 *__restrict__ vel,
                                      const float2 *__restrict__ dest, int N, int Npad, float4 *__restrict__ rec,
                                      ulonglong2 *__restrict__ colsum, unsigned *__restrict__ bad) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= Npad) return;
    ms_prep_slot(j, j < N, j, pos, vel, dest, rec, colsum, bad);
}

// Two rows (packed lanes) against one column, both directions.  Row sums accumulate in S/T; the column's share is
// returned in cS/cT (FIRST: overwritten, else accumulated) in the row's sign convention (the caller subtracts it).
template <int VERSION, bool FIRST>
__device__ __forceinline__ void pair2sym(const float2 npx, const float2 npy, const float2 vx, const float2 vy,
                                         const float2 nvx, const float2 nvy, const float2 ex, const float2 ey,
                                         const float4 cp, const float4 ce, const float2 Bl, const float2 Cl,
                                         const float2 Dl, float2 &Sx, float2 &Sy, float2 &Tx, float2 &Ty,
                                         float2 &cSx, float2 &cSy, float2 &cTx, float2 &cTy) {
    const float2 eps = splat(1e-30f);
    const float2 rx = __fadd2_rn(splat(cp.x), npx);                        // vr[n,m] = p_m - p_n     (mlapm.py:25)
    const float2 ry = __fadd2_rn(splat(cp.y), npy);
    const float2 g = __ffma2_rn(vy, ry, __fmul2_rn(vx, rx));               // v_n . vr[n,m]           (mlapm.py:27)
    const float2 gc = __ffma2_rn(splat(cp.w), ry, __fmul2_rn(splat(cp.z), rx));   // = -(v_m . vr[m,n])
    const float2 r2 = __ffma2_rn(ry, ry, __ffma2_rn(rx, rx, eps));
    const float2 ir = make_float2(rsqrt_approx(r2.x), rsqrt_approx(r2.y));
    const float2 r = __fmul2_rn(r2, ir);
    float2 w0;
    if (VERSION == 0) {
        const float2 arg = __fmul2_rn(Bl, r);
        w0 = __fmul2_rn(make_float2(ex2_approx(arg.x), ex2_approx(arg.y)), ir);
    } else {
        const float2 ux = __fadd2_rn(splat(cp.z), nvx);                    // vv[n,m] = v_m - v_n     (mlapm.py:31)
        const float2 uy = __fadd2_rn(splat(cp.w), nvy);
        const float2 u2 = __ffma2_rn(uy, uy, __ffma2_rn(ux, ux, eps));
        const float2 iu = make_float2(rsqrt_approx(u2.x), rsqrt_approx(u2.y));
        const float2 dot = __ffma2_rn(ry, uy, __fmul2_rn(rx, ux));
        const float2 q = __fmul2_rn(dot, iu);
        const float2 arg = __ffma2_rn(q, __ffma2_rn(Cl, ir, Dl), __fmul2_rn(Bl, r));
        w0 = __fmul2_rn(make_float2(ex2_approx(arg.x), ex2_approx(arg.y)), ir);
    }
    float2 w, wc;
    w.x = g.x > 0.f ? w0.x : 0.f;                                          // view gate of the row
    w.y = g.y > 0.f ? w0.y : 0.f;
    wc.x = gc.x < 0.f ? w0.x : 0.f;                                        // view gate of the column
    wc.y = gc.y < 0.f ? w0.y : 0.f;
    Sx = __ffma2_rn(w, rx, Sx);
    Sy = __ffma2_rn(w, ry, Sy);
    cSx = FIRST ? __fmul2_rn(wc, rx) : __ffma2_rn(wc, rx, cSx);
    cSy = FIRST ? __fmul2_rn(wc, ry) : __ffma2_rn(wc, ry, cSy);
    if (VERSION != 0) {
        // sign of vr x e from the order of the two rounded products, both directions             (mlapm.py:33-34)
        const float2 m1 = __fmul2_rn(rx, ey), m2 = __fmul2_rn(ry, ex);
        const float2 m1c = __fmul2_rn(rx, splat(ce.y)), m2c = __fmul2_rn(ry, splat(ce.x));
        float2 ws, wcs;
        ws.x = m1.x > m2.x ? -w.x : w.x;
        ws.y = m1.y > m2.y ? -w.y : w.y;
        wcs.x = m2c.x > m1c.x ? -wc.x : wc.x;
        wcs.y = m2c.y > m1c.y ? -wc.y : wc.y;
        Tx = __ffma2_rn(ws, rx, Tx);
        Ty = __ffma2_rn(ws, ry, Ty);
        cTx = FIRST ? __fmul2_rn(wcs, rx) : __ffma2_rn(wcs, rx, cTx);
        cTy = FIRST ? __fmul2_rn(wcs, ry) : __ffma2_rn(wcs, ry, cTy);
    } else if (FIRST) {
        cTx = cTy = make_float2(0.f, 0.f);
    }
}

// A thread's 2 * RPS rows of one row block, two per packed lane pair, and their row-direction sums.
template <int RPS>
struct MsRows {
    float2 npx[RPS], npy[RPS], vx[RPS], vy[RPS], nvx[RPS], nvy[RPS], ex[RPS], ey[RPS], Sx[RPS], Sy[RPS], Tx[RPS],
        Ty[RPS];
};

// Rows of block I: lanes x / y of pair i are the block's rows (2i) THREADS + tid and (2i + 1) THREADS + tid, with the
// CTA's THREADS = MS_BLOCK / (2 RPS) threads; the sums start at 0.
template <int RPS>
__device__ __forceinline__ void ms_load_rows(MsRows<RPS> &r, const float4 *__restrict__ rec, int I, int tid) {
    constexpr int THREADS = MS_BLOCK / (2 * RPS);
#pragma unroll
    for (int i = 0; i < RPS; ++i) {
        const int64_t na = static_cast<int64_t>(I) * MS_BLOCK + (2 * i) * THREADS + tid;
        const int64_t nb = na + THREADS;
        const float4 a0 = rec[2 * na], a1 = rec[2 * na + 1], b0 = rec[2 * nb], b1 = rec[2 * nb + 1];
        r.npx[i] = make_float2(-a0.x, -b0.x); r.npy[i] = make_float2(-a0.y, -b0.y);
        r.vx[i] = make_float2(a0.z, b0.z); r.vy[i] = make_float2(a0.w, b0.w);
        r.nvx[i] = make_float2(-a0.z, -b0.z); r.nvy[i] = make_float2(-a0.w, -b0.w);
        r.ex[i] = make_float2(a1.x, b1.x); r.ey[i] = make_float2(a1.y, b1.y);
        r.Sx[i] = r.Sy[i] = r.Tx[i] = r.Ty[i] = make_float2(0.f, 0.f);
    }
}

// One staged tile of MS_CT column records `tl` of the rows' own (diagonal) block: every ordered pair appears, so each
// is evaluated in the row direction only (pair2).
template <int VERSION, int RPS>
__device__ __forceinline__ void ms_diag_tile(MsRows<RPS> &r, const float4 *tl, float2 Bl, float2 Cl, float2 Dl) {
#pragma unroll 4
    for (int j = 0; j < MS_CT; ++j) {
        const float4 cp = tl[2 * j];
#pragma unroll
        for (int i = 0; i < RPS; ++i)
            pair2<VERSION>(r.npx[i], r.npy[i], r.vx[i], r.vy[i], r.nvx[i], r.nvy[i], r.ex[i], r.ey[i], cp, Bl, Cl, Dl,
                           r.Sx[i], r.Sy[i], r.Tx[i], r.Ty[i]);
    }
}

// One staged tile of MS_CT column records `tl` of another block: every pair feeds both directions (pair2sym).  The
// warp's column-direction sums go to colacc[column]: the two packed lanes are added, each lane parks its sums of a
// batch of MS_BATCH columns in the warp's scratch `red`, the warp transposes (lane -> column lane/LPC, every LPC-th
// entry) and finishes with shuffles.
template <int VERSION, int RPS>
__device__ __forceinline__ void ms_pair_tile(MsRows<RPS> &r, const float4 *tl, float4 *red, float4 *colacc, int lane,
                                             float2 Bl, float2 Cl, float2 Dl) {
    constexpr int LPC = 32 / MS_BATCH;                      // lanes that share a column in the transposed sum
    for (int b = 0; b < MS_CT / MS_BATCH; ++b) {
#pragma unroll
        for (int c = 0; c < MS_BATCH; ++c) {
            const float4 cp = tl[2 * (b * MS_BATCH + c)];
            const float4 ce = tl[2 * (b * MS_BATCH + c) + 1];
            float2 cSx, cSy, cTx, cTy;
            pair2sym<VERSION, true>(r.npx[0], r.npy[0], r.vx[0], r.vy[0], r.nvx[0], r.nvy[0], r.ex[0], r.ey[0], cp, ce,
                                    Bl, Cl, Dl, r.Sx[0], r.Sy[0], r.Tx[0], r.Ty[0], cSx, cSy, cTx, cTy);
#pragma unroll
            for (int i = 1; i < RPS; ++i)
                pair2sym<VERSION, false>(r.npx[i], r.npy[i], r.vx[i], r.vy[i], r.nvx[i], r.nvy[i], r.ex[i], r.ey[i], cp,
                                         ce, Bl, Cl, Dl, r.Sx[i], r.Sy[i], r.Tx[i], r.Ty[i], cSx, cSy, cTx, cTy);
            red[c * MS_RED_STRIDE + lane] = make_float4(cSx.x + cSx.y, cSy.x + cSy.y, cTx.x + cTx.y, cTy.x + cTy.y);
        }
        __syncwarp();
        const float4 *col = red + (lane / LPC) * MS_RED_STRIDE + (lane % LPC);
        float4 a = col[0];
#pragma unroll
        for (int e = 1; e < 32 / LPC; ++e) {
            const float4 t = col[LPC * e];
            a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
        }
#pragma unroll
        for (int o = 1; o < LPC; o <<= 1) {
            a.x += __shfl_xor_sync(0xffffffffu, a.x, o);
            a.y += __shfl_xor_sync(0xffffffffu, a.y, o);
            a.z += __shfl_xor_sync(0xffffffffu, a.z, o);
            a.w += __shfl_xor_sync(0xffffffffu, a.w, o);
        }
        if (lane % LPC == 0) colacc[b * MS_BATCH + lane / LPC] = a;
        __syncwarp();
    }
}

// The column-direction sums of one stage over the CTA's rows (the warps' colacc, added in warp order) into the
// crowd-wide FIXED-POINT accumulators acc[slot][4] (int64, 2^-s resolution) of the stage's slots j0 .. j0 + MS_CT - 1,
// with fire-and-forget 64-bit atomics.  Integer addition is associative, so the total does not depend on the order in
// which the block pairs that share a column arrive: deterministic like per-pair partial arrays, with O(N) instead of
// O(N^2 / 64) workspace and DRAM traffic.  A NaN or inf has no fixed-point value: it poisons the slot through its flag
// in bad, unless bad is null (see SymPartials).
template <int THREADS>
__device__ __forceinline__ void ms_add_columns(const float4 (*colacc)[MS_CT], unsigned long long *acc, unsigned *bad,
                                               int64_t j0, float colscale, int tid) {
    for (int c = tid; c < MS_CT; c += THREADS) {
        float4 a = colacc[0][c];
#pragma unroll
        for (int wv = 1; wv < THREADS / 32; ++wv) {
            const float4 t = colacc[wv][c];
            a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
        }
        if (bad && !isfinite(a.x + a.y + a.z + a.w)) bad[j0 + c] = 1u;
        unsigned long long *dst = acc + (j0 + c) * 4;
        atomicAdd(dst + 0, static_cast<unsigned long long>(__float2ll_rn(a.x * colscale)));
        atomicAdd(dst + 1, static_cast<unsigned long long>(__float2ll_rn(a.y * colscale)));
        atomicAdd(dst + 2, static_cast<unsigned long long>(__float2ll_rn(a.z * colscale)));
        atomicAdd(dst + 3, static_cast<unsigned long long>(__float2ll_rn(a.w * colscale)));
    }
}

// partialR[split][local row] = row-direction (Sx,Sy,Tx',Ty') over the split's block pairs; the column-direction sums
// of block pair (I, J = I + d mod T) go into colsum (ms_add_columns).
// RPS = packed row pairs per thread (2 * RPS rows): the CTA's 512 rows are spread over THREADS = 256 / RPS threads.
template <int VERSION, int RPS>
__global__ void __launch_bounds__(MS_BLOCK / (2 * RPS)) mlapm_sym_kernel(const float4 *__restrict__ rec, int T, int D,
                                                                         int I0, int per, int sub, M2Const k,
                                                                         float4 *__restrict__ partialR, int nrows_pad,
                                                                         unsigned long long *__restrict__ colsum,
                                                                         float colscale, unsigned *__restrict__ bad) {
    constexpr int THREADS = MS_BLOCK / (2 * RPS);
    constexpr int SPB = MS_BLOCK / MS_CT;                   // stages per block pair
    extern __shared__ __align__(128) unsigned char ms_smem_raw[];
    MsSmem<THREADS> &sm = *reinterpret_cast<MsSmem<THREADS> *>(ms_smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        mbar_init(&sm.bars[0], 1);
        mbar_init(&sm.bars[1], 1);
        mbar_fence_init();
    }
    __syncthreads();

    const int I = I0 + blockIdx.x;
    int L = D + 1;                                          // d = 0 .. D
    if (!(T & 1) && 2 * I >= T) L = D;                      // even T: the pairs at d = T/2 belong to I < T/2
    // blockIdx.y = (group of `per` block pairs) * sub + (which 1/sub of each pair's column stages): small shards use
    // sub > 1 so that the grid still has several waves of CTAs
    const int sy = blockIdx.y / sub, su = blockIdx.y - sy * sub;
    const int spc = SPB / sub;                               // stages of a block pair this CTA handles
    const int d_lo = sy * per;
    const int d_hi = min(d_lo + per, L);

    MsRows<RPS> rw;
    ms_load_rows(rw, rec, I, tid);
    const float2 Bl = splat(k.Bl), Cl = splat(k.Cl), Dl = splat(k.Dl);

    const int nst = d_hi > d_lo ? (d_hi - d_lo) * spc : 0;
    constexpr uint32_t STAGE_BYTES = MS_CT * MS_RECF * sizeof(float);
    auto stage_j0 = [&](int s) {                             // first slot of stage s
        int J = I + d_lo + s / spc;
        J = J >= T ? J - T : J;
        return static_cast<int64_t>(J) * MS_BLOCK + (su * spc + s % spc) * MS_CT;
    };
    if (tid == 0 && nst > 0) {
        mbar_expect_tx(&sm.bars[0], STAGE_BYTES);
        tma_bulk_g2s(sm.tile[0], rec + stage_j0(0) * 2, STAGE_BYTES, &sm.bars[0]);
    }
    uint32_t phase_bits = 0;
    for (int s = 0; s < nst; ++s) {
        const int buf = s & 1;
        if (tid == 0 && s + 1 < nst) {                      // tile[buf^1] was released by the barrier below
            mbar_expect_tx(&sm.bars[buf ^ 1], STAGE_BYTES);
            tma_bulk_g2s(sm.tile[buf ^ 1], rec + stage_j0(s + 1) * 2, STAGE_BYTES, &sm.bars[buf ^ 1]);
        }
        mbar_wait(&sm.bars[buf], (phase_bits >> buf) & 1u);
        phase_bits ^= (1u << buf);
        // the off-diagonal branch first: in the other order ptxas emits the diagonal loop twice
        if (d_lo + s / spc != 0) {
            ms_pair_tile<VERSION>(rw, sm.tile[buf], sm.red[warp], sm.colacc[warp], lane, Bl, Cl, Dl);
            __syncthreads();
            ms_add_columns<THREADS>(sm.colacc, colsum, bad, stage_j0(s), colscale, tid);
        } else {
            ms_diag_tile<VERSION>(rw, sm.tile[buf], Bl, Cl, Dl);
        }
        __syncthreads();
    }
    float4 *out = partialR + static_cast<int64_t>(blockIdx.y) * nrows_pad + static_cast<int64_t>(blockIdx.x) * MS_BLOCK;
#pragma unroll
    for (int i = 0; i < RPS; ++i) {
        out[(2 * i) * THREADS + tid] = make_float4(rw.Sx[i].x, rw.Sy[i].x, rw.Tx[i].x, rw.Ty[i].x);
        out[(2 * i + 1) * THREADS + tid] = make_float4(rw.Sx[i].y, rw.Sy[i].y, rw.Tx[i].y, rw.Ty[i].y);
    }
}

// =====================================================================================================================
// Culled symmetric evaluation: skip the block pairs whose weight is exactly zero.
//
// The production weight is ex2.approx.ftz(arg) / r with arg = Bl r + q (Cl / r + Dl), |q| <= r, so arg <= (Bl + |Dl|) r
// + |Cl| (raw: arg = Bl r).  sym_params_ok requires Bl + |Dl| < 0, so beyond r_cut = (127 + |Cl|) / -(Bl + |Dl|) every
// pair has arg < -127: ex2 flushes to +0, every fma(w, r, S) returns S unchanged and every fixed-point column share is
// 0.  Skipping those pairs changes nothing but the fp32 summation order.
//
// Per call: (1) a 32-bit Hilbert key of each agent's 4 m cell, sorted stably (cub::DeviceRadixSort, key + agent
// index), so that the agents of a 512-block live close together; (2) records in sorted order plus an axis-aligned box
// per 512-agent block and per 128-agent column stage; (3) the work list: every (row block I, column block J = I + d
// mod T, stage) item of the circulant schedule whose boxes are within r_cut, compacted in order (cub::DeviceSelect);
// (4) a persistent pair kernel over the list; (5) the finalize kernel reads each agent's sums through its sorted slot.
// Row and column directions both go into the crowd-wide int64 fixed-point accumulators, so the result does not depend
// on how the list is cut over the CTAs.
// =====================================================================================================================
constexpr float MC_CELL = 4.0f;                   // metres per cell of the sort key
constexpr int MC_SPB = MS_BLOCK / MS_CT;          // column stages per block
constexpr int MC_THREADS = 64;                    // pair kernel: 8 rows per thread (the dense kernel's measured best)
constexpr unsigned MC_NEAR_ALL = 1u, MC_EMPTY = 2u;   // box flags: holds a NaN / inf, holds no agent

// Hilbert index of cell (x, y) on the 2^16 x 2^16 grid.
__device__ __forceinline__ uint32_t hilbert16(uint32_t x, uint32_t y) {
    uint32_t d = 0;
    for (uint32_t s = 1u << 15; s > 0; s >>= 1) {
        const uint32_t rx = (x & s) ? 1u : 0u, ry = (y & s) ? 1u : 0u;
        d += s * s * ((3u * rx) ^ ry);
        if (ry == 0) {
            if (rx == 1) { x = 0xFFFFu - x; y = 0xFFFFu - y; }
            const uint32_t t = x; x = y; y = t;
        }
    }
    return d;
}

// key[n] = Hilbert index of floor(p_n / MC_CELL) (cell coordinates wrap modulo 2^16: only locality is lost), agent
// index as the value; a non-finite position sorts last.
__global__ void mlapm_cull_keys_kernel(const float2 *__restrict__ pos, int N, uint32_t *__restrict__ key,
                                       int *__restrict__ val) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float2 p = pos[n];
    uint32_t k = 0xFFFFFFFFu;
    if (isfinite(p.x) && isfinite(p.y)) {
        const uint32_t cx = static_cast<uint32_t>(__float2int_rd(p.x * (1.0f / MC_CELL))) & 0xFFFFu;
        const uint32_t cy = static_cast<uint32_t>(__float2int_rd(p.y * (1.0f / MC_CELL))) & 0xFFFFu;
        k = hilbert16(cx, cy);
    }
    key[n] = k;
    val[n] = n;
}

// One CTA of MS_BLOCK threads per block of the sorted crowd: slot j holds the agent perm[j] (ms_prep_slot; j >= N:
// padding), slot[agent] = j, and the boxes {min x, min y, max x, max y} of the
// block and of its MC_SPB column stages.  Agents with a non-finite position or velocity do not enter the min / max (no
// fminf / fmaxf on NaN); they flag their stage and block MC_NEAR_ALL instead, which keeps every item that touches them.
__global__ void __launch_bounds__(MS_BLOCK) mlapm_prep_cull_kernel(
    const float2 *__restrict__ pos, const float2 *__restrict__ vel, const float2 *__restrict__ dest,
    const int *__restrict__ perm, int N, float4 *__restrict__ rec, int *__restrict__ slot,
    ulonglong2 *__restrict__ acc, unsigned *__restrict__ bad, float4 *__restrict__ sbox, unsigned *__restrict__ sflag,
    float4 *__restrict__ bbox, unsigned *__restrict__ bflag) {
    __shared__ float4 wbox[MS_BLOCK / 32];
    __shared__ unsigned wflag[MS_BLOCK / 32];
    const int j = blockIdx.x * MS_BLOCK + threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool agent = j < N;
    const int n = agent ? perm[j] : 0;
    if (agent) slot[n] = j;
    const float4 pv = ms_prep_slot(j, agent, n, pos, vel, dest, rec, acc, bad);
    float4 b = make_float4(CUDART_INF_F, CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
    unsigned flag = MC_EMPTY;
    if (agent) {
        if (isfinite(pv.x) && isfinite(pv.y) && isfinite(pv.z) && isfinite(pv.w)) {
            b = make_float4(pv.x, pv.y, pv.x, pv.y);
            flag = 0u;
        } else {
            flag = MC_NEAR_ALL;
        }
    }
    // flags combine as: any MC_NEAR_ALL -> MC_NEAR_ALL, else any agent -> 0, else MC_EMPTY
    auto comb = [](unsigned a, unsigned c) { return (a | c) & MC_NEAR_ALL ? MC_NEAR_ALL : (a & c); };
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        b.x = fminf(b.x, __shfl_xor_sync(0xffffffffu, b.x, o));
        b.y = fminf(b.y, __shfl_xor_sync(0xffffffffu, b.y, o));
        b.z = fmaxf(b.z, __shfl_xor_sync(0xffffffffu, b.z, o));
        b.w = fmaxf(b.w, __shfl_xor_sync(0xffffffffu, b.w, o));
        flag = comb(flag, __shfl_xor_sync(0xffffffffu, flag, o));
    }
    if (lane == 0) { wbox[warp] = b; wflag[warp] = flag; }
    __syncthreads();
    if (threadIdx.x < MC_SPB + 1) {
        // thread s < MC_SPB: stage s (its MS_CT / 32 warps); thread MC_SPB: the whole block
        const int w0 = threadIdx.x < MC_SPB ? threadIdx.x * (MS_CT / 32) : 0;
        const int w1 = threadIdx.x < MC_SPB ? w0 + MS_CT / 32 : MS_BLOCK / 32;
        float4 u = wbox[w0];
        unsigned f = wflag[w0];
        for (int w = w0 + 1; w < w1; ++w) {
            const float4 t = wbox[w];
            u.x = fminf(u.x, t.x); u.y = fminf(u.y, t.y); u.z = fmaxf(u.z, t.z); u.w = fmaxf(u.w, t.w);
            f = comb(f, wflag[w]);
        }
        if (threadIdx.x < MC_SPB) {
            sbox[blockIdx.x * MC_SPB + threadIdx.x] = u;
            sflag[blockIdx.x * MC_SPB + threadIdx.x] = f;
        } else {
            bbox[blockIdx.x] = u;
            bflag[blockIdx.x] = f;
        }
    }
}

// Keep-predicate of the work list over candidate c = ((I * (D + 1) + d) * MC_SPB + stage): rows = block I, columns =
// stage `stage` of block J = I + d mod T (circulant schedule of mlapm_sym_kernel).  The box gap is rounded down, so a
// kept-or-not decision never depends on fp32 rounding in the skipping direction.
struct CullKeep {
    const float4 *sbox, *bbox;
    const unsigned *sflag, *bflag;
    int T, D;
    float rc;
    __device__ __forceinline__ bool operator()(int c) const {
        const int st = c % MC_SPB, pd = c / MC_SPB;
        const int I = pd / (D + 1), d = pd - I * (D + 1);
        if (!(T & 1) && d == D && 2 * I >= T) return false;     // even T: the pairs at d = T/2 belong to I < T/2
        int J = I + d;
        J = J >= T ? J - T : J;
        const int s = J * MC_SPB + st;
        const unsigned fr = bflag[I], fc = sflag[s];
        if ((fr | fc) & MC_EMPTY) return false;
        if ((fr | fc) & MC_NEAR_ALL) return true;
        const float4 a = bbox[I], b = sbox[s];
        const float gx = fmaxf(fmaxf(__fsub_rd(b.x, a.z), __fsub_rd(a.x, b.z)), 0.f);
        const float gy = fmaxf(fmaxf(__fsub_rd(b.y, a.w), __fsub_rd(a.y, b.w)), 0.f);
        return __fadd_rd(__fmul_rd(gx, gx), __fmul_rd(gy, gy)) <= rc * rc;
    }
};

// The symmetric pair kernel over the work list.  Persistent: CTA b takes the contiguous items [b n / G, (b+1) n / G)
// of the n = *nitems on the list (read on the device: no host sync).  Rows stay in registers while consecutive items
// share the row block; when it changes, and at the end, the row sums go into the fixed-point accumulators with the
// opposite sign of the column shares (acc = column share - row share; the finalize kernel subtracts acc).  The stages
// are evaluated as in mlapm_sym_kernel (ms_diag_tile, ms_pair_tile, ms_add_columns).
template <int VERSION>
__global__ void __launch_bounds__(MC_THREADS, 8) mlapm_sym_list_kernel(const float4 *__restrict__ rec,
                                                                      const int *__restrict__ items,
                                                                      const int *__restrict__ nitems, int T, int D,
                                                                      M2Const k, unsigned long long *__restrict__ acc,
                                                                      unsigned *__restrict__ bad, float colscale) {
    constexpr int THREADS = MC_THREADS, RPS = MS_BLOCK / (2 * THREADS);
    extern __shared__ __align__(128) unsigned char ms_smem_raw[];
    MsSmem<THREADS> &sm = *reinterpret_cast<MsSmem<THREADS> *>(ms_smem_raw);
    // the item of the stage in tile[buf] (I, d, first column j0 = J * MS_BLOCK + stage * MS_CT), written by the thread
    // that issues its copy; the loop state lives here too, which keeps the pair loop at 128 registers without spills
    __shared__ int meta[2][3];
    __shared__ int s_lo, s_cnt;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __builtin_assume(bad != nullptr);                          // never null here: one copy of ms_add_columns' loop
    const int n = *nitems;
    const int lo = static_cast<int>(static_cast<int64_t>(n) * blockIdx.x / gridDim.x);
    const int cnt = static_cast<int>(static_cast<int64_t>(n) * (blockIdx.x + 1) / gridDim.x) - lo;
    if (cnt <= 0) return;
    constexpr uint32_t STAGE_BYTES = MS_CT * MS_RECF * sizeof(float);
    auto stage_load = [&](int s, int buf) {                    // thread 0
        const int c = items[s];
        const int st = c % MC_SPB, pd = c / MC_SPB;
        const int I = pd / (D + 1), d = pd - I * (D + 1);
        const int J = I + d >= T ? I + d - T : I + d;
        const int j0 = J * MS_BLOCK + st * MS_CT;
        meta[buf][0] = I; meta[buf][1] = d; meta[buf][2] = j0;
        mbar_expect_tx(&sm.bars[buf], STAGE_BYTES);
        tma_bulk_g2s(sm.tile[buf], rec + static_cast<int64_t>(j0) * 2, STAGE_BYTES, &sm.bars[buf]);
    };
    if (tid == 0) {
        mbar_init(&sm.bars[0], 1);
        mbar_init(&sm.bars[1], 1);
        mbar_fence_init();
        s_lo = lo;
        s_cnt = cnt;
        stage_load(lo, 0);
    }
    __syncthreads();

    MsRows<RPS> rw;
    const float2 Bl = splat(k.Bl), Cl = splat(k.Cl), Dl = splat(k.Dl);
    auto flush_rows = [&](int I) {
#pragma unroll
        for (int i = 0; i < RPS; ++i) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int64_t j = static_cast<int64_t>(I) * MS_BLOCK + (2 * i + h) * THREADS + tid;
                const float a0 = h ? rw.Sx[i].y : rw.Sx[i].x, a1 = h ? rw.Sy[i].y : rw.Sy[i].x;
                const float a2 = h ? rw.Tx[i].y : rw.Tx[i].x, a3 = h ? rw.Ty[i].y : rw.Ty[i].x;
                if (!isfinite(a0 + a1 + a2 + a3)) bad[j] = 1u;
                unsigned long long *dst = acc + j * 4;
                atomicAdd(dst + 0, static_cast<unsigned long long>(__float2ll_rn(-a0 * colscale)));
                atomicAdd(dst + 1, static_cast<unsigned long long>(__float2ll_rn(-a1 * colscale)));
                atomicAdd(dst + 2, static_cast<unsigned long long>(__float2ll_rn(-a2 * colscale)));
                atomicAdd(dst + 3, static_cast<unsigned long long>(__float2ll_rn(-a3 * colscale)));
            }
        }
    };

    // runs of consecutive items with the same row block: rows loaded once per run, row sums flushed at its end.
    // meta[t & 1] was written before the barrier that ended item t - 1 and is rewritten only after item t's.
    int t = 0;
    while (t < s_cnt) {
        const int I = meta[t & 1][0];
        ms_load_rows(rw, rec, I, tid);
        do {
        const int buf = t & 1;
        if (tid == 0 && t + 1 < s_cnt) stage_load(s_lo + t + 1, buf ^ 1);   // tile[buf^1] was released by the
        mbar_wait(&sm.bars[buf], (t >> 1) & 1);                   // the (t/2)-th use of this buffer
        // the off-diagonal branch first: in the other order ptxas emits the diagonal loop twice
        if (meta[buf][1] != 0) {
            ms_pair_tile<VERSION>(rw, sm.tile[buf], sm.red[warp], sm.colacc[warp], lane, Bl, Cl, Dl);
            __syncthreads();
            ms_add_columns<THREADS>(sm.colacc, acc, bad, meta[buf][2], colscale, tid);
        } else {
            ms_diag_tile<VERSION>(rw, sm.tile[buf], Bl, Cl, Dl);
        }
        __syncthreads();
        ++t;
        } while (t < s_cnt && meta[t & 1][0] == I);
        flush_rows(I);
    }
}

// Exchange step of an agent-sharded crowd fused into the finalize kernel: rank g's NEXT-state arrays, mapped into this
// process over NVLink peer memory.  world == 0: no exchange.
constexpr int ML_MAX_PEERS = 16;
struct PeerPush { int world; float2 *pos[ML_MAX_PEERS]; float2 *vel[ML_MAX_PEERS]; };
// Column-direction sums of the symmetric kernel (colsum == nullptr: ordered-pair kernel, row sums only): fixed-point
// int64 accumulators per agent, value = colsum * inv_colscale.
// inbox != nullptr (agent-sharded crowd): the column-direction sums were reduced per rank and delivered to the owner
// of the rows (mlapm_sym_colpush_kernel); inbox[g * inbox_stride + local row] is rank g's share.
// slot != nullptr (culled evaluation): agent n's accumulators sit at its sorted position slot[n].  bad != nullptr: a
// flag per accumulator, set where a NaN or inf was added (fixed point has no value for them); the agent's sums then
// read NaN, as an fp32 sum would.
struct SymPartials { const long long *colsum; float inv_colscale; int nrows_pad; const float4 *inbox; int world;
                     int64_t inbox_stride; const int *slot; const unsigned *bad; };
// Owners of the 512-agent blocks (rank g owns blocks [Ib[g], Ib[g+1])) and every rank's inbox as mapped here.
struct PeerInbox { int world, rank; int Ib[ML_MAX_PEERS + 1]; float4 *inbox[ML_MAX_PEERS]; int64_t stride; };

// Agent-sharded symmetric evaluation, first half of the exchange: this rank evaluated the block pairs (I, I + d) of
// ITS row blocks I in [I0, I1); the column-direction sum of every agent m (its own or another rank's) over those block
// pairs sits in this rank's fixed-point accumulators and is stored, as fp32, into the inbox of the rank that owns m,
// over NVLink peer memory.
__global__ void mlapm_sym_colpush_kernel(const long long *__restrict__ colsum, float inv_colscale, int N,
                                         const __grid_constant__ PeerInbox peers) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m < N) {
        const int J = m / MS_BLOCK;
        const longlong2 c0 = reinterpret_cast<const longlong2 *>(colsum)[2 * m];
        const longlong2 c1 = reinterpret_cast<const longlong2 *>(colsum)[2 * m + 1];
        const double is = static_cast<double>(inv_colscale);
        const float4 u = make_float4(static_cast<float>(static_cast<double>(c0.x) * is),
                                     static_cast<float>(static_cast<double>(c0.y) * is),
                                     static_cast<float>(static_cast<double>(c1.x) * is),
                                     static_cast<float>(static_cast<double>(c1.y) * is));
        int h = 0;
        while (h + 1 < peers.world && J >= peers.Ib[h + 1]) ++h;
        peers.inbox[h][peers.rank * peers.stride + (m - peers.Ib[h] * MS_BLOCK)] = u;
    }
    __syncthreads();                                                      // one cumulative system fence per CTA:
    if (threadIdx.x == 0) __threadfence_system();                         // visible to the owner before the barrier
}

constexpr int FZ_LPR = 8;                        // lanes per row in the finalize kernel

// force = (v0*ed - v)/tau - A*R(sum partial) ; action = v + force*dt ; optional p' = p + action*dt and arrival.
__global__ void mlapm_finalize2_kernel(const float2 *__restrict__ pos, const float2 *__restrict__ vel,
                                       const float *__restrict__ ds, int ds_dim, const float2 *__restrict__ dest,
                                       int row0, int row1, int nsplit, const float4 *__restrict__ partial, float A,
                                       float cos_t, float sin_t, int version, float tau, float dt, float radius,
                                       float2 *__restrict__ action, float2 *__restrict__ pos_new,
                                       uint8_t *__restrict__ arrived, const __grid_constant__ PeerPush push,
                                       const __grid_constant__ SymPartials sym) {
    // FZ_LPR lanes share a row: lane j adds the split partials j, j + FZ_LPR, ... and the lanes' sums are combined in
    // lane order -- a fixed order (deterministic), but FZ_LPR loads in flight per row instead of one dependent chain of
    // up to 396 (an 8-way shard of 100k agents): the kernel was latency bound at 70 us of a 1.05 ms step.
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int rl_raw = gt / FZ_LPR, sub = gt % FZ_LPR;
    const int nrows = row1 - row0;
    const bool live = rl_raw < nrows;
    const int rl = live ? rl_raw : nrows - 1;                     // idle lanes shadow the last row (shuffles stay converged)
    const int64_t pstride = (sym.colsum || sym.inbox) ? sym.nrows_pad : nrows;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int q = sub; q < nsplit; q += FZ_LPR) {
        const float4 t = partial[static_cast<int64_t>(q) * pstride + rl];
        s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
    }
#pragma unroll
    for (int o = 1; o < FZ_LPR; o <<= 1) {                        // tree in a fixed shape: deterministic
        s.x += __shfl_xor_sync(0xffffffffu, s.x, o);
        s.y += __shfl_xor_sync(0xffffffffu, s.y, o);
        s.z += __shfl_xor_sync(0xffffffffu, s.z, o);
        s.w += __shfl_xor_sync(0xffffffffu, s.w, o);
    }
    const int n = row0 + rl;
    float qx = 0.f, qy = 0.f, ax = 0.f, ay = 0.f;
    if (live && sub == 0) {
    const float2 p = pos[n], v = vel[n], d = dest[n];
    const float dsx = ds[static_cast<int64_t>(n) * ds_dim];
    const float dsy = ds[static_cast<int64_t>(n) * ds_dim + (ds_dim > 1 ? 1 : 0)];
    const float2 fd = mlapm_dest_term(p, v, d, dsx, dsy, tau);
    if (sym.inbox) {
        // agent-sharded symmetric evaluation: one pre-reduced share per rank, added in rank order
        float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int g = 0; g < sym.world; ++g) {
            const float4 t = sym.inbox[g * sym.inbox_stride + rl];
            u.x += t.x; u.y += t.y; u.z += t.z; u.w += t.w;
        }
        s.x -= u.x; s.y -= u.y; s.z -= u.z; s.w -= u.w;
    } else if (sym.colsum) {
        // symmetric evaluation: this agent was a COLUMN of T/2 block pairs; their column-direction sums (exact integer
        // total of the per-pair fp32 block sums) enter with the opposite sign (vr[m,n] = -vr[n,m]).
        // culled evaluation: the row-direction sums are in the same accumulators, with the opposite sign
        const int j = sym.slot ? sym.slot[n] : n;
        const longlong2 c0 = reinterpret_cast<const longlong2 *>(sym.colsum)[2 * j];
        const longlong2 c1 = reinterpret_cast<const longlong2 *>(sym.colsum)[2 * j + 1];
        const double is = static_cast<double>(sym.inv_colscale);
        s.x -= static_cast<float>(static_cast<double>(c0.x) * is);
        s.y -= static_cast<float>(static_cast<double>(c0.y) * is);
        s.z -= static_cast<float>(static_cast<double>(c1.x) * is);
        s.w -= static_cast<float>(static_cast<double>(c1.y) * is);
        if (sym.bad && sym.bad[j]) s = make_float4(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F);
    }
    float sx, sy;
    if (version == 0) { sx = s.x; sy = s.y; }
    else {                                                        // R(sigma theta) r^ summed    (mlapm.py:35-38)
        sx = fmaf(cos_t, s.x, -(sin_t * s.w));
        sy = fmaf(sin_t, s.z, cos_t * s.y);
    }
    const float2 a = mlapm_action(v, fd, __fmul_rn(A, sx), __fmul_rn(A, sy), dt);
    ax = a.x; ay = a.y;
    if (action) action[rl] = a;
    if (pos_new || arrived || push.world > 0) {
        const float2 q = mlapm_move(p, a, dt);
        qx = q.x; qy = q.y;
        if (pos_new) pos_new[rl] = q;
        if (arrived) arrived[rl] = mlapm_arrived(q, d, radius) ? 1 : 0;
    }
    }
    if (push.world > 0) {
        // the path's one exchange, fused: the row's new state goes into EVERY rank's next-state arrays; the row's
        // FZ_LPR lanes take one peer each, so the remote stores of a row are issued in parallel
        const int lead = (threadIdx.x & 31) & ~(FZ_LPR - 1);
        qx = __shfl_sync(0xffffffffu, qx, lead); qy = __shfl_sync(0xffffffffu, qy, lead);
        ax = __shfl_sync(0xffffffffu, ax, lead); ay = __shfl_sync(0xffffffffu, ay, lead);
        if (live)
            for (int g = sub; g < push.world; g += FZ_LPR) {
                push.pos[g][n] = make_float2(qx, qy);
                push.vel[g][n] = make_float2(ax, ay);
            }
        // one system-scope fence per CTA (fences are cumulative over the CTA barrier): the stores are visible to the
        // peers before the step barrier that follows the kernel
        __syncthreads();
        if (threadIdx.x == 0) __threadfence_system();
    }
}

// =====================================================================================================================
// Many independent scenes in one launch (piml_mlapm_scenes_advance_f32).  Layout padded (S, N): a scene's active slots
// are its agents, the inactive ones take part in nothing.
//
// One thread owns one row and sums its scene's active columns in ascending slot order (pair_fast / pair_exact), so a
// scene's result does not depend on the batch, on S or on the launch shape.  A "chunk" is C lanes of one scene:
//   N <= 32    C = the power of two >= N, 256 / C scenes per CTA (8 scenes of 32 lanes ... 256 of 1)
//   N <= 256   C = N rounded up to whole warps, floor(256 / C) scenes per CTA
//   N  > 256   the rows split over ceil(N / 256) CTAs of C <= 256 lanes each (balanced, whole warps)
// Every CTA stages the columns of its scenes (position, velocity: TMA bulk copies where 16 B aligned, like the dense
// kernel's tiles; activity flags) and their constants in shared memory: 17 B per column, 139 KB at N = 8192.
// =====================================================================================================================
constexpr int MSC_THREADS = 256;
static_assert(PIML_MLAPM_SCENES_MAX_N * 17 + 1024 <= 227 * 1024, "mlapm_scenes_kernel: columns exceed shared memory");

struct MscShape { int C, k, nchunk; };       // lanes per chunk, scenes per CTA, chunks (CTAs) per scene
struct MscSmem { int pv, cst, act, total; }; // byte offsets: positions + velocities, constants, flags; total

static MscShape msc_shape(int N) {
    MscShape sh;
    sh.nchunk = (N + MSC_THREADS - 1) / MSC_THREADS;
    if (N <= 32) {
        sh.C = 1;
        while (sh.C < N) sh.C *= 2;
    } else {
        const int rows = (N + sh.nchunk - 1) / sh.nchunk;
        sh.C = (rows + 31) / 32 * 32;
    }
    sh.k = sh.nchunk == 1 ? MSC_THREADS / sh.C : 1;
    return sh;
}

__host__ __device__ __forceinline__ MscSmem msc_smem(int ncol, int k) {
    MscSmem m;
    m.pv = 16;                                                    // after the mbarrier
    const int pv_bytes = (ncol + 1) / 2 * 16;                     // each array a whole number of 16 B
    m.cst = m.pv + 2 * pv_bytes;
    m.act = m.cst + k * static_cast<int>(sizeof(MlConst));
    m.total = m.act + ncol;
    return m;
}

template <int VERSION, bool EXACT>
__global__ void __launch_bounds__(MSC_THREADS) mlapm_scenes_kernel(
    const float2 *__restrict__ pos, const float2 *__restrict__ vel, const float *__restrict__ ds, int ds_dim,
    const float2 *__restrict__ dest, const uint8_t *__restrict__ active, int S, int N, MscShape sh, MlConst k0,
    const float *__restrict__ scene_params, float dt, float radius, float2 *__restrict__ action,
    float2 *__restrict__ pos_new, uint8_t *__restrict__ arrived) {
    extern __shared__ __align__(128) unsigned char msc_raw[];
    const int group = blockIdx.x / sh.nchunk, chunk = blockIdx.x % sh.nchunk;
    const int s0 = group * sh.k;
    const int ks = min(sh.k, S - s0);                             // scenes this CTA holds
    const int ncol = ks * N;
    const MscSmem lay = msc_smem(ncol, sh.k);
    uint64_t *bar = reinterpret_cast<uint64_t *>(msc_raw);
    float2 *sp = reinterpret_cast<float2 *>(msc_raw + lay.pv);
    float2 *sv = sp + (ncol + 1) / 2 * 2;
    MlConst *sk = reinterpret_cast<MlConst *>(msc_raw + lay.cst);
    uint8_t *sa = msc_raw + lay.act;
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    const int64_t base = static_cast<int64_t>(s0) * N;
    const bool tma = stage_tile_pv(sp, sv, pos + base, vel + base, ncol, bar);
    for (int i = threadIdx.x; i < ncol; i += blockDim.x) sa[i] = active[base + i];
    if (static_cast<int>(threadIdx.x) < ks) {
        MlConst c = k0;
        if (scene_params) {
            const float *q = scene_params + 6 * static_cast<int64_t>(s0 + threadIdx.x);
            c = mlapm_derive(VERSION, q[0], q[1], q[2], q[3], q[4], q[5]);
        }
        sk[threadIdx.x] = c;
    }
    if (tma) mbar_wait(bar, 0);
    __syncthreads();

    const int ls = threadIdx.x / sh.C, row = chunk * sh.C + threadIdx.x % sh.C;
    if (ls >= ks || row >= N) return;
    const int c0 = ls * N;
    const int64_t n = base + c0 + row;
    if (!sa[c0 + row]) {
        action[n] = make_float2(CUDART_NAN_F, CUDART_NAN_F);
        pos_new[n] = make_float2(CUDART_NAN_F, CUDART_NAN_F);
        arrived[n] = 0;
        return;
    }
    const MlConst k = sk[ls];
    const float2 p = sp[c0 + row], v = sv[c0 + row], d = dest[n];
    const float2 e = mlapm_dest_dir(p, d);
    float fx = 0.f, fy = 0.f;
    const float2 *cp = sp + c0, *cv = sv + c0;
    const uint8_t *ca = sa + c0;
#pragma unroll 4
    for (int j = 0; j < N; ++j) {
        if (!ca[j]) continue;
        if (EXACT) pair_exact<VERSION>(p.x, p.y, v.x, v.y, e.x, e.y, cp[j], cv[j], k, fx, fy);
        else pair_fast<VERSION>(p.x, p.y, v.x, v.y, e.x, e.y, cp[j], cv[j], k, fx, fy);
    }
    const float dsx = ds[n * ds_dim];
    const float dsy = ds[n * ds_dim + (ds_dim > 1 ? 1 : 0)];
    const float2 a = mlapm_action(v, mlapm_dest_term(p, v, d, dsx, dsy, k.tau), fx, fy, dt);
    const float2 q = mlapm_move(p, a, dt);
    action[n] = a;
    pos_new[n] = q;
    arrived[n] = mlapm_arrived(q, d, radius) ? 1 : 0;
}

constexpr int ML_MAX_SPLIT = 64;

static int pick_rows_per_thread(int64_t nrows) { return nrows >= 4096 ? 4 : (nrows >= 1024 ? 2 : 1); }

// Row pairs per thread of the packed kernel (2*RP rows per thread).
// 4 rows per thread (RP = 2) is ~0.5 % faster per pair, but halves the CTA count: with few row blocks (an 8-way
// shard of 100k agents has 25) the last wave is mostly idle, so small grids use 2 rows per thread.  Does not change
// any result (each row's column order is the same).
static int pick_row_pairs(int64_t nrows, int64_t N) {
    const int64_t tiles = (N + 511) / 512;
    const int64_t nsplit = tiles < 64 ? tiles : 64;
    const int64_t ctas2 = ((nrows + 511) / 512) * nsplit;
    return (nrows >= 8192 && ctas2 >= 10LL * 4 * sm_count()) ? 2 : 1;   // measured: 12.5k..50k rows of 100k prefer 1
}

// Column splits: enough CTAs for ~8 waves over the SMs, each split a multiple of `tile` columns.
static void pick_split(int64_t nrows, int64_t N, int rows_per_cta, int tile, int *nsplit, int *cols_per_split) {
    const int64_t row_blocks = (nrows + rows_per_cta - 1) / rows_per_cta;
    const int64_t want_ctas = 8LL * 6 * sm_count();
    int64_t s = (want_ctas + row_blocks - 1) / row_blocks;
    const int64_t max_by_cols = (N + tile - 1) / tile;
    if (s > max_by_cols) s = max_by_cols;
    if (s > ML_MAX_SPLIT) s = ML_MAX_SPLIT;
    if (s < 1) s = 1;
    int64_t cps = (N + s - 1) / s;
    cps = (cps + tile - 1) / tile * tile;
    *cols_per_split = static_cast<int>(cps);
    *nsplit = static_cast<int>((N + cps - 1) / cps);
}

// Column splits for the packed kernel, each a whole number of tiles: one tile per split up to ML_MAX_SPLIT.  Measured
// at N = 100k (profiles/r01_mlapm_experiments.md): 27-36 splits (6-8 waves) are ~2% faster than the exact 2- or 4-wave
// fits (9, 18), 4 splits (1 wave) 18% slower.
// The column partition depends on N ONLY: a row's sum is then evaluated in the same order whichever row range (rank) it
// is computed in, so an agent-sharded crowd is bit-identical to the unsharded one (SURVEY.md A.2b).  As many splits as
// allowed also gives every rank of an 8-way shard enough CTAs to fill its GPU.
static void pick_split2(int64_t N, int *nsplit, int *cols_per_split) {
    const int64_t tiles = (N + M2_TILE - 1) / M2_TILE;
    int64_t s = tiles < ML_MAX_SPLIT ? tiles : ML_MAX_SPLIT;
    if (s < 1) s = 1;
    const int64_t per = (tiles + s - 1) / s;
    *cols_per_split = static_cast<int>(per * M2_TILE);
    *nsplit = static_cast<int>((tiles + per - 1) / per);
}

template <int VERSION, bool EXACT>
static void launch_pairs(int R, dim3 grid, cudaStream_t st, const float2 *pos, const float2 *vel, const float2 *dest,
                         int N, int row0, int row1, int cps, const MlConst &k, float2 *partial) {
    if (R == 4)
        mlapm_pairs_kernel<VERSION, 4, EXACT><<<grid, ML_THREADS, 0, st>>>(pos, vel, dest, N, row0, row1, cps, k, partial);
    else if (R == 2)
        mlapm_pairs_kernel<VERSION, 2, EXACT><<<grid, ML_THREADS, 0, st>>>(pos, vel, dest, N, row0, row1, cps, k, partial);
    else
        mlapm_pairs_kernel<VERSION, 1, EXACT><<<grid, ML_THREADS, 0, st>>>(pos, vel, dest, N, row0, row1, cps, k, partial);
}

template <int VERSION>
static void launch_pairs2(int RP, dim3 grid, cudaStream_t st, const float2 *pos, const float2 *vel, const float2 *dest,
                          const float4 *col8, int N, int row0, int row1, int cps, const M2Const &k, float4 *partial) {
    if (RP == 2)
        mlapm_pairs2_kernel<VERSION, 2><<<grid, M2_THREADS, 0, st>>>(pos, vel, dest, col8, N, row0, row1, cps, k, partial);
    else
        mlapm_pairs2_kernel<VERSION, 1><<<grid, M2_THREADS, 0, st>>>(pos, vel, dest, col8, N, row0, row1, cps, k, partial);
}

}  // namespace piml

using namespace piml;

// ---- symmetric evaluation: selection and workspace ------------------------------------------------------------------
static int g_mlapm_algorithm = 0;                 // 0 automatic, 1 ordered pairs (v2), 2 symmetric culled, 3 dense
constexpr int64_t MS_AUTO_MIN_AGENTS = 16384;     // below this the ordered-pair kernel fills the GPU better

static int64_t sym_blocks(int64_t N) { return (N + MS_BLOCK - 1) / MS_BLOCK; }
// Block pairs per CTA for nI row blocks of a crowd of T blocks: >= 64 CTAs per SM (measured best at N = 100k on one
// GPU: 2; an 8-way shard of the same crowd gets 1).
static int sym_per(int64_t nI, int64_t T) {
    const int64_t pairs = nI * (T / 2 + 1), want = 64LL * sm_count();
    const int64_t per = pairs / want;
    return per < 1 ? 1 : static_cast<int>(per);
}
// CTAs per block pair (1, 2 or 4 = the 4 column stages of a pair split over that many CTAs): a shard with few row
// blocks (8 ranks at N = 100k: 25 blocks x 99 pairs) would otherwise run ~2 waves of CTAs with a nearly empty last one.
static int sym_sub(int64_t nI, int64_t T, int per) {
    const int64_t ctas = nI * ((T / 2 + 1 + per - 1) / per), wave = 8LL * sm_count();
    int sub = 1;
    while (sub < MS_BLOCK / MS_CT && ctas * sub < 6 * wave) sub *= 2;
    return sub;
}
// Row-partial splits of a launch over nI row blocks: (groups of `per` block pairs) x sub.
static int sym_splits(int64_t nI, int64_t T, int *per, int *sub) {
    *per = sym_per(nI, T);
    *sub = sym_sub(nI, T, *per);
    return static_cast<int>((T / 2 + 1 + *per - 1) / *per) * *sub;
}

// Consecutive 256-byte aligned regions of a workspace; base == nullptr only adds up their sizes.
struct WsCarve {
    char *base;
    int64_t off;
    void *take(int64_t bytes) {
        char *q = base ? base + off : nullptr;
        off += (bytes + 255) / 256 * 256;
        return q;
    }
};
// The caller's workspace rounded up to 256 bytes (every layout's total has room for it).
static void *ws_align(const void *ws) {
    return reinterpret_cast<void *>((reinterpret_cast<uintptr_t>(ws) + 255) & ~static_cast<uintptr_t>(255));
}

// Dense symmetric evaluation (mlapm_sym_kernel) of a crowd split over `world` ranks (1: the whole crowd): records (32 B
// per agent), the row-direction partials of the largest shard (16 B per row and split, so that every rank's layout is
// the same), column-direction fixed-point accumulators (4 x int64 per agent) and poison flags: O(N) -- 0.15 GB at
// N = 10^6 (the per-pair column partials this replaces: 15.6 GB).
struct SymLayout { int per, sub, S; float4 *rec, *partialR; long long *colsum; unsigned *bad; int64_t total; };
static SymLayout sym_layout(int64_t N, int world, void *base) {
    const int64_t T = sym_blocks(N), npad = T * MS_BLOCK, nI = (T + world - 1) / world;
    SymLayout l{};
    l.S = sym_splits(nI, T, &l.per, &l.sub);
    WsCarve c{static_cast<char *>(base), 0};
    l.rec = static_cast<float4 *>(c.take(npad * MS_RECF * sizeof(float)));
    l.partialR = static_cast<float4 *>(c.take(l.S * nI * MS_BLOCK * sizeof(float4)));
    l.colsum = static_cast<long long *>(c.take(npad * 4 * sizeof(long long)));
    l.bad = static_cast<unsigned *>(c.take(npad * sizeof(unsigned)));
    l.total = c.off + 256;                                        // + 256: room to align the caller's base
    return l;
}

// Culled symmetric evaluation (mlapm_sym_list_kernel).  Candidates of the work list: T * (floor(T/2) + 1) * MC_SPB,
// the dense worst case (every item within r_cut); the list index is an int.
static int64_t cull_candidates(int64_t N) {
    const int64_t T = sym_blocks(N);
    return T * (T / 2 + 1) * MC_SPB;
}
// Reserved CUB scratch, computable without a device (CUB's own size query needs one).  Radix sort on DoubleBuffers
// (onesweep): 4 passes x 256 bins of 8 B, and 256 look-back counters of 4 B per tile of >= 256 keys -- at most 4 B
// per key.  Select: one 16 B tile descriptor per tile of >= 128 candidates -- at most 1 B per candidate.  64 KB for
// the counters, padding and alignment of both.  The real size is checked against this at every call.
static int64_t cull_cub_bound(int64_t N) {
    const int64_t a = 4 * N, b = cull_candidates(N);
    return (int64_t{1} << 16) + (a > b ? a : b);
}
struct CullLayout {
    float4 *rec; long long *acc; unsigned *bad; uint32_t *key[2]; int *val[2]; int *slot;
    float4 *sbox, *bbox; unsigned *sflag, *bflag; int *items, *nitems; void *temp; int64_t temp_bytes, total;
};
// records, accumulators (4 x int64) and flags per padded agent; keys, values (both double-buffered) and slots per
// agent; boxes and flags per stage and block; the work list; CUB's scratch.  0.1 GB at N = 10^6.
static CullLayout cull_layout(int64_t N, void *base) {
    const int64_t T = sym_blocks(N), npad = T * MS_BLOCK;
    CullLayout l{};
    WsCarve c{static_cast<char *>(base), 0};
    l.rec = static_cast<float4 *>(c.take(npad * MS_RECF * sizeof(float)));
    l.acc = static_cast<long long *>(c.take(npad * 4 * sizeof(long long)));
    l.bad = static_cast<unsigned *>(c.take(npad * sizeof(unsigned)));
    for (int b = 0; b < 2; ++b) {
        l.key[b] = static_cast<uint32_t *>(c.take(N * sizeof(uint32_t)));
        l.val[b] = static_cast<int *>(c.take(N * sizeof(int)));
    }
    l.slot = static_cast<int *>(c.take(N * sizeof(int)));
    l.sbox = static_cast<float4 *>(c.take(T * MC_SPB * sizeof(float4)));
    l.bbox = static_cast<float4 *>(c.take(T * sizeof(float4)));
    l.sflag = static_cast<unsigned *>(c.take(T * MC_SPB * sizeof(unsigned)));
    l.bflag = static_cast<unsigned *>(c.take(T * sizeof(unsigned)));
    l.items = static_cast<int *>(c.take(cull_candidates(N) * sizeof(int)));
    l.nitems = static_cast<int *>(c.take(sizeof(int)));
    l.temp_bytes = cull_cub_bound(N);
    l.temp = c.take(l.temp_bytes);
    l.total = c.off + 256;                                          // + 256: room to align the caller's base
    return l;
}
static int64_t cull_workspace_bytes(int64_t N) { return cull_layout(N, nullptr).total; }

// Fixed-point scale 2^s of the column accumulators: one pair contributes |w r| = exp(arg) <= exp(|C|) (B r + D r cos <= 0
// is required by sym_params_ok), a column at most N of them; keep two bits of headroom below 2^63.
static int sym_colscale_log2(int64_t N, const piml_mlapm_params *prm) {
    const double c = prm->version == 0 ? 0.0 : fabs(static_cast<double>(prm->C));
    const double bound = static_cast<double>(N) * exp(c);
    return 61 - static_cast<int>(ceil(log2(bound > 1.0 ? bound : 1.0)));
}

extern "C" int piml_set_mlapm_algorithm(int algo) {
    PIML_REQUIRE(algo >= 0 && algo <= 3,
                 "piml_set_mlapm_algorithm: 0 = automatic, 1 = ordered pairs, 2 = symmetric (unordered pairs, culled "
                 "at the radius where the weight is exactly 0), 3 = symmetric, dense (no culling)");
    g_mlapm_algorithm = algo;
    return PIML_OK;
}

extern "C" int64_t piml_mlapm_workspace_bytes_sym(int64_t N) {
    if (N <= 0) return 0;
    const int64_t a = piml_mlapm_workspace_bytes(N), b = sym_layout(N, 1, nullptr).total, c = cull_workspace_bytes(N);
    return a > b ? (a > c ? a : c) : (b > c ? b : c);
}

extern "C" int piml_mlapm_cull_items(const void *workspace, int64_t N, int64_t *items) {
    PIML_REQUIRE(workspace && items && N > 0 && N < (1LL << 31), "piml_mlapm_cull_items: bad arguments");
    const CullLayout l = cull_layout(N, ws_align(workspace));
    int n = 0;
    PIML_CUDA(cudaMemcpy(&n, l.nitems, sizeof(int), cudaMemcpyDeviceToHost));
    *items = n;
    return PIML_OK;
}

extern "C" int64_t piml_mlapm_workspace_bytes(int64_t N) {
    if (N < 0) return 0;
    // column records (32 B per agent, padded to a tile) + per-split partial sums (16 B per row and split)
    const int64_t npad = (N + M2_TILE - 1) / M2_TILE * M2_TILE;
    return npad * M2_COLF * sizeof(float) + static_cast<int64_t>(ML_MAX_SPLIT) * N * 4 * sizeof(float) + 256;
}

static MlConst mlapm_consts(const piml_mlapm_params *prm) {
    return mlapm_derive(prm->version, prm->tau, prm->A, prm->B, prm->C, prm->D, prm->theta_deg);
}

// The padding agents of the symmetric kernel need a weight that underflows to 0 at large r.
static bool sym_params_ok(const piml_mlapm_params *prm, const MlConst &k, int64_t N) {
    return !prm->exact_math && (prm->version == 0 ? k.Bl < 0.f : k.Bl + fabsf(k.Dl) < 0.f) &&
           sym_colscale_log2(N, prm) >= 30;                        // 2^-30 resolution at the very least (|C| < ~15)
}

// Distance beyond which every pair's production weight is exactly +0 (see mlapm_sym_list_kernel): arg <= (Bl + |Dl|) r
// + |Cl| < -127 (raw: Bl r < -127), from the same fp32 constants the kernels use.  The margin (1 % + 0.01 m) covers
// the rsqrt.approx error in r and q and fp32 rounding of coordinates; ex2.approx.ftz already returns 0 below -126.
// +inf (no culling) where the symmetric kernels do not run.
static float cull_radius(const piml_mlapm_params *prm, const MlConst &k) {
    if (prm->exact_math) return HUGE_VALF;
    const double slope = prm->version == 0 ? static_cast<double>(k.Bl)
                                           : static_cast<double>(k.Bl) + fabs(static_cast<double>(k.Dl));
    if (!(slope < 0.0)) return HUGE_VALF;
    const double c = prm->version == 0 ? 0.0 : fabs(static_cast<double>(k.Cl));
    const double r0 = (127.0 + c) / -slope;
    return static_cast<float>(r0 * 1.01 + 0.01);
}

extern "C" float piml_mlapm_cull_radius(const piml_mlapm_params *prm) {
    if (!prm || (prm->version != 0 && prm->version != 1)) return HUGE_VALF;
    return cull_radius(prm, mlapm_consts(prm));
}

// prep + symmetric pair kernel for the row blocks [I0, I0 + nI) of a crowd of T blocks, in workspace l; bad: the NaN
// flags, or null.
static int launch_sym_pairs(int version, const float2 *p2, const float2 *v2, const float2 *d2, int N, int64_t T,
                            int64_t I0, int64_t nI, const SymLayout &l, const MlConst &k, float colscale,
                            unsigned *bad, cudaStream_t st) {
    const int64_t npad = T * MS_BLOCK;
    const int threads = 256;
    mlapm_prep_sym_kernel<<<static_cast<unsigned>((npad + threads - 1) / threads), threads, 0, st>>>(
        p2, v2, d2, N, static_cast<int>(npad), l.rec, reinterpret_cast<ulonglong2 *>(l.colsum), bad);
    count_launch();
    int rc = check_launch("mlapm_prep_sym_kernel");
    if (rc) return rc;
    const M2Const k2{k.Bl, k.Cl, k.Dl};
    const dim3 grid(static_cast<unsigned>(nI), static_cast<unsigned>(l.S));
    const int iT = static_cast<int>(T), iI0 = static_cast<int>(I0), nrows_pad = static_cast<int>(nI * MS_BLOCK);
    unsigned long long *colsum = reinterpret_cast<unsigned long long *>(l.colsum);
    static_assert(sizeof(MsSmem<MS_BLOCK / 4>) <= 48 * 1024 && sizeof(MsSmem<MS_BLOCK / 8>) <= 48 * 1024,
                  "mlapm_sym_kernel: shared memory above the default limit");
    // measured at N = 100k (ms per step): 8 rows per thread (64 threads) 6.81, 4 rows (128 threads) 6.99, 2 rows 7.16
    if (version == 0)
        mlapm_sym_kernel<0, 2><<<grid, MS_BLOCK / 4, sizeof(MsSmem<MS_BLOCK / 4>), st>>>(
            l.rec, iT, iT / 2, iI0, l.per, l.sub, k2, l.partialR, nrows_pad, colsum, colscale, bad);
    else
        mlapm_sym_kernel<1, 4><<<grid, MS_BLOCK / 8, sizeof(MsSmem<MS_BLOCK / 8>), st>>>(
            l.rec, iT, iT / 2, iI0, l.per, l.sub, k2, l.partialR, nrows_pad, colsum, colscale, bad);
    count_launch();
    return check_launch("mlapm_sym_kernel");
}

// Launches of one CUB radix sort of n 32-bit keys with int values on DoubleBuffers (CUB 2.x, sm_100 policy): one
// single-tile kernel up to 256 x 19 keys, else histogram + exclusive sum + one onesweep kernel per 8-bit digit.
static int cub_sort_launches(int64_t n, int bits) { return n <= 256 * 19 ? 1 : 2 + (bits + 7) / 8; }

// Culled symmetric evaluation of the whole crowd: keys, sort, prep + boxes, work list, pair kernel.  The finalize
// kernel follows in the caller.  No host synchronisation: the list length stays on the device.
static int launch_sym_culled(int version, const float2 *p2, const float2 *v2, const float2 *d2, int N,
                             const MlConst &k, float rc, const CullLayout &l, float colscale, cudaStream_t st) {
    const int64_t T = sym_blocks(N), D = T / 2;
    const int threads = 256;
    mlapm_cull_keys_kernel<<<static_cast<unsigned>((N + threads - 1) / threads), threads, 0, st>>>(p2, N, l.key[0],
                                                                                                     l.val[0]);
    count_launch();
    int rc_ = check_launch("mlapm_cull_keys_kernel");
    if (rc_) return rc_;
    cub::DoubleBuffer<uint32_t> keys(l.key[0], l.key[1]);
    cub::DoubleBuffer<int> vals(l.val[0], l.val[1]);
    size_t need = 0;
    PIML_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, need, keys, vals, N, 0, 32, st));
    PIML_REQUIRE(static_cast<int64_t>(need) <= l.temp_bytes,
                 "piml_mlapm: CUB radix sort needs %lld bytes of scratch, %lld reserved", static_cast<long long>(need),
                 static_cast<long long>(l.temp_bytes));
    size_t temp_bytes = static_cast<size_t>(l.temp_bytes);
    PIML_CUDA(cub::DeviceRadixSort::SortPairs(l.temp, temp_bytes, keys, vals, N, 0, 32, st));
    count_launch(cub_sort_launches(N, 32));
    mlapm_prep_cull_kernel<<<static_cast<unsigned>(T), MS_BLOCK, 0, st>>>(
        p2, v2, d2, vals.Current(), N, l.rec, l.slot, reinterpret_cast<ulonglong2 *>(l.acc), l.bad, l.sbox, l.sflag,
        l.bbox, l.bflag);
    count_launch();
    rc_ = check_launch("mlapm_prep_cull_kernel");
    if (rc_) return rc_;
    const CullKeep keep{l.sbox, l.bbox, l.sflag, l.bflag, static_cast<int>(T), static_cast<int>(D), rc};
    const int ncand = static_cast<int>(cull_candidates(N));
    cub::CountingInputIterator<int> cand(0);
    need = 0;
    PIML_CUDA(cub::DeviceSelect::If(nullptr, need, cand, l.items, l.nitems, ncand, keep, st));
    PIML_REQUIRE(static_cast<int64_t>(need) <= l.temp_bytes,
                 "piml_mlapm: CUB select needs %lld bytes of scratch, %lld reserved", static_cast<long long>(need),
                 static_cast<long long>(l.temp_bytes));
    temp_bytes = static_cast<size_t>(l.temp_bytes);
    PIML_CUDA(cub::DeviceSelect::If(l.temp, temp_bytes, cand, l.items, l.nitems, ncand, keep, st));
    count_launch(2);                                              // tile-state init + select
    using Smem = MsSmem<MC_THREADS>;
    static_assert(sizeof(Smem) <= 48 * 1024, "mlapm_sym_list_kernel: shared memory above the default limit");
    const void *kfn = version == 0 ? reinterpret_cast<const void *>(&mlapm_sym_list_kernel<0>)
                                   : reinterpret_cast<const void *>(&mlapm_sym_list_kernel<1>);
    static const void *cached_fn = nullptr;
    static int cached_occ = 0;
    if (kfn != cached_fn) {
        int occ = 0;
        PIML_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kfn, MC_THREADS, sizeof(Smem)));
        cached_occ = occ < 1 ? 1 : occ;
        cached_fn = kfn;
    }
    // persistent grid: one CTA per resident slot, capped by the largest list (it can never have more items)
    int64_t grid = static_cast<int64_t>(cached_occ) * sm_count();
    if (grid > ncand) grid = ncand;
    M2Const k2{k.Bl, k.Cl, k.Dl};
    unsigned long long *acc = reinterpret_cast<unsigned long long *>(l.acc);
    if (version == 0)
        mlapm_sym_list_kernel<0><<<static_cast<unsigned>(grid), MC_THREADS, sizeof(Smem), st>>>(
            l.rec, l.items, l.nitems, static_cast<int>(T), static_cast<int>(D), k2, acc, l.bad, colscale);
    else
        mlapm_sym_list_kernel<1><<<static_cast<unsigned>(grid), MC_THREADS, sizeof(Smem), st>>>(
            l.rec, l.items, l.nitems, static_cast<int>(T), static_cast<int>(D), k2, acc, l.bad, colscale);
    count_launch();
    return check_launch("mlapm_sym_list_kernel");
}

static int mlapm_advance_impl(const float *pos, const float *vel, const float *desired_speed, int ds_dim,
                              const float *dest, int64_t N, int64_t row0, int64_t row1, const piml_mlapm_params *prm,
                              float dt, float radius, float *action, float *pos_new, uint8_t *arrived, void *workspace,
                              int64_t workspace_bytes, const PeerPush &push, void *stream) {
    if (N == 0) return PIML_OK;                                    // empty crowd: nothing to do, pointers may be null
    PIML_REQUIRE(pos && vel && desired_speed && dest && prm && (action || push.world > 0) && workspace,
                 "piml_mlapm: null pointer");
    PIML_REQUIRE(ds_dim == 1 || ds_dim == 2, "piml_mlapm: desired_speed must be (N,1) or (N,2), got ds_dim=%d", ds_dim);
    PIML_REQUIRE(N >= 0 && N < (1LL << 31), "piml_mlapm: N=%lld out of range", static_cast<long long>(N));
    PIML_REQUIRE(0 <= row0 && row0 <= row1 && row1 <= N, "piml_mlapm: bad row range [%lld,%lld) for N=%lld",
                 static_cast<long long>(row0), static_cast<long long>(row1), static_cast<long long>(N));
    PIML_REQUIRE(prm->version == 0 || prm->version == 1,
                 "piml_mlapm: version %d unsupported (0='raw', 1='GC'; 'UCY' is not runnable in the reference)",
                 prm->version);
    PIML_REQUIRE((reinterpret_cast<uintptr_t>(pos) & 7u) == 0 && (reinterpret_cast<uintptr_t>(vel) & 7u) == 0 &&
                     (reinterpret_cast<uintptr_t>(dest) & 7u) == 0 && (reinterpret_cast<uintptr_t>(action) & 7u) == 0,
                 "piml_mlapm: pointers must be 8-byte aligned");
    const int64_t nrows = row1 - row0;
    if (nrows == 0) return PIML_OK;

    const MlConst k = mlapm_consts(prm);

    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float2 *p2 = reinterpret_cast<const float2 *>(pos), *v2 = reinterpret_cast<const float2 *>(vel);
    const float2 *d2 = reinterpret_cast<const float2 *>(dest);
    const int iN = static_cast<int>(N), r0 = static_cast<int>(row0), r1 = static_cast<int>(row1);
    int rc;
    if (prm->exact_math) {
        PIML_REQUIRE(push.world == 0, "piml_mlapm: the fused exchange is only available on the production math path");
        // validation variant: IEEE arithmetic in the reference's operation order
        const int R = pick_rows_per_thread(nrows);
        int nsplit, cps;
        pick_split(nrows, N, ML_THREADS * R, ML_TILE, &nsplit, &cps);
        dim3 grid(static_cast<unsigned>((nrows + ML_THREADS * R - 1) / (ML_THREADS * R)),
                  static_cast<unsigned>(nsplit));
        float2 *partial = reinterpret_cast<float2 *>(workspace);
        if (prm->version == 0) launch_pairs<0, true>(R, grid, st, p2, v2, d2, iN, r0, r1, cps, k, partial);
        else launch_pairs<1, true>(R, grid, st, p2, v2, d2, iN, r0, r1, cps, k, partial);
        count_launch();
        rc = check_launch("mlapm_pairs_kernel");
        if (rc) return rc;
        const int threads = 256;
        mlapm_finalize_kernel<<<static_cast<unsigned>((nrows + threads - 1) / threads), threads, 0, st>>>(
            p2, v2, desired_speed, ds_dim, d2, r0, r1, nsplit, partial, prm->tau, dt, radius,
            reinterpret_cast<float2 *>(action), reinterpret_cast<float2 *>(pos_new), arrived);
        count_launch();
        return check_launch("mlapm_finalize_kernel");
    }
    // production, whole crowd: symmetric evaluation (every unordered pair once) when the caller's workspace holds
    // the column-direction sums; row ranges (agent-sharded ranks) and small crowds use the ordered-pair kernel.
    int nsplit = 0;                                                // row-direction partials of the finalize kernel
    const float4 *partial = nullptr;
    SymPartials symp{nullptr, 0.f, 0, nullptr, 0, 0, nullptr, nullptr};
    const bool sym_ok = row0 == 0 && row1 == N && sym_params_ok(prm, k, N);
    const bool want_sym = g_mlapm_algorithm >= 2 || (g_mlapm_algorithm == 0 && N >= MS_AUTO_MIN_AGENTS);
    if (sym_ok && want_sym && g_mlapm_algorithm != 3 && workspace_bytes >= cull_workspace_bytes(N) &&
        cull_candidates(N) < (int64_t{1} << 31)) {
        // culled (0, 2): skips the work beyond the radius where the weight is exactly 0; the list index is an int
        const CullLayout l = cull_layout(N, ws_align(workspace));
        const int sl = sym_colscale_log2(N, prm);
        rc = launch_sym_culled(prm->version, p2, v2, d2, iN, k, cull_radius(prm, k), l, ldexpf(1.0f, sl), st);
        if (rc) return rc;
        symp = SymPartials{l.acc, ldexpf(1.0f, -sl), 0, nullptr, 0, 0, l.slot, l.bad};
    } else if (sym_ok && want_sym && workspace_bytes >= sym_layout(N, 1, nullptr).total) {
        // dense (3, or a workspace without room for the culled path's list)
        const int64_t T = sym_blocks(N);
        const SymLayout l = sym_layout(N, 1, ws_align(workspace));
        const int sl = sym_colscale_log2(N, prm);
        rc = launch_sym_pairs(prm->version, p2, v2, d2, iN, T, 0, T, l, k, ldexpf(1.0f, sl), l.bad, st);
        if (rc) return rc;
        nsplit = l.S;
        partial = l.partialR;
        symp = SymPartials{l.colsum, ldexpf(1.0f, -sl), static_cast<int>(T * MS_BLOCK), nullptr, 0, 0, nullptr, l.bad};
    } else {
        // ordered pairs: packed-FP32 kernel on 16 B column records
        const int64_t npad = (N + M2_TILE - 1) / M2_TILE * M2_TILE;
        float4 *col8 = reinterpret_cast<float4 *>(workspace);
        float4 *partial4 = col8 + npad;
        const int threads = 256;
        mlapm_prep_kernel<<<static_cast<unsigned>((npad + threads - 1) / threads), threads, 0, st>>>(
            p2, v2, iN, static_cast<int>(npad), col8);
        count_launch();
        rc = check_launch("mlapm_prep_kernel");
        if (rc) return rc;
        const int RP = pick_row_pairs(nrows, N);
        int cps;
        pick_split2(N, &nsplit, &cps);
        const dim3 grid(static_cast<unsigned>((nrows + M2_THREADS * 2 * RP - 1) / (M2_THREADS * 2 * RP)),
                        static_cast<unsigned>(nsplit));
        const M2Const k2{k.Bl, k.Cl, k.Dl};
        if (prm->version == 0) launch_pairs2<0>(RP, grid, st, p2, v2, d2, col8, iN, r0, r1, cps, k2, partial4);
        else launch_pairs2<1>(RP, grid, st, p2, v2, d2, col8, iN, r0, r1, cps, k2, partial4);
        count_launch();
        rc = check_launch("mlapm_pairs2_kernel");
        if (rc) return rc;
        partial = partial4;
    }
    const int threads = 256;
    mlapm_finalize2_kernel<<<static_cast<unsigned>((nrows * FZ_LPR + threads - 1) / threads), threads, 0, st>>>(
        p2, v2, desired_speed, ds_dim, d2, r0, r1, nsplit, partial, prm->A, k.cos_t, k.sin_t, prm->version, prm->tau,
        dt, radius, reinterpret_cast<float2 *>(action), reinterpret_cast<float2 *>(pos_new), arrived, push, symp);
    count_launch();
    return check_launch("mlapm_finalize2_kernel");
}

extern "C" int piml_mlapm_scenes_advance_f32(const float *pos, const float *vel, const float *desired_speed,
                                             int ds_dim, const float *dest, const uint8_t *active, int64_t S,
                                             int64_t N, const piml_mlapm_params *prm, const float *scene_params,
                                             float dt, float radius, float *action, float *pos_new, uint8_t *arrived,
                                             void *stream) {
    PIML_REQUIRE(pos && vel && desired_speed && dest && active && prm && action && pos_new && arrived,
                 "piml_mlapm_scenes_advance_f32: null pointer");
    PIML_REQUIRE(S >= 1 && N >= 1 && S * N < (int64_t{1} << 31),
                 "piml_mlapm_scenes_advance_f32: S=%lld, N=%lld out of range (S, N >= 1, S*N < 2^31)",
                 static_cast<long long>(S), static_cast<long long>(N));
    PIML_REQUIRE(N <= PIML_MLAPM_SCENES_MAX_N,
                 "piml_mlapm_scenes_advance_f32: N=%lld slots per scene, at most %d are supported (a scene's columns "
                 "stay in shared memory); step a larger crowd with piml_mlapm_advance_ws_f32 (MLAPM.advance)",
                 static_cast<long long>(N), PIML_MLAPM_SCENES_MAX_N);
    PIML_REQUIRE(ds_dim == 1 || ds_dim == 2, "piml_mlapm_scenes_advance_f32: ds_dim=%d, must be 1 or 2", ds_dim);
    PIML_REQUIRE(prm->version == 0 || prm->version == 1,
                 "piml_mlapm_scenes_advance_f32: version %d unsupported (0='raw', 1='GC')", prm->version);
    PIML_REQUIRE(((reinterpret_cast<uintptr_t>(pos) | reinterpret_cast<uintptr_t>(vel) |
                   reinterpret_cast<uintptr_t>(dest) | reinterpret_cast<uintptr_t>(action) |
                   reinterpret_cast<uintptr_t>(pos_new)) & 7u) == 0,
                 "piml_mlapm_scenes_advance_f32: pointers must be 8-byte aligned");
    int iS = static_cast<int>(S), iN = static_cast<int>(N);
    MscShape sh = msc_shape(iN);
    const int64_t grid = (S + sh.k - 1) / sh.k * sh.nchunk;
    const int smem = msc_smem(sh.k * iN, sh.k).total;
    MlConst k0 = mlapm_consts(prm);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const void *kfn = prm->version == 0 ? (prm->exact_math ? reinterpret_cast<const void *>(&mlapm_scenes_kernel<0, true>)
                                                           : reinterpret_cast<const void *>(&mlapm_scenes_kernel<0, false>))
                                        : (prm->exact_math ? reinterpret_cast<const void *>(&mlapm_scenes_kernel<1, true>)
                                                           : reinterpret_cast<const void *>(&mlapm_scenes_kernel<1, false>));
    if (smem > 48 * 1024)                                         // per device: a process may drive several GPUs
        PIML_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const float2 *p2 = reinterpret_cast<const float2 *>(pos), *v2 = reinterpret_cast<const float2 *>(vel);
    const float2 *d2 = reinterpret_cast<const float2 *>(dest);
    float2 *a2 = reinterpret_cast<float2 *>(action), *q2 = reinterpret_cast<float2 *>(pos_new);
    void *args[] = {&p2, &v2, &desired_speed, &ds_dim, &d2, &active, &iS, &iN, &sh, &k0, &scene_params, &dt, &radius,
                    &a2, &q2, &arrived};
    PIML_CUDA(cudaLaunchKernel(kfn, dim3(static_cast<unsigned>(grid)), dim3(sh.k * sh.C), args,
                               static_cast<size_t>(smem), st));
    count_launch();
    return check_launch("mlapm_scenes_kernel");
}

extern "C" int piml_mlapm_advance_f32(const float *pos, const float *vel, const float *desired_speed, int ds_dim,
                                      const float *dest, int64_t N, int64_t row0, int64_t row1,
                                      const piml_mlapm_params *prm, float dt, float radius, float *action,
                                      float *pos_new, uint8_t *arrived, void *workspace, void *stream) {
    PeerPush none;
    none.world = 0;
    return mlapm_advance_impl(pos, vel, desired_speed, ds_dim, dest, N, row0, row1, prm, dt, radius, action, pos_new,
                              arrived, workspace, 0, none, stream);
}

extern "C" int piml_mlapm_advance_ws_f32(const float *pos, const float *vel, const float *desired_speed, int ds_dim,
                                         const float *dest, int64_t N, int64_t row0, int64_t row1,
                                         const piml_mlapm_params *prm, float dt, float radius, float *action,
                                         float *pos_new, uint8_t *arrived, void *workspace, int64_t workspace_bytes,
                                         void *stream) {
    if (N == 0) return PIML_OK;
    PIML_REQUIRE(workspace_bytes >= piml_mlapm_workspace_bytes(N),
                 "piml_mlapm_advance_ws_f32: workspace of %lld bytes, need >= %lld",
                 static_cast<long long>(workspace_bytes), static_cast<long long>(piml_mlapm_workspace_bytes(N)));
    PeerPush none;
    none.world = 0;
    return mlapm_advance_impl(pos, vel, desired_speed, ds_dim, dest, N, row0, row1, prm, dt, radius, action, pos_new,
                              arrived, workspace, workspace_bytes, none, stream);
}

extern "C" int piml_mlapm_advance_push_f32(const float *pos, const float *vel, const float *desired_speed, int ds_dim,
                                           const float *dest, int64_t N, int64_t row0, int64_t row1,
                                           const piml_mlapm_params *prm, float dt, float radius, int world,
                                           const uint64_t *peer_pos_next_host, const uint64_t *peer_vel_next_host,
                                           uint8_t *arrived, void *workspace, void *stream) {
    PIML_REQUIRE(world >= 1 && world <= ML_MAX_PEERS, "piml_mlapm_advance_push_f32: world=%d not in [1,%d]", world,
                 ML_MAX_PEERS);
    PIML_REQUIRE(peer_pos_next_host && peer_vel_next_host, "piml_mlapm_advance_push_f32: null peer pointer table");
    PeerPush push;
    push.world = world;
    for (int g = 0; g < ML_MAX_PEERS; ++g) {
        push.pos[g] = g < world ? reinterpret_cast<float2 *>(static_cast<uintptr_t>(peer_pos_next_host[g])) : nullptr;
        push.vel[g] = g < world ? reinterpret_cast<float2 *>(static_cast<uintptr_t>(peer_vel_next_host[g])) : nullptr;
        PIML_REQUIRE(g >= world || (push.pos[g] && push.vel[g] && (peer_pos_next_host[g] & 7u) == 0 &&
                                    (peer_vel_next_host[g] & 7u) == 0),
                     "piml_mlapm_advance_push_f32: bad peer pointer for rank %d", g);
    }
    return mlapm_advance_impl(pos, vel, desired_speed, ds_dim, dest, N, row0, row1, prm, dt, radius, nullptr, nullptr,
                              arrived, workspace, 0, push, stream);
}

extern "C" int piml_mlapm_step_f32(const float *pos, const float *vel, const float *desired_speed, int ds_dim,
                                   const float *dest, int64_t N, int64_t row0, int64_t row1,
                                   const piml_mlapm_params *prm, float dt, float *action, void *workspace,
                                   void *stream) {
    return piml_mlapm_advance_f32(pos, vel, desired_speed, ds_dim, dest, N, row0, row1, prm, dt, 0.f, action,
                                  nullptr, nullptr, workspace, stream);
}

// ---- agent-sharded symmetric evaluation ------------------------------------------------------------------------------
// Rank g owns the 512-agent blocks [g T / G, (g+1) T / G) and evaluates the block pairs (I, I + d mod T) of its own
// row blocks.  Row-direction sums stay local; the column-direction sums of OTHER ranks' agents are reduced per rank and
// stored into the owner's inbox over NVLink peer memory (phase A).  After one barrier the owner's finalize kernel adds
// the ranks' shares in rank order and pushes the new state into every rank's next-state arrays (phase B); a second
// barrier ends the step.  Traffic per step and rank: 16 B per agent (shares) + 16 B per agent (state) to each peer.

static void sym_block_bounds(int64_t T, int world, int *Ib) {
    for (int g = 0; g <= world; ++g) Ib[g] = static_cast<int>(T * g / world);
}

extern "C" int piml_mlapm_sym_shard_rows(int64_t N, int world, int rank, int64_t *row0, int64_t *row1) {
    PIML_REQUIRE(N > 0 && world >= 1 && world <= ML_MAX_PEERS && rank >= 0 && rank < world && row0 && row1,
                 "piml_mlapm_sym_shard_rows: bad arguments (N=%lld, world=%d, rank=%d)", static_cast<long long>(N),
                 world, rank);
    const int64_t T = sym_blocks(N);
    PIML_REQUIRE(T >= world, "piml_mlapm_sym_shard_rows: %lld blocks of %d agents cannot be split over %d ranks",
                 static_cast<long long>(T), MS_BLOCK, world);
    int Ib[ML_MAX_PEERS + 1];
    sym_block_bounds(T, world, Ib);
    *row0 = static_cast<int64_t>(Ib[rank]) * MS_BLOCK;
    *row1 = static_cast<int64_t>(Ib[rank + 1]) * MS_BLOCK;
    if (*row1 > N) *row1 = N;
    return PIML_OK;
}

// Floats4 per (rank, row) slot of an inbox: the largest shard, so every rank's inbox has the same shape.
static int64_t sym_inbox_stride(int64_t N, int world) {
    const int64_t T = sym_blocks(N);
    return ((T + world - 1) / world) * MS_BLOCK;
}

extern "C" int64_t piml_mlapm_sym_inbox_bytes(int64_t N, int world) {
    if (N <= 0 || world < 1 || world > ML_MAX_PEERS) return 0;
    return sym_inbox_stride(N, world) * world * 4 * sizeof(float);
}

extern "C" int64_t piml_mlapm_sym_shard_workspace_bytes(int64_t N, int world) {
    if (N <= 0 || world < 1 || world > ML_MAX_PEERS) return 0;
    return sym_layout(N, world, nullptr).total;
}

struct SymShardPlan { int64_t T, I0, nI; SymLayout l; };

static int sym_shard_plan(int64_t N, int world, int rank, void *workspace, int64_t workspace_bytes, SymShardPlan *pl) {
    PIML_REQUIRE(N > 0 && N < (1LL << 31) && world >= 1 && world <= ML_MAX_PEERS && rank >= 0 && rank < world,
                 "piml_mlapm_sym: bad shard (N=%lld, world=%d, rank=%d)", static_cast<long long>(N), world, rank);
    PIML_REQUIRE(workspace && workspace_bytes >= piml_mlapm_sym_shard_workspace_bytes(N, world),
                 "piml_mlapm_sym: workspace of %lld bytes, need >= %lld", static_cast<long long>(workspace_bytes),
                 static_cast<long long>(piml_mlapm_sym_shard_workspace_bytes(N, world)));
    pl->T = sym_blocks(N);
    PIML_REQUIRE(pl->T >= world, "piml_mlapm_sym: fewer blocks than ranks");
    int Ib[ML_MAX_PEERS + 1];
    sym_block_bounds(pl->T, world, Ib);
    pl->I0 = Ib[rank];
    pl->nI = Ib[rank + 1] - Ib[rank];
    pl->l = sym_layout(N, world, ws_align(workspace));
    return PIML_OK;
}

extern "C" int piml_mlapm_sym_pairs_push_f32(const float *pos, const float *vel, const float *dest, int64_t N,
                                             int world, int rank, const piml_mlapm_params *prm,
                                             const uint64_t *peer_inbox_host, void *workspace,
                                             int64_t workspace_bytes, void *stream) {
    PIML_REQUIRE(pos && vel && dest && prm && peer_inbox_host, "piml_mlapm_sym_pairs_push_f32: null pointer");
    PIML_REQUIRE(prm->version == 0 || prm->version == 1, "piml_mlapm_sym_pairs_push_f32: version %d unsupported",
                 prm->version);
    const MlConst k = mlapm_consts(prm);
    PIML_REQUIRE(sym_params_ok(prm, k, N), "piml_mlapm_sym_pairs_push_f32: parameters outside the symmetric kernel's "
                                            "domain (exact_math, or a weight that does not decay with distance)");
    SymShardPlan pl;
    int rc = sym_shard_plan(N, world, rank, workspace, workspace_bytes, &pl);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    rc = launch_sym_pairs(prm->version, reinterpret_cast<const float2 *>(pos), reinterpret_cast<const float2 *>(vel),
                          reinterpret_cast<const float2 *>(dest), static_cast<int>(N), pl.T, pl.I0, pl.nI, pl.l, k,
                          ldexpf(1.0f, sym_colscale_log2(N, prm)), nullptr, st);
    if (rc) return rc;
    PeerInbox peers;
    peers.world = world;
    peers.rank = rank;
    sym_block_bounds(pl.T, world, peers.Ib);
    for (int g = world + 1; g <= ML_MAX_PEERS; ++g) peers.Ib[g] = peers.Ib[world];
    peers.stride = sym_inbox_stride(N, world);
    for (int g = 0; g < ML_MAX_PEERS; ++g) {
        peers.inbox[g] = g < world ? reinterpret_cast<float4 *>(static_cast<uintptr_t>(peer_inbox_host[g])) : nullptr;
        PIML_REQUIRE(g >= world || (peers.inbox[g] && (peer_inbox_host[g] & 15u) == 0),
                     "piml_mlapm_sym_pairs_push_f32: bad inbox pointer for rank %d", g);
    }
    const int threads = 256;
    mlapm_sym_colpush_kernel<<<static_cast<unsigned>((N + threads - 1) / threads), threads, 0, st>>>(
        pl.l.colsum, ldexpf(1.0f, -sym_colscale_log2(N, prm)), static_cast<int>(N), peers);
    count_launch();
    return check_launch("mlapm_sym_colpush_kernel");
}

extern "C" int piml_mlapm_sym_finalize_push_f32(const float *pos, const float *vel, const float *desired_speed,
                                                int ds_dim, const float *dest, int64_t N, int world, int rank,
                                                const piml_mlapm_params *prm, float dt, float radius,
                                                const float *inbox_local, const uint64_t *peer_pos_next_host,
                                                const uint64_t *peer_vel_next_host, uint8_t *arrived, void *workspace,
                                                int64_t workspace_bytes, void *stream) {
    PIML_REQUIRE(pos && vel && desired_speed && dest && prm && inbox_local && peer_pos_next_host && peer_vel_next_host,
                 "piml_mlapm_sym_finalize_push_f32: null pointer");
    PIML_REQUIRE(ds_dim == 1 || ds_dim == 2, "piml_mlapm_sym_finalize_push_f32: ds_dim=%d", ds_dim);
    SymShardPlan pl;
    int rc = sym_shard_plan(N, world, rank, workspace, workspace_bytes, &pl);
    if (rc) return rc;
    const MlConst k = mlapm_consts(prm);
    PeerPush push;
    push.world = world;
    for (int g = 0; g < ML_MAX_PEERS; ++g) {
        push.pos[g] = g < world ? reinterpret_cast<float2 *>(static_cast<uintptr_t>(peer_pos_next_host[g])) : nullptr;
        push.vel[g] = g < world ? reinterpret_cast<float2 *>(static_cast<uintptr_t>(peer_vel_next_host[g])) : nullptr;
        PIML_REQUIRE(g >= world || (push.pos[g] && push.vel[g]), "piml_mlapm_sym_finalize_push_f32: bad peer pointer");
    }
    const int64_t row0 = pl.I0 * MS_BLOCK;
    int64_t row1 = (pl.I0 + pl.nI) * MS_BLOCK;
    row1 = row1 > N ? N : row1;
    const int64_t nrows = row1 - row0;
    if (nrows <= 0) return PIML_OK;
    SymPartials symp{nullptr, 0.f, static_cast<int>(pl.nI * MS_BLOCK), reinterpret_cast<const float4 *>(inbox_local),
                     world, sym_inbox_stride(N, world)};
    const int threads = 256;
    mlapm_finalize2_kernel<<<static_cast<unsigned>((nrows * FZ_LPR + threads - 1) / threads), threads, 0,
                             static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const float2 *>(pos), reinterpret_cast<const float2 *>(vel), desired_speed, ds_dim,
        reinterpret_cast<const float2 *>(dest), static_cast<int>(row0), static_cast<int>(row1), pl.l.S, pl.l.partialR,
        prm->A, k.cos_t, k.sin_t, prm->version, prm->tau, dt, radius, nullptr, nullptr, arrived, push, symp);
    count_launch();
    return check_launch("mlapm_finalize2_kernel");
}

// ---- host-buffer entry of an agent-sharded step ------------------------------------------------------------------------
// Every rank uploads ONLY its own rows (1/G of the state over PCIe); this kernel stores them into every rank's
// current-state arrays over NVLink peer memory in ONE launch (the caller follows with a cross-rank barrier).
namespace piml {
struct ScatterPeers { int world; float2 *pos[ML_MAX_PEERS]; float2 *vel[ML_MAX_PEERS]; float2 *dest[ML_MAX_PEERS]; };

__global__ void scatter_rows_push_kernel(const float2 *__restrict__ pos_rows, const float2 *__restrict__ vel_rows,
                                         const float2 *__restrict__ dest_rows, int64_t row0, int64_t nrows,
                                         const __grid_constant__ ScatterPeers peers) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < nrows) {
        const float2 p = pos_rows[i], v = vel_rows[i];
        const float2 d = dest_rows ? dest_rows[i] : make_float2(0.f, 0.f);
        for (int g = 0; g < peers.world; ++g) {
            peers.pos[g][row0 + i] = p;
            peers.vel[g][row0 + i] = v;
            if (dest_rows) peers.dest[g][row0 + i] = d;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) __threadfence_system();
}
}  // namespace piml

extern "C" int piml_scatter_rows_push_f32(const float *pos_rows, const float *vel_rows, const float *dest_rows,
                                          int64_t row0, int64_t nrows, int world, const uint64_t *peer_pos_host,
                                          const uint64_t *peer_vel_host, const uint64_t *peer_dest_host, void *stream) {
    PIML_REQUIRE(world >= 1 && world <= ML_MAX_PEERS && row0 >= 0 && nrows >= 0, "piml_scatter_rows_push_f32: bad shard");
    if (nrows == 0) return PIML_OK;
    PIML_REQUIRE(pos_rows && vel_rows && peer_pos_host && peer_vel_host && (!dest_rows || peer_dest_host),
                 "piml_scatter_rows_push_f32: null pointer");
    ScatterPeers peers;
    peers.world = world;
    for (int g = 0; g < ML_MAX_PEERS; ++g) {
        peers.pos[g] = g < world ? reinterpret_cast<float2 *>(static_cast<uintptr_t>(peer_pos_host[g])) : nullptr;
        peers.vel[g] = g < world ? reinterpret_cast<float2 *>(static_cast<uintptr_t>(peer_vel_host[g])) : nullptr;
        peers.dest[g] = (g < world && dest_rows) ? reinterpret_cast<float2 *>(static_cast<uintptr_t>(peer_dest_host[g]))
                                                 : nullptr;
        PIML_REQUIRE(g >= world || (peers.pos[g] && peers.vel[g] && (!dest_rows || peers.dest[g])),
                     "piml_scatter_rows_push_f32: bad peer pointer for rank %d", g);
    }
    const int threads = 256;
    scatter_rows_push_kernel<<<static_cast<unsigned>((nrows + threads - 1) / threads), threads, 0,
                               static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const float2 *>(pos_rows), reinterpret_cast<const float2 *>(vel_rows),
        reinterpret_cast<const float2 *>(dest_rows), row0, nrows, peers);
    count_launch();
    return check_launch("scatter_rows_push_kernel");
}

