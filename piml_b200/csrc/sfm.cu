// sfm.cu -- social-force pairwise repulsion per neighbour slot for sm_100a.
// Replaces UTILS.calc_acceleration (reference src/utils/utils.py:31-100).
#include "sfm_common.cuh"

namespace piml {

// v1/v2 use the relative POSITION as dv (reference quirk utils.py:67,84), so cos = (dr.dr)/(r+eps)/(r+eps).
__global__ void calc_acceleration_kernel(const float *__restrict__ rel, int64_t S, int stride, int version, float A,
                                         float B, float C, float D, float ct, float st, float eps,
                                         float2 *__restrict__ out) {
    const int64_t s = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const float dx = rel[s * stride], dy = rel[s * stride + 1];
    const float r = __fadd_rn(norm2_rn(dx, dy), eps);                          // r += eps        (:56)
    const float nx = __fdiv_rn(dx, r), ny = __fdiv_rn(dy, r);                  // dir = dr / r    (:58)
    float a;
    if (version == 0) {
        a = __fmul_rn(A, expf(__fmul_rn(B, r)));                               // A*exp(B*r)      (:57)
        out[s] = make_float2(__fmul_rn(-a, nx), __fmul_rn(-a, ny));
        return;
    }
    // cos = sum(dr*dv)/r/v with dv == dr and v == r                           (:73,:90)
    const float c = __fdiv_rn(__fdiv_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), r), r);
    if (version == 1) {
        a = __fmul_rn(A, expf(__fadd_rn(__fmul_rn(B, r), __fmul_rn(C, c))));   // (:74)
        out[s] = make_float2(__fmul_rn(-a, nx), __fmul_rn(-a, ny));
    } else {
        a = __fmul_rn(A, expf(__fadd_rn(__fadd_rn(__fmul_rn(B, r), __fmul_rn(C, c)),
                                        __fmul_rn(__fmul_rn(D, r), c))));      // (:91)
        const float bx = __fadd_rn(__fmul_rn(ct, nx), __fmul_rn(-st, ny));     // rotate by theta (:93-99)
        const float by = __fadd_rn(__fmul_rn(st, nx), __fmul_rn(ct, ny));
        out[s] = make_float2(__fmul_rn(-a, bx), __fmul_rn(-a, by));
    }
}

// Pure social-force "model" (BASELINE config 2): v0 repulsion per ped / obstacle slot (utils.py:53-58), slot sums,
// destination term (model.py:1205-1210).  One thread per agent: 16 slots x 8 B + 28 B read, 8 B written (+ messages).
__device__ __forceinline__ void sfm_forward_row(const float *__restrict__ ped, const float *__restrict__ obs,
                                                const float *__restrict__ self, int64_t r, int kp, int ko,
                                                const piml_sfm_params &c, float2 *__restrict__ acc,
                                                float2 *__restrict__ ped_msgs, float2 *__restrict__ obs_msgs) {
    float ax = 0.f, ay = 0.f, ox = 0.f, oy = 0.f;
    for (int j = 0; j < kp; ++j) {
        const float2 d = *reinterpret_cast<const float2 *>(ped + (r * kp + j) * 6);
        const float2 m = sfm_v0(d.x, d.y, c.A_ped, c.B_ped, c.eps);
        if (ped_msgs) ped_msgs[r * kp + j] = m;
        ax = __fadd_rn(ax, m.x); ay = __fadd_rn(ay, m.y);
    }
    for (int j = 0; j < ko; ++j) {
        const float2 d = *reinterpret_cast<const float2 *>(obs + (r * ko + j) * 6);
        const float2 m = sfm_v0(d.x, d.y, c.A_obs, c.B_obs, c.eps);
        if (obs_msgs) obs_msgs[r * ko + j] = m;
        ox = __fadd_rn(ox, m.x); oy = __fadd_rn(oy, m.y);
    }
    const float *s = self + r * 7;
    acc[r] = sfm_total(ax, ay, ox, oy, s[0], s[1], s[2], s[3], s[6], c.tau);
}

__global__ void sfm_forward_kernel(const float *__restrict__ ped, const float *__restrict__ obs,
                                   const float *__restrict__ self, int64_t R, int kp, int ko, piml_sfm_params c,
                                   float2 *__restrict__ acc, float2 *__restrict__ ped_msgs,
                                   float2 *__restrict__ obs_msgs) {
    const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= R) return;
    sfm_forward_row(ped, obs, self, r, kp, ko, c, acc, ped_msgs, obs_msgs);
}

// The same per row with the constants of the row's set (row r belongs to set r / N): the forward of a constants sweep.
__global__ void sfm_forward_sets_kernel(const float *__restrict__ ped, const float *__restrict__ obs,
                                        const float *__restrict__ self, int64_t R, int kp, int ko,
                                        const piml_sfm_params *__restrict__ sets, int N, float2 *__restrict__ acc) {
    const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const piml_sfm_params c = sets[r / N];
    sfm_forward_row(ped, obs, self, r, kp, ko, c, acc, nullptr, nullptr);
}

int sfm_forward_sets_launch(const piml_sfm_params *sets, int N, const float *ped_f, const float *obs_f,
                            const float *self_f, int64_t R, int kp, int ko, float *acc, cudaStream_t st) {
    const int threads = 128;
    sfm_forward_sets_kernel<<<static_cast<unsigned>((R + threads - 1) / threads), threads, 0, st>>>(
        ped_f, obs_f, self_f, R, kp, ko, sets, N, reinterpret_cast<float2 *>(acc));
    count_launch();
    return check_launch("sfm_forward_sets_kernel");
}

}  // namespace piml

using namespace piml;

extern "C" int piml_sfm_forward_f32(const piml_sfm_params *prm, const float *ped_f, const float *obs_f,
                                    const float *self_f, int64_t R, int kp, int ko, float *acc, float *ped_msgs,
                                    float *obs_msgs, void *stream) {
    if (R == 0) return PIML_OK;
    PIML_REQUIRE(prm && ped_f && self_f && acc, "piml_sfm_forward_f32: null pointer");
    PIML_REQUIRE(R >= 0 && kp >= 0 && ko >= 0 && (ko == 0 || obs_f), "piml_sfm_forward_f32: bad sizes R=%lld kp=%d ko=%d",
                 static_cast<long long>(R), kp, ko);
    PIML_REQUIRE(prm->tau != 0.f, "piml_sfm_forward_f32: tau must be non-zero");
    PIML_REQUIRE((reinterpret_cast<uintptr_t>(ped_f) & 7u) == 0 && (reinterpret_cast<uintptr_t>(obs_f) & 7u) == 0 &&
                     (reinterpret_cast<uintptr_t>(acc) & 7u) == 0,
                 "piml_sfm_forward_f32: pointers must be 8-byte aligned");
    if (R == 0) return PIML_OK;
    const int threads = 128;
    sfm_forward_kernel<<<static_cast<unsigned>((R + threads - 1) / threads), threads, 0,
                         static_cast<cudaStream_t>(stream)>>>(ped_f, obs_f, self_f, R, kp, ko, *prm,
                                                              reinterpret_cast<float2 *>(acc),
                                                              reinterpret_cast<float2 *>(ped_msgs),
                                                              reinterpret_cast<float2 *>(obs_msgs));
    count_launch();
    return check_launch("sfm_forward_kernel");
}

extern "C" int piml_calc_acceleration_f32(const float *rel, int64_t S, int stride, int version, float A, float B,
                                          float C, float D, float theta, float eps, float *out, void *stream) {
    if (S == 0) return PIML_OK;
    PIML_REQUIRE(rel && out, "piml_calc_acceleration_f32: null pointer");
    PIML_REQUIRE(S >= 0 && stride >= 2, "piml_calc_acceleration_f32: bad size/stride");
    PIML_REQUIRE(version >= 0 && version <= 2, "piml_calc_acceleration_f32: equation version %d unknown", version);
    if (S == 0) return PIML_OK;
    const float ct = static_cast<float>(cos(static_cast<double>(theta)));
    const float st = static_cast<float>(sin(static_cast<double>(theta)));
    const int threads = 256;
    calc_acceleration_kernel<<<static_cast<unsigned>((S + threads - 1) / threads), threads, 0,
                               static_cast<cudaStream_t>(stream)>>>(rel, S, stride, version, A, B, C, D, ct, st, eps,
                                                                    reinterpret_cast<float2 *>(out));
    count_launch();
    return check_launch("calc_acceleration_kernel");
}
