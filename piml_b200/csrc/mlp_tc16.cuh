// mlp_tc16.cuh -- plan / argument structures of the 16-bit tensor-core forward (mlp_tc16.cu), shared with mlp_tc.cu,
// which owns the C entry points (packing both images, choosing the kernel, compaction and finish kernels).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/piml_b200.h"

namespace piml {

constexpr int T16_THREADS = 576;               // loader warp + MMA warp + 2 slots x 8 epilogue warps
constexpr int T16_MAXL = 12;
constexpr int T16_SLOT_COLS = 256;             // TMEM columns per tile slot: D 128 | A_hi 64 | A_lo 64
constexpr int T16_COL_D = 0, T16_COL_AH = 128, T16_COL_AL = 192;

struct Tc16Layer { int K, Kp, N, relu, bias_off, w_off, bytes; };   // w_off / bytes: into the branch's weight image
struct Tc16Plan {
    int nl, dw;
    Tc16Layer L[T16_MAXL];
    int w_bytes;                               // weight images of one branch (hi then lo per layer)
    int predw_off, predb_off, winv_off, bias_floats;   // inside the branch's fp32 block behind the images
    int64_t branch_floats;                     // floats per branch (images + fp32 block)
    int64_t base;                              // float offset of branch 0 inside the packed buffer
};
// where the torch-order parameters of each (branch, layer) live in the source vector
struct Tc16Src { int64_t src_w[2 * T16_MAXL], src_b[2 * T16_MAXL], pred_src[2]; float scale[T16_MAXL]; };

struct Tc16Args {
    const float *params; const float *ped; const float *obs;
    int64_t R; int kp, ko, ag_ped, ag_obs; int64_t n_ped_tiles, n_obs_tiles;
    float *sums; float *ped_msgs; float *obs_msgs;
    int compact, has_obs;
    const int *list_ped, *list_obs; const int *counts;   // lists NULL: ped / obs hold the compact rows themselves (nn_step.cu)
    float *cmsg_ped, *cmsg_obs; float *f0;
    int64_t set_stride; int ctas_per_set;                 // per-set launch only: floats between the sets' vectors
};

int tc16_build_plan(const piml_net_desc *d, int64_t base_floats, Tc16Plan *P);   // 0 = the network fits this path
size_t tc16_smem_bytes(const Tc16Plan &P);
int tc16_pack(const Tc16Plan &P, const Tc16Src &S, const float *params_torch, float *packed, cudaStream_t st);
int tc16_launch(const Tc16Plan &P, const Tc16Args &a, int64_t tiles_bound, cudaStream_t st);
// one network per set: rows [s a.R, (s+1) a.R) use the vector at a.params + s a.set_stride; dense mode, no messages
int tc16_launch_sets(const Tc16Plan &P, Tc16Args a, int S, cudaStream_t st);
int tc16_plan_for(const piml_net_desc *d, Tc16Plan *P);    // mlp_tc.cu: plan inside a piml_pinnsf_pack_tc_f32 vector; 0 = ok

}  // namespace piml
