// Host-side plan of the scorer tower: parameter offsets and workspace carving.
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "tc_gemm.cuh"
#include "tfr_b200.h"

namespace tfr {

struct MlpPlan {
  int n_dense;
  int dims[TFR_MLP_MAX_LAYERS + 1];
  int activation;
  // flat parameter layout (floats)
  size_t w_off[TFR_MLP_MAX_LAYERS], b_off[TFR_MLP_MAX_LAYERS], n_params;
  // workspace layout (floats)
  size_t act_off[TFR_MLP_MAX_LAYERS];  // post-activation output of hidden layer d
  size_t bits_off[TFR_MLP_MAX_LAYERS]; // ReLU sign bits of hidden layer d: [ceil(h/32)][M] words
  size_t dz_off[2];                    // ping-pong dZ buffers
  size_t partial_off, partial_stride;  // split partials for dW / db
  int splits, rows_per_split;
  size_t whi_off, wlo_off;             // TF32 hi / lo copies of the flat parameters
  size_t wthi_off, wtlo_off;           // ... and of the per-layer transposes W^T [out, in]
                                       //   (same offsets: K-major B operand of the forward)
  // tensor-core path: per-tile column sums and the fine-grain output-layer slots
  size_t tile_off, tile_stride;        // [4 * ceil(M / 128)][tile_stride]
  int tile_slots;
  size_t oslot_off, oslot_stride;      // [ceil(M / out_rows)][oslot_stride]
  int out_rows, out_slots;
  // BatchNormalization / Dropout (create_tower options)
  int use_bn, input_bn, training;
  float bn_eps, bn_mom, dropout;
  unsigned long long seed;
  float* bn_state;                              // moving mean / variance (device)
  size_t g_off[TFR_MLP_MAX_LAYERS], be_off[TFR_MLP_MAX_LAYERS];   // gamma / beta of hidden BN d
  size_t gin_off, bein_off;                     // input BN gamma / beta
  size_t st_off[TFR_MLP_MAX_LAYERS], stin_off;  // offsets into bn_state (mean; var at +w)
  size_t n_state;
  size_t xhat_off[TFR_MLP_MAX_LAYERS];          // normalised pre-activations of hidden layer d
  size_t xin_off;                               // batch-normalised inputs
  size_t bnstat_off[TFR_MLP_MAX_LAYERS], bnstat_in_off;   // batch mean[w], rstd[w] (fwd -> bwd)
  size_t red_off, red_stride;                   // column-reduction partials [red_blocks][stride]
  int red_rows, red_blocks;
  size_t ws_floats;
  bool post() const { return use_bn || dropout > 0.f; }   // hidden layers need a post pass
};

// BatchNormalization / Dropout passes shared by both scorer paths (mlp_norm.cu).
// Forward, hidden layer d: Z (in the xhat buffer when BN) -> H (act buffer).
int mlp_hidden_post_fwd(int d, int M, const MlpPlan& p, const float* params, float* ws,
                        cudaStream_t st);
// Backward, hidden layer d: dz holds dL/dH_d on entry, dL/dZ_d on exit; writes the
// BN gamma / beta gradients.
int mlp_hidden_pre_bwd(int d, int M, const MlpPlan& p, const float* params, float* ws,
                       float* dz, float* grads, cudaStream_t st);
// Input BN: X -> ws + xin_off; and its parameter gradients from dL/dXin.
int mlp_input_bn_fwd(const float* X, int M, const MlpPlan& p, const float* params, float* ws,
                     cudaStream_t st);
int mlp_input_bn_bwd(const float* X, int M, const MlpPlan& p, const float* params, float* ws,
                     const float* dxin, float* grads, cudaStream_t st);

// Returns 0 on success and fills `p`; sets the error string otherwise.
int make_mlp_plan(const tfr_mlp_cfg* cfg, int M, MlpPlan* p);

// The caller's workspace from its first 256-byte boundary (the *_workspace_bytes queries
// include the 256 bytes).
inline float* ws_base(void* workspace) {
  uintptr_t a = reinterpret_cast<uintptr_t>(workspace);
  a = (a + 255) & ~(uintptr_t)255;
  return reinterpret_cast<float*>(a);
}

int mlp_simt_fwd(const float* X, int M, const MlpPlan& p, const float* params,
                 const uint8_t* mask, float* ws, float* scores, cudaStream_t st);
int mlp_simt_bwd(const float* X, int M, const MlpPlan& p, const float* params,
                 const float* dscores, const uint8_t* mask, float* ws, float* grads,
                 cudaStream_t st);

// tensor-core (tcgen05) path; passes = 1 (TF32) or 3 (3xTF32, fp32-faithful)
int mlp_tc_fwd(const float* X, int M, const MlpPlan& p, const float* params,
               const uint8_t* mask, float* ws, float* scores, int passes, cudaStream_t st);
int mlp_tc_bwd(const float* X, int M, const MlpPlan& p, const float* params,
               const float* dscores, const uint8_t* mask, float* ws, float* grads,
               int passes, cudaStream_t st);

// bf16 tensor-core path (tcgen05 kind::f16): X and all activations are bf16 in HBM
int mlp_bf16_fwd(const void* X, int M, const MlpPlan& p, const float* params,
                 const uint8_t* mask, float* ws, float* scores, cudaStream_t st);
int mlp_bf16_bwd(const void* X, int M, const MlpPlan& p, const float* params,
                 const float* dscores, const uint8_t* mask, float* ws, float* grads,
                 cudaStream_t st);

// partial walks of the tensor-core path (the groupwise fold supplies / consumes layer 0)
struct MlpBwdTail {
  float* dz;               // dL/dZ of Dense stop_layer - 1, [M, dims[stop_layer]]
  float* dz_other;         // the other ping-pong buffer (free)
  const float* bias_src;   // per-slot column sums of dz
  int bias_slots;
  size_t bias_stride;
};
int mlp_tc_split_params(const MlpPlan& p, const float* params, float* ws, int passes,
                        cudaStream_t st);
int mlp_tc_fwd_from(int first_layer, const float* X, int M, const MlpPlan& p,
                    const float* params, const uint8_t* mask, float* ws, float* scores,
                    int passes, cudaStream_t st);
int mlp_tc_bwd_until(int stop_layer, MlpBwdTail* tail, const float* X, int M, const MlpPlan& p,
                     const float* params, const float* dscores, const uint8_t* mask,
                     float* ws, float* grads, int passes, cudaStream_t st);

// Dense layers as 3xTF32 / TF32 GEMMs (mlp_tc.cu), shared by the tower and the groupwise fold.
// Forward of Dense d over rows k0 .. k0 + K - 1 of its kernel W [dims[d], dims[d + 1]]:
// C[M, dims[d + 1]] = A[M, K] W[k0 : k0 + K, :].  C and the epilogue are the caller's.
tc::GemmDesc dense_fwd_gemm(const MlpPlan& p, int d, int k0, int K, const float* A, int M,
                            const float* params, const float* ws, int passes);
// dW[Kin, Nout] = A^T dZ over `rows` rows (A [rows, Kin], dZ [rows, Nout], row-major), as
// `splits` row-range partials C + z * split_stride, each [Kin, Nout] row-major.
tc::GemmDesc dense_dw_gemm(const float* A, int Kin, const float* dZ, int Nout, int rows,
                           int passes, float* C, int splits, size_t split_stride);
// Row ranges the dW GEMMs over `rows` rows are split into (about one per SM).
int dw_row_splits(int rows, int* rows_per_split);

// pieces of the CUDA-core path reused by the tensor-core path
int mlp_out_layer_fwd(const float* H, int M, int K, int O, const float* W, const float* bias,
                      const uint8_t* mask, float* scores, cudaStream_t st);
int mlp_out_layer_bwd(const float* H, int M, int K, int O, const float* W, const float* dS,
                      const uint8_t* mask, int act, int rows_per, int splits, float* dH,
                      float* partial, size_t pstride, cudaStream_t st);
int mlp_out_layer_bwd2(const float* H, int M, int K, int O, const float* W, const float* dS,
                       const uint8_t* mask, int act, int rows_per, float* dH, float* slots,
                       size_t slot_stride, cudaStream_t st);
int mlp_regroup_sum(const float* src, int slots_in, size_t src_stride, size_t src_off, int n,
                    int group, float* dst, int slots_out, size_t dst_stride, size_t dst_off,
                    cudaStream_t st);
int mlp_reduce2(const float* srcA, int slotsA, size_t strideA, size_t nA, const float* srcB,
                int slotsB, size_t strideB, size_t nB, float* out, cudaStream_t st);
int mlp_colsum(const float* dZ, int M, int N, int rows_per, int splits, float* partial,
               size_t pstride, size_t col_offset, cudaStream_t st);
int mlp_reduce_partials(const float* partial, int splits, size_t stride, size_t n, float* out,
                        cudaStream_t st);

}  // namespace tfr
