// K5/K6 tensor-core path: the scorer tower's Dense layers on the tcgen05 TF32
// engine (tc_gemm.cu).  passes = 3 is the fp32-faithful 3xTF32 mode used for the
// fp32 configuration; passes = 1 is plain TF32.
//
//   forward  H_d   = act(A_d W_d + b_d)        A K-major, W MN-major (pre-split hi/lo)
//   backward dW_d  = A_d^T dZ_d                both operands MN-major, split on the fly,
//                                              rows split over CTAs -> partials -> reduce
//            dZ_d-1 = (dZ_d W_d^T) * act'(H)   dZ K-major, W K-major (pre-split hi/lo)
// The [K -> output_units] layer and the bias column sums stay on CUDA cores
// (GEMV / reductions, HBM-bound).
#include "common.cuh"
#include "mlp.h"
#include "tc_gemm.cuh"
#include "tc_host.h"

namespace tfr {

struct SplitTable {
  int n;                                    // hidden Dense layers (their kernels get a transpose)
  unsigned long long w_off[TFR_MLP_MAX_LAYERS];
  int kin[TFR_MLP_MAX_LAYERS], nout[TFR_MLP_MAX_LAYERS];
};

// hi = round-to-nearest TF32 of every parameter, lo = the fp32 residual; blockIdx.y = 1 + d
// additionally writes the transposes W_d^T [out, in] of the hidden kernels (hi / lo), the
// K-major B operand of the forward GEMMs: one TMA box per stage instead of one per 32
// output columns.
__global__ void __launch_bounds__(256)
split_params_kernel(const float* __restrict__ p, size_t n, SplitTable t, float* __restrict__ hi,
                    float* __restrict__ lo, float* __restrict__ thi, float* __restrict__ tlo) {
  if (blockIdx.y == 0) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (size_t)gridDim.x * blockDim.x) {
      const float v = p[i];
      uint32_t r;
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));   // round-to-nearest TF32
      const float h = __uint_as_float(r);
      hi[i] = h;
      lo[i] = v - h;
    }
    return;
  }
  const int d = blockIdx.y - 1;
  if (d >= t.n) return;
  const size_t cnt = (size_t)t.kin[d] * t.nout[d];
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < cnt;
       i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i / t.nout[d]), o = (int)(i % t.nout[d]);
    const float v = p[t.w_off[d] + i];
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    const float h = __uint_as_float(r);
    const size_t j = t.w_off[d] + (size_t)o * t.kin[d] + k;
    thi[j] = h;
    tlo[j] = v - h;
  }
}

static int check_dims(const MlpPlan& p) {
  const int L = p.n_dense - 1;
  for (int d = 0; d <= L; ++d)
    if (p.dims[d] % 4 != 0) {
      set_error("tensor-core scorer path needs layer widths that are multiples of 4 "
                "(dims[%d] = %d); use precision fp32", d, p.dims[d]);
      return TFR_UNSUPPORTED;
    }
  return TFR_OK;
}

static int split_params(const MlpPlan& p, const float* params, float* ws, int passes,
                        cudaStream_t st) {
  if (passes != 3) return TFR_OK;
  SplitTable t{};
  t.n = p.n_dense - 1;
  for (int d = 0; d < t.n; ++d) {
    t.w_off[d] = p.w_off[d];
    t.kin[d] = p.dims[d];
    t.nout[d] = p.dims[d + 1];
  }
  dim3 grid(64, (unsigned)(1 + t.n));
  split_params_kernel<<<grid, 256, 0, st>>>(params, p.n_params, t, ws + p.whi_off,
                                            ws + p.wlo_off, ws + p.wthi_off, ws + p.wtlo_off);
  TFR_LAUNCH_OK();
  return TFR_OK;
}

tc::GemmDesc dense_fwd_gemm(const MlpPlan& p, int d, int k0, int K, const float* A, int M,
                            const float* params, const float* ws, int passes) {
  const int N = p.dims[d + 1];
  tc::GemmDesc g{};
  g.A = A; g.lda = K;
  if (passes == 3) {   // W^T [out, in], pre-split: K-major
    g.B = ws + p.wthi_off + p.w_off[d] + k0; g.ldb = p.dims[d];
    g.B_lo = ws + p.wtlo_off + p.w_off[d] + k0;
    g.b_mn = 0;
  } else {             // single-pass TF32 reads the fp32 kernel [in, out] as is: MN-major
    g.B = params + p.w_off[d] + (size_t)k0 * N; g.ldb = N;
    g.B_lo = nullptr;
    g.b_mn = 1;
  }
  g.GM = M; g.GN = N; g.GK = K;
  g.a_mn = 0; g.passes = passes; g.split_b = 0;
  g.splits = 1; g.split_stride = 0;
  return g;
}

tc::GemmDesc dense_dw_gemm(const float* A, int Kin, const float* dZ, int Nout, int rows,
                           int passes, float* C, int splits, size_t split_stride) {
  // dW[Kin, Nout] = A^T dZ in one of two orientations:
  //   direct : GM = Kin (tiles of 128), GN = Nout
  //   swapped: GM = Nout,               GN = Kin, stored transposed
  // Cost of one 32-row k block (tools/mma_rate.cu: a 128 x N x 8 TF32 MMA takes N / 2
  // cycles; profiles/r02_tc_gemm_wait_cycles.txt: the dW GEMMs are bound by shared-memory
  // traffic, 128 B / cycle): per 128-row block of the M side the stage is written by TMA,
  // read by the splitters (the M side goes to tensor memory), the N side is rewritten as
  // hi / lo and read by 12 MMAs.  Fewer than 3 pipeline stages expose the load latency.
  auto cost = [](int gm, int gn) {
    const int n16 = (gn + 15) / 16 * 16;
    const int ntiles = (n16 + 255) / 256;
    const int n_umma = n16 < 256 ? n16 : 256;
    const long long tiles = (long long)((gm + 127) / 128) * ntiles;
    const long long mma = tiles * 12 * (n_umma / 2);
    const long long smem = tiles * (32768 + 896LL * n_umma) / 128;
    const long long stage = 16384 + 256LL * n_umma;
    long long c = mma > smem ? mma : smem;
    if (200 * 1024 / stage < 3) c = c * 3 / 2;
    return c;
  };
  const bool swapped = cost(Nout, Kin) < cost(Kin, Nout);
  tc::GemmDesc g{};
  if (!swapped) {
    g.A = A; g.lda = Kin; g.B = dZ; g.ldb = Nout;
    g.GM = Kin; g.GN = Nout; g.store_transposed = 0;
  } else {
    g.A = dZ; g.lda = Nout; g.B = A; g.ldb = Kin;
    g.GM = Nout; g.GN = Kin; g.store_transposed = 1;
  }
  g.B_lo = nullptr;
  g.C = C; g.ldc = Nout;
  g.GK = rows;
  g.a_mn = 1; g.b_mn = 1; g.passes = passes; g.split_b = 1;
  g.epi = tc::EPI_STORE;
  g.splits = splits; g.split_stride = split_stride;
  return g;
}

int dw_row_splits(int rows, int* rows_per_split) {
  const int sms = num_sms();
  const int per = (rows + sms - 1) / sms;
  *rows_per_split = per < 256 ? 256 : ((per + 127) / 128) * 128;
  return rows > 0 ? (rows + *rows_per_split - 1) / *rows_per_split : 1;
}

int mlp_tc_split_params(const MlpPlan& p, const float* params, float* ws, int passes,
                        cudaStream_t st) {
  int rc = check_dims(p);
  if (rc) return rc;
  return split_params(p, params, ws, passes, st);
}

int mlp_tc_fwd(const float* X, int M, const MlpPlan& p, const float* params,
               const uint8_t* mask, float* ws, float* scores, int passes, cudaStream_t st) {
  return mlp_tc_fwd_from(0, X, M, p, params, mask, ws, scores, passes, st);
}

// Layers first_layer .. L-1 and the output layer.  first_layer > 0: `X` is the activation
// that feeds Dense `first_layer` (the caller produced it and already split the parameters).
int mlp_tc_fwd_from(int first_layer, const float* X, int M, const MlpPlan& p,
                    const float* params, const uint8_t* mask, float* ws, float* scores,
                    int passes, cudaStream_t st) {
  int rc = check_dims(p);
  if (rc) return rc;
  if (first_layer == 0) {
    rc = split_params(p, params, ws, passes, st);
    if (rc) return rc;
  }
  const int L = p.n_dense - 1;
  const float* in = X;
  if (p.input_bn && first_layer == 0) {
    rc = mlp_input_bn_fwd(X, M, p, params, ws, st);
    if (rc) return rc;
    in = ws + p.xin_off;
  }
  for (int d = first_layer; d < L; ++d) {
    tc::GemmDesc g = dense_fwd_gemm(p, d, 0, p.dims[d], in, M, params, ws, passes);
    g.C = ws + (p.use_bn ? p.xhat_off[d] : p.act_off[d]); g.ldc = p.dims[d + 1];
    g.epi = tc::EPI_BIAS_ACT; g.bias = params + p.b_off[d];
    g.act = p.use_bn ? TFR_ACT_NONE : p.activation;   // BN sits before the activation
    // ReLU sign bits for the backward mask: 1 bit per activation instead of re-reading H
    if (p.activation == TFR_ACT_RELU && !p.post())
      g.mask_bits_out = reinterpret_cast<uint32_t*>(ws + p.bits_off[d]);
    rc = tc::gemm(g, st);
    if (rc) return rc;
    rc = mlp_hidden_post_fwd(d, M, p, params, ws, st);
    if (rc) return rc;
    in = ws + p.act_off[d];
  }
  return mlp_out_layer_fwd(in, M, p.dims[L], p.dims[L + 1], params + p.w_off[L],
                           params + p.b_off[L], mask, scores, st);
}

int mlp_tc_bwd(const float* X, int M, const MlpPlan& p, const float* params,
               const float* dscores, const uint8_t* mask, float* ws, float* grads,
               int passes, cudaStream_t st) {
  return mlp_tc_bwd_until(0, nullptr, X, M, p, params, dscores, mask, ws, grads, passes, st);
}

// Backward of the output layer and of Dense L-1 .. stop_layer.  With stop_layer > 0 the
// walk ends after producing dL/dZ of Dense stop_layer - 1 (activation mask applied, bias
// column sums taken); `tail` then describes where that signal and its column sums live.
int mlp_tc_bwd_until(int stop_layer, MlpBwdTail* tail, const float* X, int M, const MlpPlan& p,
                     const float* params, const float* dscores, const uint8_t* mask,
                     float* ws, float* grads, int passes, cudaStream_t st) {
  int rc = check_dims(p);
  if (rc) return rc;
  const int L = p.n_dense - 1;
  float* partial = ws + p.partial_off;
  const size_t pstride = p.partial_stride;
  const int splits = p.splits;
  const float* whi = passes == 3 ? ws + p.whi_off : params;   // written by the forward
  const float* wlo = passes == 3 ? ws + p.wlo_off : nullptr;
  float* dz_cur = ws + p.dz_off[0];
  float* dz_nxt = ws + p.dz_off[1];
  float* tiles = ws + p.tile_off;
  float* oslots = ws + p.oslot_off;
  const float* X0 = p.input_bn ? ws + p.xin_off : X;   // what Dense 0 consumed
  // With BN / dropout the producers emit raw dL/dH; mlp_hidden_pre_bwd turns it into dL/dZ.
  const int mact = p.post() ? TFR_ACT_NONE : p.activation;
  {
    // Output layer (GEMV-shaped, CUDA cores): dZ of the last hidden layer, plus per
    // 256-row block {dW_out, db_out, column sums of dZ}; regrouped to the
    // `splits` partial slots and reduced.
    const int K = p.dims[L], O = p.dims[L + 1];
    const float* H = L > 0 ? ws + p.act_off[L - 1] : X0;
    rc = mlp_out_layer_bwd2(H, M, K, O, params + p.w_off[L], dscores, mask,
                            L > 0 ? mact : TFR_ACT_NONE, p.out_rows,
                            (L > 0 || p.input_bn) ? dz_cur : nullptr, oslots, p.oslot_stride,
                            st);
    if (rc) return rc;
    // out-layer gradient: [K*O + O] summed over the block slots
    rc = mlp_reduce2(oslots, p.out_slots, p.oslot_stride, (size_t)K * O + O, nullptr, 0, 0, 0,
                     grads + p.w_off[L], st);
    if (rc) return rc;
  }
  // Source of the bias partials of the layer being processed: per-slot column sums of
  // its dZ, produced by whichever kernel wrote that dZ.
  const float* bsrc = oslots + (((size_t)p.dims[L] * p.dims[L + 1] + p.dims[L + 1] + 3) & ~(size_t)3);
  int bslots = p.out_slots;
  size_t bstride = p.oslot_stride;
  for (int d = L - 1; d >= stop_layer; --d) {
    const int Kin = p.dims[d], Nout = p.dims[d + 1];
    const float* A = d > 0 ? ws + p.act_off[d - 1] : X0;
    if (p.post()) {
      rc = mlp_hidden_pre_bwd(d, M, p, params, ws, dz_cur, grads, st);
      if (rc) return rc;
      rc = mlp_colsum(dz_cur, M, Nout, p.rows_per_split, splits, tiles, p.tile_stride, 0, st);
      if (rc) return rc;
      bsrc = tiles;
      bslots = splits;
      bstride = p.tile_stride;
    }
    rc = tc::gemm(dense_dw_gemm(A, Kin, dz_cur, Nout, M, passes, partial, splits, pstride), st);
    if (rc) return rc;
    rc = mlp_reduce2(partial, splits, pstride, (size_t)Kin * Nout, bsrc, bslots, bstride,
                     (size_t)Nout, grads + p.w_off[d], st);
    if (rc) return rc;
    if (d > 0 || p.input_bn) {   // d == 0 with input BN: dL/dXin for its gamma / beta
      tc::GemmDesc g{};
      g.A = dz_cur; g.lda = Nout;
      g.B = whi + p.w_off[d]; g.ldb = Nout;     // W [Kin rows (GN), Nout (GK)] : K-major
      g.B_lo = wlo ? wlo + p.w_off[d] : nullptr;
      g.C = dz_nxt; g.ldc = Kin;
      g.GM = M; g.GN = Kin; g.GK = Nout;
      g.a_mn = 0; g.b_mn = 0; g.passes = passes; g.split_b = 0;
      const bool masked = d > 0 && mact != TFR_ACT_NONE;
      g.epi = masked ? tc::EPI_MASK_BITS : tc::EPI_STORE;
      g.mask_bits_in = masked ? reinterpret_cast<const uint32_t*>(ws + p.bits_off[d - 1]) : nullptr;
      g.act = mact;
      g.splits = 1; g.split_stride = 0;
      int cslots = 0;
      if (d > 0 && !p.post()) {
        g.colsum = tiles; g.colsum_stride = (int)p.tile_stride; g.colsum_slots_out = &cslots;
      }
      rc = tc::gemm(g, st);
      if (rc) return rc;
      bsrc = tiles;            // column sums of dZ_{d-1}: one slot per CTA and quarter
      bslots = cslots;
      bstride = p.tile_stride;
      float* t = dz_cur; dz_cur = dz_nxt; dz_nxt = t;
    }
  }
  if (tail) {
    tail->dz = dz_cur;
    tail->dz_other = dz_nxt;
    tail->bias_src = bsrc;
    tail->bias_slots = bslots;
    tail->bias_stride = bstride;
  }
  if (stop_layer > 0) return TFR_OK;
  if (p.input_bn) return mlp_input_bn_bwd(X, M, p, params, ws, dz_cur, grads, st);
  return TFR_OK;
}

}  // namespace tfr
