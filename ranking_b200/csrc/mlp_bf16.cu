// K5/K6, bf16 mode (TFR_PREC_BF16, BASELINE config 3): the scorer tower's Dense layers on
// the tcgen05 kind::f16 engine (tc_gemm_bf16.cu).
//
//   storage   X, hidden activations H_d and the backward signals dZ_d are bf16 in HBM
//             (half the bytes of every activation term); parameters stay fp32 (master
//             copy, optimizer, all-reduce), a bf16 shadow W_d [in, out] and its transpose
//             W_d^T [out, in] are refreshed by one small kernel per forward;
//   forward   H_d   = act(A_d W_d + b_d)        A K-major, W_d^T K-major, fp32 accumulate,
//                                               bias / ReLU / sign bits in the epilogue
//   backward  dW_d  = A_d^T dZ_d                both MN-major from their row-major storage,
//                                               fp32 partials per row range -> mlp_reduce2
//             dZ_d-1 = (dZ_d W_d^T) * act'      dZ K-major, W_d K-major; ReLU mask from the
//                                               sign bits, bias-gradient column sums (fp32)
//                                               in the epilogue
//   the [h_L -> output_units] layer and RestoreList's fill are HBM-bound CUDA-core kernels
//   over the bf16 activations (fp32 weights, fp32 accumulation, fp32 scores).
// BatchNormalization / Dropout are not offered in this mode.
#include <cuda_bf16.h>

#include "common.cuh"
#include "mlp.h"
#include "tc_gemm_bf16.cuh"
#include "tc_host.h"

namespace tfr {

namespace {

struct LayerTable {
  int n;                                    // hidden Dense layers converted
  unsigned long long w_off[TFR_MLP_MAX_LAYERS];
  int kin[TFR_MLP_MAX_LAYERS], nout[TFR_MLP_MAX_LAYERS];
};

// Wb = bf16(W) in the flat layout, WbT = per-layer transposes [out, in].
__global__ void __launch_bounds__(256)
shadow_params_kernel(const float* __restrict__ p, LayerTable t, __nv_bfloat16* __restrict__ wb,
                     __nv_bfloat16* __restrict__ wbt) {
  const int d = blockIdx.y;
  if (d >= t.n) return;
  const size_t cnt = (size_t)t.kin[d] * t.nout[d];
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < cnt;
       i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i / t.nout[d]), n = (int)(i % t.nout[d]);
    const __nv_bfloat16 v = __float2bfloat16_rn(p[t.w_off[d] + i]);
    wb[t.w_off[d] + i] = v;
    wbt[t.w_off[d] + (size_t)n * t.kin[d] + k] = v;
  }
}

constexpr int kMaxOut = 8;

// scores[m, o] = sum_k H[m, k] W[k, o] + b[o]; masked rows (O == 1) -> ln(1e-10).
// One warp per row, lanes over bf16 pairs.
__global__ void __launch_bounds__(256)
out_fwd_bf16_kernel(const __nv_bfloat162* __restrict__ H2, int M, int K2, int O,
                    const float* __restrict__ W, const float* __restrict__ bias,
                    const uint8_t* __restrict__ mask, float* __restrict__ scores) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int m = warp; m < M; m += nwarps) {
    float acc[kMaxOut];
#pragma unroll
    for (int o = 0; o < kMaxOut; ++o) acc[o] = 0.f;
    for (int k2 = lane; k2 < K2; k2 += 32) {
      const float2 h = __bfloat1622float2(H2[(size_t)m * K2 + k2]);
#pragma unroll
      for (int o = 0; o < kMaxOut; ++o)
        if (o < O) {
          acc[o] = fmaf(h.x, __ldg(W + (size_t)(2 * k2) * O + o), acc[o]);
          acc[o] = fmaf(h.y, __ldg(W + (size_t)(2 * k2 + 1) * O + o), acc[o]);
        }
    }
#pragma unroll
    for (int o = 0; o < kMaxOut; ++o)
      if (o < O) acc[o] = warp_sum(acc[o]);
    if (lane == 0) {
      for (int o = 0; o < O; ++o) {
        float v = acc[o] + bias[o];
        if (mask && O == 1 && !mask[m]) v = kLogEpsilon;
        scores[(size_t)m * O + o] = v;
      }
    }
  }
}

// Output-layer backward over bf16 activations; one block per `rows_per` rows, a thread owns
// two adjacent k.  Per block b: slot[b] = { dW[K*O], db[O], pad to 4, csum[K] } (the layout
// of out_layer_bwd2_kernel, so the reductions downstream are shared); dH (bf16) gets the
// ReLU mask of H.
__global__ void __launch_bounds__(256)
out_bwd_bf16_kernel(const __nv_bfloat162* __restrict__ H2, int M, int K, int O,
                    const float* __restrict__ W, const float* __restrict__ dS,
                    const uint8_t* __restrict__ mask, int act, int rows_per, int KP, int RL,
                    __nv_bfloat162* __restrict__ dH2, float* __restrict__ slots,
                    size_t slot_stride) {
  extern __shared__ float sm[];   // [RL][round4(K * O + O) + K]
  const int K2 = K >> 1;
  const int kp = threadIdx.x % KP, rl = threadIdx.x / KP;
  const int mbeg = blockIdx.x * rows_per, mend = min(M, mbeg + rows_per);
  const bool live_k = kp < K2 && rl < RL;
  float w0[kMaxOut], w1[kMaxOut], dw0[kMaxOut], dw1[kMaxOut], db[kMaxOut];
  float cs0 = 0.f, cs1 = 0.f;
#pragma unroll
  for (int o = 0; o < kMaxOut; ++o) {
    w0[o] = (live_k && o < O) ? W[(size_t)(2 * kp) * O + o] : 0.f;
    w1[o] = (live_k && o < O) ? W[(size_t)(2 * kp + 1) * O + o] : 0.f;
    dw0[o] = dw1[o] = db[o] = 0.f;
  }
  if (rl < RL) {
#pragma unroll 4
    for (int m = mbeg + rl; m < mend; m += RL) {
      const bool live = !(mask && O == 1 && !mask[m]);
      float ds[kMaxOut];
#pragma unroll
      for (int o = 0; o < kMaxOut; ++o) ds[o] = (o < O && live) ? dS[(size_t)m * O + o] : 0.f;
      if (kp < K2) {
        const float2 h = __bfloat1622float2(H2[(size_t)m * K2 + kp]);
        float d0 = 0.f, d1 = 0.f;
#pragma unroll
        for (int o = 0; o < kMaxOut; ++o) {
          d0 = fmaf(ds[o], w0[o], d0);
          d1 = fmaf(ds[o], w1[o], d1);
          dw0[o] = fmaf(h.x, ds[o], dw0[o]);
          dw1[o] = fmaf(h.y, ds[o], dw1[o]);
        }
        if (dH2) {
          if (act == TFR_ACT_RELU) {
            if (!(h.x > 0.f)) d0 = 0.f;
            if (!(h.y > 0.f)) d1 = 0.f;
          }
          dH2[(size_t)m * K2 + kp] = __floats2bfloat162_rn(d0, d1);
          cs0 += d0;
          cs1 += d1;
        }
      }
#pragma unroll
      for (int o = 0; o < kMaxOut; ++o) db[o] += ds[o];
    }
  }
  const int co = (K * O + O + 3) & ~3;
  const int per = co + K;
  if (rl < RL) {
    float* mine = sm + (size_t)rl * per;
    if (kp < K2) {
      for (int o = 0; o < O; ++o) {
        mine[(2 * kp) * O + o] = dw0[o];
        mine[(2 * kp + 1) * O + o] = dw1[o];
      }
      mine[co + 2 * kp] = cs0;
      mine[co + 2 * kp + 1] = cs1;
    }
    if (kp == 0) {
      for (int i = K * O + O; i < co; ++i) mine[i] = 0.f;
      for (int o = 0; o < O; ++o) mine[K * O + o] = db[o];
    }
  }
  __syncthreads();
  float* out = slots + (size_t)blockIdx.x * slot_stride;
  for (int i = threadIdx.x; i < per; i += blockDim.x) {
    float acc = 0.f;
    for (int r = 0; r < RL; ++r) acc += sm[(size_t)r * per + i];
    out[i] = acc;
  }
}

// ---- streaming versions for narrow last layers (K <= 128, O <= 2: the benchmark towers) ----
// Eight lanes share a row: a lane owns 8 consecutive k (one 16-byte load) per 64-wide chunk,
// a warp instruction covers four rows and the loop is unrolled over four of them, so a warp
// keeps 16 rows (2 KB) in flight.  The row-per-warp kernels above move 128 B per warp and
// load round trip: 58 us / 97 us for 34 MB at config 3 (profiles/r02_launches_c3.txt).
constexpr int kFastK = 128, kFastO = 2;

__device__ __forceinline__ void unpack8(const uint4& v, float (&h)[8]) {
  const __nv_bfloat162* p = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 f = __bfloat1622float2(p[j]);
    h[2 * j] = f.x;
    h[2 * j + 1] = f.y;
  }
}

template <int CPL, int O>   // CPL = 64-wide chunks per row (1 or 2)
__global__ void __launch_bounds__(256)
out_fwd_bf16_fast_kernel(const uint4* __restrict__ H8, int M, int K, const float* __restrict__ W,
                         const float* __restrict__ bias, const uint8_t* __restrict__ mask,
                         float* __restrict__ scores) {
  const int l8 = threadIdx.x & 7;
  const int K8 = K >> 3;
  float w[CPL][8][O];
#pragma unroll
  for (int c = 0; c < CPL; ++c)
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int o = 0; o < O; ++o) {
        const int k = (c * 8 + l8) * 8 + j;
        w[c][j][o] = k < K ? __ldg(W + (size_t)k * O + o) : 0.f;
      }
  const int rows_per_it = (gridDim.x * blockDim.x) >> 3;
  const int iters = (M + rows_per_it - 1) / rows_per_it;   // uniform: every lane joins the shuffles
  for (int it = 0; it < iters; ++it) {
    const int m = it * rows_per_it + ((blockIdx.x * blockDim.x + threadIdx.x) >> 3);
    const bool live = m < M;
    float acc[O];
#pragma unroll
    for (int o = 0; o < O; ++o) acc[o] = 0.f;
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
      const int k8 = c * 8 + l8;
      if (live && k8 < K8) {
        float h[8];
        unpack8(__ldg(H8 + (size_t)m * K8 + k8), h);
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
          for (int o = 0; o < O; ++o) acc[o] = fmaf(h[j], w[c][j][o], acc[o]);
      }
    }
#pragma unroll
    for (int o = 0; o < O; ++o) {
      acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 1);
      acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 2);
      acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 4);
    }
    if (live && l8 == 0) {
#pragma unroll
      for (int o = 0; o < O; ++o) {
        float v = acc[o] + bias[o];
        if (mask && O == 1 && !mask[m]) v = kLogEpsilon;
        scores[(size_t)m * O + o] = v;
      }
    }
  }
}

// Slot layout per block as out_bwd_bf16_kernel: { dW[K*O], db[O], pad to 4, csum[K] }.
template <int CPL, int O>
__global__ void __launch_bounds__(256)
out_bwd_bf16_fast_kernel(const uint4* __restrict__ H8, int M, int K, const float* __restrict__ W,
                         const float* __restrict__ dS, const uint8_t* __restrict__ mask, int act,
                         int rows_per, uint4* __restrict__ dH8, float* __restrict__ slots,
                         size_t slot_stride) {
  extern __shared__ float sm[];   // [32 row groups][per]
  const int l8 = threadIdx.x & 7, rg = threadIdx.x >> 3;   // 32 row groups of 8 lanes
  const int K8 = K >> 3;
  const int mbeg = blockIdx.x * rows_per, mend = min(M, mbeg + rows_per);
  float w[CPL][8][O], dw[CPL][8][O], cs[CPL][8], db[O];
#pragma unroll
  for (int c = 0; c < CPL; ++c)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      cs[c][j] = 0.f;
#pragma unroll
      for (int o = 0; o < O; ++o) {
        const int k = (c * 8 + l8) * 8 + j;
        w[c][j][o] = k < K ? __ldg(W + (size_t)k * O + o) : 0.f;
        dw[c][j][o] = 0.f;
      }
    }
#pragma unroll
  for (int o = 0; o < O; ++o) db[o] = 0.f;
#pragma unroll 4
  for (int m = mbeg + rg; m < mend; m += 32) {
    const bool live = !(mask && O == 1 && !mask[m]);
    float ds[O];
#pragma unroll
    for (int o = 0; o < O; ++o) ds[o] = live ? __ldg(dS + (size_t)m * O + o) : 0.f;
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
      const int k8 = c * 8 + l8;
      if (k8 < K8) {
        float h[8], d[8];
        unpack8(__ldg(H8 + (size_t)m * K8 + k8), h);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float dj = 0.f;
#pragma unroll
          for (int o = 0; o < O; ++o) {
            dj = fmaf(ds[o], w[c][j][o], dj);
            dw[c][j][o] = fmaf(h[j], ds[o], dw[c][j][o]);
          }
          if (act == TFR_ACT_RELU && !(h[j] > 0.f)) dj = 0.f;
          d[j] = dj;
          cs[c][j] += dj;
        }
        if (dH8) {
          uint4 o4;
          __nv_bfloat162* q = reinterpret_cast<__nv_bfloat162*>(&o4);
#pragma unroll
          for (int j = 0; j < 4; ++j) q[j] = __floats2bfloat162_rn(d[2 * j], d[2 * j + 1]);
          dH8[(size_t)m * K8 + k8] = o4;
        }
      }
    }
    if (l8 == 0) {
#pragma unroll
      for (int o = 0; o < O; ++o) db[o] += ds[o];
    }
  }
  const int co = (K * O + O + 3) & ~3;
  const int per = co + K;
  float* mine = sm + (size_t)rg * per;
#pragma unroll
  for (int c = 0; c < CPL; ++c)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = (c * 8 + l8) * 8 + j;
      if (k < K) {
#pragma unroll
        for (int o = 0; o < O; ++o) mine[k * O + o] = dw[c][j][o];
        mine[co + k] = cs[c][j];
      }
    }
  if (l8 == 0) {
    for (int i = K * O + O; i < co; ++i) mine[i] = 0.f;
#pragma unroll
    for (int o = 0; o < O; ++o) mine[K * O + o] = db[o];
  }
  __syncthreads();
  float* out = slots + (size_t)blockIdx.x * slot_stride;
  for (int i = threadIdx.x; i < per; i += blockDim.x) {
    float acc = 0.f;
#pragma unroll 8
    for (int r = 0; r < 32; ++r) acc += sm[(size_t)r * per + i];
    out[i] = acc;
  }
}

int check_bf16(const MlpPlan& p) {
  const int L = p.n_dense - 1;
  if (p.post() || p.input_bn) {
    set_error("precision bf16 does not offer BatchNormalization / Dropout");
    return TFR_UNSUPPORTED;
  }
  for (int d = 0; d <= L; ++d)
    if (p.dims[d] % 8 != 0) {
      set_error("precision bf16 needs layer widths that are multiples of 8 (dims[%d] = %d)", d,
                p.dims[d]);
      return TFR_UNSUPPORTED;
    }
  if (p.dims[L] > 512) {
    set_error("precision bf16: the width feeding the output layer must be <= 512 (got %d)",
              p.dims[L]);
    return TFR_UNSUPPORTED;
  }
  return TFR_OK;
}

}  // namespace

static __nv_bfloat16* as_bf16(float* p) { return reinterpret_cast<__nv_bfloat16*>(p); }

int mlp_bf16_fwd(const void* X, int M, const MlpPlan& p, const float* params,
                 const uint8_t* mask, float* ws, float* scores, cudaStream_t st) {
  int rc = check_bf16(p);
  if (rc) return rc;
  const int L = p.n_dense - 1;
  __nv_bfloat16* wb = as_bf16(ws + p.whi_off);    // bf16 shadow, flat layout
  __nv_bfloat16* wbt = as_bf16(ws + p.wlo_off);   // per-layer transposes
  if (L > 0) {
    LayerTable t{};
    t.n = L;
    size_t mx = 0;
    for (int d = 0; d < L; ++d) {
      t.w_off[d] = p.w_off[d];
      t.kin[d] = p.dims[d];
      t.nout[d] = p.dims[d + 1];
      const size_t c = (size_t)p.dims[d] * p.dims[d + 1];
      if (c > mx) mx = c;
    }
    dim3 grid((unsigned)((mx + 255) / 256 < 64 ? (mx + 255) / 256 : 64), (unsigned)L);
    shadow_params_kernel<<<grid, 256, 0, st>>>(params, t, wb, wbt);
    TFR_LAUNCH_OK();
  }
  const void* in = X;
  for (int d = 0; d < L; ++d) {
    tcb::GemmDesc g{};
    g.A = in; g.lda = p.dims[d];
    g.B = wbt + p.w_off[d]; g.ldb = p.dims[d];          // W^T [out, in]: K-major
    g.C = as_bf16(ws + p.act_off[d]); g.ldc = p.dims[d + 1];
    g.GM = M; g.GN = p.dims[d + 1]; g.GK = p.dims[d];
    g.mn = 0;
    g.epi = tcb::EPI_BIAS_ACT; g.bias = params + p.b_off[d]; g.act = p.activation;
    if (p.activation == TFR_ACT_RELU)
      g.mask_bits_out = reinterpret_cast<uint32_t*>(ws + p.bits_off[d]);
    g.splits = 1;
    rc = tcb::gemm(g, st);
    if (rc) return rc;
    in = as_bf16(ws + p.act_off[d]);
  }
  const int K = p.dims[L], O = p.dims[L + 1];
  if (K <= kFastK && O <= kFastO) {
    const int nb = (M + 31) / 32 < num_sms() * 8 ? (M + 31) / 32 : num_sms() * 8;   // 32 rows a pass
    const uint4* H8 = reinterpret_cast<const uint4*>(in);
    const float* Wl = params + p.w_off[L];
    const float* bl = params + p.b_off[L];
#define TFR_OUT_FWD(C_, O_) \
  out_fwd_bf16_fast_kernel<C_, O_><<<nb, 256, 0, st>>>(H8, M, K, Wl, bl, mask, scores)
    if (K <= 64 && O == 1) TFR_OUT_FWD(1, 1);
    else if (K <= 64) TFR_OUT_FWD(1, 2);
    else if (O == 1) TFR_OUT_FWD(2, 1);
    else TFR_OUT_FWD(2, 2);
#undef TFR_OUT_FWD
    TFR_LAUNCH_OK();
    return TFR_OK;
  }
  const int blocks = (M + 7) / 8 < num_sms() * 16 ? (M + 7) / 8 : num_sms() * 16;
  out_fwd_bf16_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat162*>(in), M,
                                              K / 2, O, params + p.w_off[L], params + p.b_off[L],
                                              mask, scores);
  TFR_LAUNCH_OK();
  return TFR_OK;
}

int mlp_bf16_bwd(const void* X, int M, const MlpPlan& p, const float* params,
                 const float* dscores, const uint8_t* mask, float* ws, float* grads,
                 cudaStream_t st) {
  int rc = check_bf16(p);
  if (rc) return rc;
  const int L = p.n_dense - 1;
  const __nv_bfloat16* wb = as_bf16(ws + p.whi_off);   // written by the forward
  float* partial = ws + p.partial_off;
  __nv_bfloat16* dz_cur = as_bf16(ws + p.dz_off[0]);
  __nv_bfloat16* dz_nxt = as_bf16(ws + p.dz_off[1]);
  float* tiles = ws + p.tile_off;
  float* oslots = ws + p.oslot_off;
  {
    const int K = p.dims[L], O = p.dims[L + 1];
    const void* H = L > 0 ? (const void*)as_bf16(ws + p.act_off[L - 1]) : X;
    if (K <= kFastK && O <= kFastO) {
      const int co = (K * O + O + 3) & ~3;
      const size_t smem = (size_t)32 * (co + K) * sizeof(float);
      const uint4* H8 = reinterpret_cast<const uint4*>(H);
      uint4* dH8 = L > 0 ? reinterpret_cast<uint4*>(dz_cur) : nullptr;
      const int actl = L > 0 ? p.activation : TFR_ACT_NONE;
#define TFR_OUT_BWD(C_, O_)                                                                     \
  {                                                                                             \
    if (smem > 48 * 1024)                                                                       \
      TFR_CUDA_OK(cudaFuncSetAttribute(out_bwd_bf16_fast_kernel<C_, O_>,                        \
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    out_bwd_bf16_fast_kernel<C_, O_><<<p.out_slots, 256, smem, st>>>(                           \
        H8, M, K, params + p.w_off[L], dscores, mask, actl, p.out_rows, dH8, oslots,            \
        p.oslot_stride);                                                                        \
  }
      if (K <= 64 && O == 1) TFR_OUT_BWD(1, 1)
      else if (K <= 64) TFR_OUT_BWD(1, 2)
      else if (O == 1) TFR_OUT_BWD(2, 1)
      else TFR_OUT_BWD(2, 2)
#undef TFR_OUT_BWD
      TFR_LAUNCH_OK();
    } else {
    const int K2 = K / 2;
    const int KP = (K2 + 31) / 32 * 32;
    const int RL = 256 / KP;
    const int co = (K * O + O + 3) & ~3;
    const size_t smem = (size_t)RL * (co + K) * sizeof(float);
    if (smem > 48 * 1024)
      TFR_CUDA_OK(cudaFuncSetAttribute(out_bwd_bf16_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    out_bwd_bf16_kernel<<<p.out_slots, 256, smem, st>>>(
        reinterpret_cast<const __nv_bfloat162*>(H), M, K, O, params + p.w_off[L], dscores, mask,
        L > 0 ? p.activation : TFR_ACT_NONE, p.out_rows, KP, RL,
        L > 0 ? reinterpret_cast<__nv_bfloat162*>(dz_cur) : nullptr, oslots, p.oslot_stride);
    TFR_LAUNCH_OK();
    }
    rc = mlp_reduce2(oslots, p.out_slots, p.oslot_stride, (size_t)K * O + O, nullptr, 0, 0, 0,
                     grads + p.w_off[L], st);
    if (rc) return rc;
  }
  const float* bsrc = oslots + (((size_t)p.dims[L] * p.dims[L + 1] + p.dims[L + 1] + 3) & ~(size_t)3);
  int bslots = p.out_slots;
  size_t bstride = p.oslot_stride;
  for (int d = L - 1; d >= 0; --d) {
    const int Kin = p.dims[d], Nout = p.dims[d + 1];
    const void* A = d > 0 ? (const void*)as_bf16(ws + p.act_off[d - 1]) : X;
    const size_t pstride = (size_t)((Kin + 127) / 128 * 128) * Nout;
    {
      tcb::GemmDesc g{};
      g.A = A; g.lda = Kin;
      g.B = dz_cur; g.ldb = Nout;
      g.C = partial; g.ldc = Nout;
      g.GM = Kin; g.GN = Nout; g.GK = M;
      g.mn = 1; g.epi = tcb::EPI_STORE;
      g.splits = p.splits; g.split_stride = pstride;
      rc = tcb::gemm(g, st);
      if (rc) return rc;
    }
    rc = mlp_reduce2(partial, p.splits, pstride, (size_t)Kin * Nout, bsrc, bslots, bstride,
                     (size_t)Nout, grads + p.w_off[d], st);
    if (rc) return rc;
    if (d > 0) {
      tcb::GemmDesc g{};
      g.A = dz_cur; g.lda = Nout;
      g.B = wb + p.w_off[d]; g.ldb = Nout;      // W [in (GN), out (GK)]: K-major
      g.C = dz_nxt; g.ldc = Kin;
      g.GM = M; g.GN = Kin; g.GK = Nout;
      g.mn = 0;
      const bool masked = p.activation == TFR_ACT_RELU;
      g.epi = masked ? tcb::EPI_MASK_BITS : tcb::EPI_STORE;
      g.mask_bits_in = masked ? reinterpret_cast<const uint32_t*>(ws + p.bits_off[d - 1]) : nullptr;
      g.act = p.activation;
      int cslots = 0;
      g.colsum = tiles; g.colsum_stride = (int)p.tile_stride; g.colsum_slots_out = &cslots;
      g.splits = 1;
      rc = tcb::gemm(g, st);
      if (rc) return rc;
      bsrc = tiles;
      bslots = cslots;
      bstride = p.tile_stride;
      __nv_bfloat16* t = dz_cur; dz_cur = dz_nxt; dz_nxt = t;
    }
  }
  return TFR_OK;
}

}  // namespace tfr
