// C-ABI glue: error string, scorer-tower dispatch, fused optimizer.
#include <cstring>

#include "common.cuh"
#include "mlp.h"

namespace tfr {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static unsigned long long g_launches = 0;
void count_launch() { __atomic_add_fetch(&g_launches, 1ull, __ATOMIC_RELAXED); }

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int make_mlp_plan(const tfr_mlp_cfg* cfg, int M, MlpPlan* p) {
  TFR_REQUIRE(cfg != nullptr, "cfg must not be NULL");
  TFR_REQUIRE(cfg->n_dense >= 1 && cfg->n_dense <= TFR_MLP_MAX_LAYERS,
              "n_dense %d must be in [1, %d]", cfg->n_dense, TFR_MLP_MAX_LAYERS);
  TFR_REQUIRE(M >= 0, "M must be >= 0");
  TFR_REQUIRE(cfg->activation == TFR_ACT_NONE || cfg->activation == TFR_ACT_RELU,
              "activation %d unsupported", cfg->activation);
  for (int i = 0; i <= cfg->n_dense; ++i)
    TFR_REQUIRE(cfg->dims[i] >= 1, "dims[%d] = %d must be >= 1", i, cfg->dims[i]);
  const int L = cfg->n_dense - 1;
  TFR_REQUIRE(cfg->dims[L] <= 1024, "width %d feeding the output layer exceeds 1024", cfg->dims[L]);
  TFR_REQUIRE(cfg->dims[L + 1] <= 8, "output_units %d exceeds 8", cfg->dims[L + 1]);
  std::memset(p, 0, sizeof(*p));
  p->n_dense = cfg->n_dense;
  p->activation = cfg->activation;
  size_t off = 0, max_wb = 0;
  int max_hidden = 1;
  for (int d = 0; d <= cfg->n_dense; ++d) p->dims[d] = cfg->dims[d];
  for (int d = 0; d < cfg->n_dense; ++d) {
    p->w_off[d] = off;
    off += (size_t)p->dims[d] * p->dims[d + 1];
    p->b_off[d] = off;
    off += p->dims[d + 1];
    // (rows rounded up to 128: the bf16 dW GEMM stores whole 128-row blocks per split)
    const size_t wb = (size_t)((p->dims[d] + 127) / 128 * 128) * p->dims[d + 1] + p->dims[d + 1];
    if (wb > max_wb) max_wb = wb;
    if (d < L && p->dims[d + 1] > max_hidden) max_hidden = p->dims[d + 1];
  }
  // BatchNormalization / Dropout options
  TFR_REQUIRE(cfg->dropout >= 0.f && cfg->dropout < 1.f, "dropout %g must be in [0, 1)",
              (double)cfg->dropout);
  p->use_bn = cfg->use_batch_norm != 0 && L > 0;
  p->input_bn = cfg->input_batch_norm != 0;
  p->training = cfg->training != 0;
  p->bn_eps = cfg->bn_epsilon;
  p->bn_mom = cfg->bn_momentum;
  p->dropout = L > 0 ? cfg->dropout : 0.f;
  p->seed = cfg->dropout_seed;
  p->bn_state = cfg->bn_state;
  if (p->use_bn || p->input_bn) {
    TFR_REQUIRE(cfg->bn_epsilon > 0.f, "bn_epsilon must be > 0");
    TFR_REQUIRE(cfg->bn_momentum >= 0.f && cfg->bn_momentum <= 1.f,
                "bn_momentum %g must be in [0, 1]", (double)cfg->bn_momentum);
  }
  size_t soff = 0;
  int max_bn_w = 1;
  if (p->input_bn) {
    p->gin_off = off; off += p->dims[0];
    p->bein_off = off; off += p->dims[0];
    p->stin_off = soff; soff += 2 * (size_t)p->dims[0];
    max_bn_w = p->dims[0];
  }
  if (p->use_bn)
    for (int d = 0; d < L; ++d) {
      p->g_off[d] = off; off += p->dims[d + 1];
      p->be_off[d] = off; off += p->dims[d + 1];
      p->st_off[d] = soff; soff += 2 * (size_t)p->dims[d + 1];
      if (p->dims[d + 1] > max_bn_w) max_bn_w = p->dims[d + 1];
    }
  p->n_state = soff;
  p->n_params = off;
  // workspace
  size_t w = 0;
  for (int d = 0; d < L; ++d) {
    p->act_off[d] = w;
    w += align_up((size_t)M * p->dims[d + 1], 64);
    p->bits_off[d] = w;
    w += align_up((size_t)M * ((p->dims[d + 1] + 31) / 32), 64);
  }
  if (p->use_bn)
    for (int d = 0; d < L; ++d) {
      p->xhat_off[d] = w;
      w += align_up((size_t)M * p->dims[d + 1], 64);
      p->bnstat_off[d] = w;
      w += align_up(2 * (size_t)p->dims[d + 1], 64);
    }
  if (p->input_bn) {
    p->xin_off = w;
    w += align_up((size_t)M * p->dims[0], 64);
    p->bnstat_in_off = w;
    w += align_up(2 * (size_t)p->dims[0], 64);
    if (p->dims[0] > max_hidden) max_hidden = p->dims[0];   // dZ ping-pong also holds dL/dXin
  }
  if (p->use_bn || p->input_bn) {
    p->red_rows = 256;
    p->red_blocks = M > 0 ? (M + p->red_rows - 1) / p->red_rows : 1;
    p->red_stride = align_up(2 * (size_t)max_bn_w, 64);
    p->red_off = w;
    w += (size_t)p->red_blocks * p->red_stride + align_up(2 * (size_t)max_bn_w, 64);
  }
  for (int i = 0; i < 2; ++i) {
    p->dz_off[i] = w;
    w += align_up((size_t)M * max_hidden, 64);
  }
  // Row splits of the dW GEMMs / bias partials: about one per SM, so that the
  // persistent GEMM's tile list (m_tiles x splits) divides evenly over the SMs.
  p->splits = dw_row_splits(M, &p->rows_per_split);
  p->partial_stride = align_up(max_wb, 64);
  p->partial_off = w;
  w += (size_t)p->splits * p->partial_stride;
  p->whi_off = w;
  w += align_up(p->n_params, 64);
  p->wlo_off = w;
  w += align_up(p->n_params, 64);
  p->wthi_off = w;
  w += align_up(p->n_params, 64);
  p->wtlo_off = w;
  w += align_up(p->n_params, 64);
  p->tile_slots = 4 * 1024;   // upper bound: 4 quarters x persistent CTAs (<= SM count)
  p->tile_stride = align_up((size_t)max_hidden, 64);
  p->tile_off = w;
  w += (size_t)p->tile_slots * p->tile_stride;
  // output-layer backward: about 4 blocks per SM, each owning one slot
  p->out_rows = M > 0 ? ((M + 591) / 592 + 3) / 4 * 4 : 4;
  if (p->out_rows < 16) p->out_rows = 16;
  p->out_slots = (M + p->out_rows - 1) / p->out_rows;
  p->oslot_stride = align_up((size_t)p->dims[L] * (p->dims[L + 1] + 1) + p->dims[L + 1] + 4, 64);
  p->oslot_off = w;
  w += (size_t)p->out_slots * p->oslot_stride;
  p->ws_floats = w;
  return TFR_OK;
}

__global__ void __launch_bounds__(256)
optimizer_kernel(float* __restrict__ params, const float* __restrict__ grads,
                 float* __restrict__ accum, size_t n, int kind, float lr, float eps,
                 float grad_scale) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float g = grads[i] * grad_scale;
  if (kind == 0) {
    params[i] -= lr * g;
  } else {
    // tf.keras.optimizers.Adagrad: accum += g^2; var -= lr * g / (sqrt(accum) + eps)
    const float a = accum[i] + g * g;
    accum[i] = a;
    params[i] -= lr * g / (sqrtf(a) + eps);
  }
}

}  // namespace tfr

using namespace tfr;

extern "C" const char* tfr_last_error(void) { return g_err; }
extern "C" int tfr_version(void) { return 2; }
extern "C" unsigned long long tfr_launch_count(void) {
  return __atomic_load_n(&g_launches, __ATOMIC_RELAXED);
}

extern "C" size_t tfr_mlp_param_count(const tfr_mlp_cfg* cfg) {
  MlpPlan p;
  if (make_mlp_plan(cfg, 0, &p)) return 0;
  return p.n_params;
}

extern "C" size_t tfr_mlp_bn_state_count(const tfr_mlp_cfg* cfg) {
  MlpPlan p;
  if (make_mlp_plan(cfg, 0, &p)) return 0;
  return p.n_state;
}

extern "C" size_t tfr_mlp_workspace_bytes(const tfr_mlp_cfg* cfg, int M) {
  MlpPlan p;
  if (make_mlp_plan(cfg, M, &p)) return 0;
  return p.ws_floats * sizeof(float) + 256;
}

extern "C" int tfr_mlp_fwd(const void* Xv, int M, const tfr_mlp_cfg* cfg,
                           const float* params, const uint8_t* mask, void* workspace,
                           float* scores_out, int precision, void* stream) {
  MlpPlan p;
  int rc = make_mlp_plan(cfg, M, &p);
  if (rc) return rc;
  const float* X = static_cast<const float*>(Xv);   // bf16 when precision == TFR_PREC_BF16
  TFR_REQUIRE(X && params && workspace && scores_out, "NULL argument");
  TFR_REQUIRE(!(p.use_bn || p.input_bn) || p.bn_state, "cfg->bn_state must be set with BN");
  if (M == 0) return TFR_OK;
  switch (precision) {
    case TFR_PREC_FP32:
      return mlp_simt_fwd(X, M, p, params, mask, ws_base(workspace), scores_out,
                          (cudaStream_t)stream);
    case TFR_PREC_TF32X3:
    case TFR_PREC_TF32:
      return mlp_tc_fwd(X, M, p, params, mask, ws_base(workspace), scores_out,
                        precision == TFR_PREC_TF32X3 ? 3 : 1, (cudaStream_t)stream);
    case TFR_PREC_BF16:
      return mlp_bf16_fwd(Xv, M, p, params, mask, ws_base(workspace), scores_out,
                          (cudaStream_t)stream);
    default:
      set_error("precision %d is not available in this build", precision);
      return TFR_UNSUPPORTED;
  }
}

extern "C" int tfr_mlp_bwd(const void* Xv, int M, const tfr_mlp_cfg* cfg,
                           const float* params, const float* dscores, const uint8_t* mask,
                           void* workspace, float* grads, int precision, void* stream) {
  MlpPlan p;
  int rc = make_mlp_plan(cfg, M, &p);
  if (rc) return rc;
  const float* X = static_cast<const float*>(Xv);
  TFR_REQUIRE(X && params && workspace && dscores && grads, "NULL argument");
  TFR_REQUIRE(!(p.use_bn || p.input_bn) || p.bn_state, "cfg->bn_state must be set with BN");
  if (M == 0) {   // an empty shard contributes a zero gradient (never stale memory)
    TFR_CUDA_OK(cudaMemsetAsync(grads, 0, p.n_params * sizeof(float), (cudaStream_t)stream));
    return TFR_OK;
  }
  switch (precision) {
    case TFR_PREC_FP32:
      return mlp_simt_bwd(X, M, p, params, dscores, mask, ws_base(workspace), grads,
                          (cudaStream_t)stream);
    case TFR_PREC_TF32X3:
    case TFR_PREC_TF32:
      return mlp_tc_bwd(X, M, p, params, dscores, mask, ws_base(workspace), grads,
                        precision == TFR_PREC_TF32X3 ? 3 : 1, (cudaStream_t)stream);
    case TFR_PREC_BF16:
      return mlp_bf16_bwd(Xv, M, p, params, dscores, mask, ws_base(workspace), grads,
                          (cudaStream_t)stream);
    default:
      set_error("precision %d is not available in this build", precision);
      return TFR_UNSUPPORTED;
  }
}

extern "C" int tfr_optimizer_step(float* params, const float* grads, float* accum, size_t n,
                                  int kind, float lr, float eps, float grad_scale,
                                  void* stream) {
  TFR_REQUIRE(params && grads, "NULL argument");
  TFR_REQUIRE(kind == 0 || kind == 1, "optimizer kind %d unsupported", kind);
  TFR_REQUIRE(kind == 0 || accum != nullptr, "Adagrad needs an accumulator");
  if (n == 0) return TFR_OK;
  optimizer_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      params, grads, accum, n, kind, lr, eps, grad_scale);
  TFR_LAUNCH_OK();
  return TFR_OK;
}
