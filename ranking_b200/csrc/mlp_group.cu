// K8: groupwise scoring (tfr.model._GroupwiseRankingModel, model.py:273-421) folded into
// the tensor-core scorer tower.
//
// The reference gathers the features of every group member into [B * G, gs, D] (gs =
// group_size, G groups per list), flattens to [B * G, gs * D] and runs the tower; the
// gathered tensor is gs times the input (1.07 GB at BASELINE config 4).  Here the first
// Dense layer is applied BEFORE the gather: with W_1 = [W_1^(0); ...; W_1^(gs-1)] stacked by
// member slot,
//     Z_1[b, g, :] = b_1 + sum_j  X[b, idx[b, g, j], :] W_1^(j)  =  b_1 + sum_j P_j[b, idx[b, g, j], :]
// with P_j = X W_1^(j) one GEMM over the UNGATHERED [B * N, D] matrix per slot.  A small
// gather-add kernel forms H_1 = act(Z_1) (+ ReLU sign bits), the remaining layers run as
// in the univariate tower on [B * G, h_1], and the per-member scores are averaged back
// onto the items (scatter_nd + div_no_nan, model.py:388-412) through an inverse index.
// Backward mirrors it: d logits -> d member scores -> tower backward down to dZ_1 ->
// dP_j[b, i, :] = sum over the groups that hold item i in slot j of dZ_1[b, g, :] (a gather
// through the inverse index: deterministic, no atomics) -> dW_1^(j) = X^T dP_j.
//
// Inverse index: inv[s][b, i, j] = the group of shuffle block s (groups s N .. s N + N - 1)
// that holds item i in slot j, or -1.  The rolling windows of model.py:164-244 place every
// valid item exactly once per slot and shuffle, which is what makes the inverse a function;
// tfr_group_mlp_fwd checks it (a duplicate is reported, not silently dropped).
#include "common.cuh"
#include "mlp.h"
#include "tc_gemm.cuh"
#include "tc_host.h"

namespace tfr {

namespace {

__global__ void __launch_bounds__(256)
group_inv_init_kernel(int* __restrict__ inv, size_t n, int* __restrict__ dup_flag) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) inv[i] = -1;
  if (i == 0) *dup_flag = 0;
}

// inv[s][b, idx[b, g, j], j] = g for valid groups; G = S * N.
__global__ void __launch_bounds__(256)
group_inv_fill_kernel(const int32_t* __restrict__ idx, const uint8_t* __restrict__ gmask, int B,
                      int N, int G, int gs, int* __restrict__ inv, int* __restrict__ dup_flag) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)B * G * gs;
  if (t >= total) return;
  const int j = (int)(t % gs);
  const size_t bg = t / gs;
  const int g = (int)(bg % G), b = (int)(bg / G);
  if (!gmask[bg]) return;
  const int i = idx[t];
  if (i < 0 || i >= N) {
    atomicExch(dup_flag, 2);
    return;
  }
  const int s = g / N;
  const int old = atomicExch(&inv[(((size_t)s * B + b) * N + i) * gs + j], g);
  if (old != -1) atomicExch(dup_flag, 1);
}

// cnt[b, i] = number of (shuffle, slot) pairs that score item i.
__global__ void __launch_bounds__(256)
group_count_kernel(const int* __restrict__ inv, int S, int B, int N, int gs,
                   float* __restrict__ cnt) {
  const size_t bi = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (bi >= (size_t)B * N) return;
  int c = 0;
  for (int s = 0; s < S; ++s)
    for (int j = 0; j < gs; ++j) c += inv[(((size_t)s * B * N) + bi) * gs + j] >= 0;
  cnt[bi] = (float)c;
}

// H1[r, :] = act(b1 + sum_j P_j[b * N + idx[r, j], :]), r = b * G + g; sign bits as in the
// GEMM epilogue: word [(col / 32) * M + r].  One thread per 4 columns.
__global__ void __launch_bounds__(256)
group_gather_fwd_kernel(const float* __restrict__ P, size_t p_stride, const int32_t* __restrict__ idx,
                        int M, int N, int G, int gs, int H, const float* __restrict__ bias, int act,
                        float* __restrict__ out, uint32_t* __restrict__ bits) {
  const int h4 = H >> 2;
  const int lanes_per_row = (h4 + 7) & ~7;       // 8 threads = one 32-column bit word
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t r = t / lanes_per_row;
  const int c4 = (int)(t % lanes_per_row);
  const bool live = r < (size_t)M && c4 < h4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (live) {
    const int b = (int)(r / G);
    acc = __ldg(reinterpret_cast<const float4*>(bias) + c4);
    for (int j = 0; j < gs; ++j) {
      const int i = idx[r * gs + j];
      const float4 v = __ldg(reinterpret_cast<const float4*>(P + (size_t)j * p_stride +
                                                             ((size_t)b * N + i) * H) + c4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    if (act == TFR_ACT_RELU) {
      acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f);
      acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f);
    }
    reinterpret_cast<float4*>(out + r * H)[c4] = acc;
  }
  if (bits) {
    uint32_t w = 0;
    if (live)
      w = ((acc.x > 0.f) ? 1u : 0u) | ((acc.y > 0.f) ? 2u : 0u) | ((acc.z > 0.f) ? 4u : 0u) |
          ((acc.w > 0.f) ? 8u : 0u);
    w <<= 4 * (c4 & 7);
    w |= __shfl_xor_sync(0xffffffffu, w, 1);
    w |= __shfl_xor_sync(0xffffffffu, w, 2);
    w |= __shfl_xor_sync(0xffffffffu, w, 4);
    if ((c4 & 7) == 0 && r < (size_t)M && 4 * c4 < H) bits[(size_t)(c4 >> 3) * M + r] = w;
  }
}

// dP_j[b * N + i, :] = sum_s dZ1[b * G + inv[s][b, i, j], :]   (fixed order: deterministic)
__global__ void __launch_bounds__(256)
group_gather_bwd_kernel(const float* __restrict__ dz, const int* __restrict__ inv, int S, int B,
                        int N, int G, int gs, int j, int H, float* __restrict__ dP) {
  const int h4 = H >> 2;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t bi = t / h4;
  const int c4 = (int)(t % h4);
  if (bi >= (size_t)B * N) return;
  const int b = (int)(bi / N);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s = 0; s < S; ++s) {
    const int g = inv[(((size_t)s * B * N) + bi) * gs + j];
    if (g >= 0) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(dz + ((size_t)b * G + g) * H) + c4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  reinterpret_cast<float4*>(dP + bi * H)[c4] = acc;
}

// logits[b, i] = sum of the member scores item i received / their count (0 when none)
__global__ void __launch_bounds__(256)
group_scatter_mean_fwd_kernel(const float* __restrict__ gscore, const int* __restrict__ inv,
                              const float* __restrict__ cnt, int S, int B, int N, int G, int gs,
                              float* __restrict__ logits) {
  const size_t bi = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (bi >= (size_t)B * N) return;
  const int b = (int)(bi / N);
  float acc = 0.f;
  for (int s = 0; s < S; ++s)
    for (int j = 0; j < gs; ++j) {
      const int g = inv[(((size_t)s * B * N) + bi) * gs + j];
      if (g >= 0) acc += gscore[((size_t)b * G + g) * gs + j];
    }
  const float c = cnt[bi];
  logits[bi] = c > 0.f ? acc / c : 0.f;
}

__global__ void __launch_bounds__(256)
group_scatter_mean_bwd_kernel(const float* __restrict__ dlogits, const int32_t* __restrict__ idx,
                              const uint8_t* __restrict__ gmask, const float* __restrict__ cnt,
                              int B, int N, int G, int gs, float* __restrict__ dgscore) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)B * G * gs) return;
  const size_t bg = t / gs;
  const int b = (int)(bg / G);
  float v = 0.f;
  if (gmask[bg]) {
    const size_t bi = (size_t)b * N + idx[t];
    const float c = cnt[bi];
    v = c > 0.f ? dlogits[bi] / c : 0.f;
  }
  dgscore[t] = v;
}

// Group formation (model.py:164-244, shuffle taken from `perm` when given): one CTA per
// list.  organized = valid positions in order, then invalid ones (utils.py:203-235 without
// shuffling); idx[b, s N + g, j] = organized[perm_s[(g + j) mod max(nv, 1)]],
// gmask[b, s N + g] = g < nv.
__global__ void __launch_bounds__(256)
group_indices_kernel(const uint8_t* __restrict__ is_valid, const int32_t* __restrict__ perm,
                     int N, int S, int gs, int32_t* __restrict__ idx,
                     uint8_t* __restrict__ gmask) {
  extern __shared__ int sm_i[];   // organized [N], warp totals [8], [8]
  int* organized = sm_i;
  int* wtot = sm_i + N;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint8_t* v = is_valid + (size_t)b * N;
  // stable partition by chunks of blockDim items
  int base_valid = 0, nv = 0;
  for (int i = tid; i < N; i += blockDim.x) nv += v[i] != 0;
  nv = warp_sum_int(nv);
  if (lane == 0) wtot[warp] = nv;
  __syncthreads();
  nv = 0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) nv += wtot[w];
  __syncthreads();
  int base_invalid = nv;
  for (int i0 = 0; i0 < N; i0 += blockDim.x) {
    const int i = i0 + tid;
    const bool in = i < N;
    const bool ok = in && v[i] != 0;
    const unsigned bal = __ballot_sync(0xffffffffu, ok);
    const unsigned bin = __ballot_sync(0xffffffffu, in && !ok);
    if (lane == 0) {
      wtot[warp] = __popc(bal);
      wtot[8 + warp] = __popc(bin);
    }
    __syncthreads();
    int pv = 0, pi = 0, tv = 0, ti = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
      if (w < warp) { pv += wtot[w]; pi += wtot[8 + w]; }
      tv += wtot[w];
      ti += wtot[8 + w];
    }
    const unsigned below = (1u << lane) - 1u;
    if (ok) organized[base_valid + pv + __popc(bal & below)] = i;
    else if (in) organized[base_invalid + pi + __popc(bin & below)] = i;
    base_valid += tv;
    base_invalid += ti;
    __syncthreads();
  }
  const int nv1 = nv < 1 ? 1 : nv;
  for (int t = tid; t < S * N * gs; t += blockDim.x) {
    const int j = t % gs, sg = t / gs;
    const int g = sg % N, s_ = sg / N;
    int pos = (g + j) % nv1;
    if (perm) pos = perm[((size_t)s_ * gridDim.x + b) * N + pos];
    idx[((size_t)b * S * N + sg) * gs + j] = organized[pos];
  }
  for (int sg = tid; sg < S * N; sg += blockDim.x)
    gmask[(size_t)b * S * N + sg] = (sg % N) < nv;
}

// K9: out[b, p, :] = in[b, idx[b, p], :] (16-byte vectors): FlattenList's circular padding
// (keras/layers.py:163-173, utils.py:272-356) with idx from group_indices_kernel
// (group_size 1: idx[b, p] = organized[p mod nv]).
__global__ void __launch_bounds__(256)
gather_rows_kernel(const uint4* __restrict__ in, const int32_t* __restrict__ idx, int N,
                   int row_vecs, size_t total_vecs, uint4* __restrict__ out) {
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total_vecs;
       t += (size_t)gridDim.x * blockDim.x) {
    const size_t row = t / row_vecs;
    const int v = (int)(t % row_vecs);
    const size_t b = row / N;
    const int src = idx[row];
    out[t] = __ldg(in + (b * N + src) * row_vecs + v);
  }
}

struct GroupWs {
  float* P;        // [gs][B * N, h1]  first-layer partial products / dP_j
  size_t p_stride;
  int* inv;        // [S][B, N, gs]
  float* cnt;      // [B, N]
  float* gscore;   // [B * G, gs]
  int* dup;        // 1 int
};

size_t group_extra_floats(int B, int N, int G, int gs, int h1) {
  const size_t bn = (size_t)B * N;
  const int S = (G + N - 1) / N;
  auto al = [](size_t x) { return (x + 63) / 64 * 64; };
  return al((size_t)gs * bn * h1) + al((size_t)S * bn * gs) + al(bn) + al((size_t)B * G * gs) + 64;
}

GroupWs carve_group(float* base, int B, int N, int G, int gs, int h1) {
  const size_t bn = (size_t)B * N;
  const int S = (G + N - 1) / N;
  auto al = [](size_t x) { return (x + 63) / 64 * 64; };
  GroupWs w;
  w.P = base;
  w.p_stride = bn * h1;
  base += al((size_t)gs * bn * h1);
  w.inv = reinterpret_cast<int*>(base);
  base += al((size_t)S * bn * gs);
  w.cnt = base;
  base += al(bn);
  w.gscore = base;
  base += al((size_t)B * G * gs);
  w.dup = reinterpret_cast<int*>(base);
  return w;
}

int check_group(const tfr_mlp_cfg* cfg, int B, int N, int G, int gs, int precision, MlpPlan* p) {
  TFR_REQUIRE(B >= 1 && N >= 1 && G >= 1 && gs >= 1, "groupwise tower: empty problem");
  TFR_REQUIRE(G % N == 0, "groupwise tower: G (%d) must be num_shuffles * list_size (%d)", G, N);
  TFR_REQUIRE(precision == TFR_PREC_TF32X3 || precision == TFR_PREC_TF32,
              "groupwise tower: precision must be tf32x3 or tf32 (tensor-core path)");
  int rc = make_mlp_plan(cfg, B * G, p);
  if (rc) return rc;
  TFR_REQUIRE(p->n_dense >= 2, "groupwise tower: needs at least one hidden layer");
  TFR_REQUIRE(p->dims[0] % gs == 0, "groupwise tower: dims[0] (%d) must be group_size * D",
              p->dims[0]);
  TFR_REQUIRE(p->dims[p->n_dense] == gs, "groupwise tower: output_units must equal group_size");
  TFR_REQUIRE(!p->post() && !p->input_bn,
              "groupwise tower: BatchNormalization / Dropout are not offered on the folded path");
  TFR_REQUIRE((p->dims[0] / gs) % 4 == 0 && p->dims[1] % 4 == 0,
              "groupwise tower: D and the first hidden width must be multiples of 4");
  return TFR_OK;
}

}  // namespace

}  // namespace tfr

using namespace tfr;

extern "C" int tfr_group_indices(const uint8_t* is_valid, const int32_t* perm, int B, int N,
                                 int num_shuffles, int gs, int32_t* idx, uint8_t* gmask,
                                 void* stream) {
  TFR_REQUIRE(is_valid && idx && gmask, "NULL argument");
  TFR_REQUIRE(B >= 0 && N >= 1 && N <= 8192 && num_shuffles >= 1 && gs >= 1,
              "group indices: bad sizes (B=%d N=%d shuffles=%d group_size=%d)", B, N,
              num_shuffles, gs);
  if (B == 0) return TFR_OK;
  group_indices_kernel<<<B, 256, (N + 16) * sizeof(int), (cudaStream_t)stream>>>(
      is_valid, perm, N, num_shuffles, gs, idx, gmask);
  TFR_LAUNCH_OK();
  return TFR_OK;
}

extern "C" int tfr_circular_pad_gather(const void* x, const uint8_t* is_valid, int B, int N,
                                       int row_bytes, int32_t* idx_out, void* out,
                                       void* stream) {
  TFR_REQUIRE(x && is_valid && idx_out && out, "NULL argument");
  TFR_REQUIRE(B >= 0 && N >= 1 && N <= 8192, "circular padding: bad sizes (B=%d N=%d)", B, N);
  TFR_REQUIRE(row_bytes > 0 && row_bytes % 16 == 0,
              "circular padding: rows must be multiples of 16 bytes (got %d)", row_bytes);
  TFR_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(out) & 15) == 0, "circular padding: alignment");
  if (B == 0) return TFR_OK;
  cudaStream_t st = (cudaStream_t)stream;
  // idx[b, p] = organized[p mod max(nv, 1)]: group formation with group_size 1; the group
  // mask lands in the tail of idx_out's buffer? no: it is not needed, write it to `out`
  // first (it is overwritten by the gather below)
  group_indices_kernel<<<B, 256, (N + 16) * sizeof(int), st>>>(
      is_valid, nullptr, N, 1, 1, idx_out, static_cast<uint8_t*>(out));
  TFR_LAUNCH_OK();
  const int row_vecs = row_bytes / 16;
  const size_t total = (size_t)B * N * row_vecs;
  size_t blocks = (total + 255) / 256;
  if (blocks > (size_t)num_sms() * 16) blocks = (size_t)num_sms() * 16;
  gather_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(static_cast<const uint4*>(x), idx_out, N,
                                                      row_vecs, total, static_cast<uint4*>(out));
  TFR_LAUNCH_OK();
  return TFR_OK;
}

extern "C" size_t tfr_group_mlp_workspace_bytes(const tfr_mlp_cfg* cfg, int B, int N, int G,
                                                int gs) {
  MlpPlan p;
  if (B < 1 || N < 1 || G < 1 || gs < 1) return 0;
  if (make_mlp_plan(cfg, B * G, &p)) return 0;
  return (p.ws_floats + group_extra_floats(B, N, G, gs, p.dims[1])) * sizeof(float) + 256;
}

extern "C" int tfr_group_mlp_fwd(const float* X, int B, int N, int G, int gs, const int32_t* idx,
                                 const uint8_t* gmask, const tfr_mlp_cfg* cfg,
                                 const float* params, void* workspace, float* logits_out,
                                 int precision, void* stream) {
  MlpPlan p;
  int rc = check_group(cfg, B, N, G, gs, precision, &p);
  if (rc) return rc;
  TFR_REQUIRE(X && idx && gmask && params && workspace && logits_out, "NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int passes = precision == TFR_PREC_TF32X3 ? 3 : 1;
  float* ws = ws_base(workspace);
  const int D = p.dims[0] / gs, H = p.dims[1], M = B * G, S = G / N;
  const size_t bn = (size_t)B * N;
  GroupWs gw = carve_group(ws + p.ws_floats, B, N, G, gs, H);
  // inverse index + counts
  {
    const size_t n = (size_t)S * bn * gs;
    group_inv_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(gw.inv, n, gw.dup);
    TFR_LAUNCH_OK();
    const size_t t = (size_t)M * gs;
    group_inv_fill_kernel<<<(unsigned)((t + 255) / 256), 256, 0, st>>>(idx, gmask, B, N, G, gs,
                                                                       gw.inv, gw.dup);
    TFR_LAUNCH_OK();
    group_count_kernel<<<(unsigned)((bn + 255) / 256), 256, 0, st>>>(gw.inv, S, B, N, gs, gw.cnt);
    TFR_LAUNCH_OK();
  }
  rc = mlp_tc_split_params(p, params, ws, passes, st);
  if (rc) return rc;
  // P_j = X W_1^(j): the first Dense layer on the ungathered [B * N, D] matrix, with slot j's
  // rows j D .. (j + 1) D of W_1
  for (int j = 0; j < gs; ++j) {
    tc::GemmDesc g = dense_fwd_gemm(p, 0, j * D, D, X, (int)bn, params, ws, passes);
    g.C = gw.P + (size_t)j * gw.p_stride; g.ldc = H;
    g.epi = tc::EPI_STORE; g.act = TFR_ACT_NONE;
    rc = tc::gemm(g, st);
    if (rc) return rc;
  }
  {
    const int lanes = ((H >> 2) + 7) & ~7;
    const size_t t = (size_t)M * lanes;
    group_gather_fwd_kernel<<<(unsigned)((t + 255) / 256), 256, 0, st>>>(
        gw.P, gw.p_stride, idx, M, N, G, gs, H, params + p.b_off[0], p.activation,
        ws + p.act_off[0],
        p.activation == TFR_ACT_RELU ? reinterpret_cast<uint32_t*>(ws + p.bits_off[0]) : nullptr);
    TFR_LAUNCH_OK();
  }
  rc = mlp_tc_fwd_from(1, ws + p.act_off[0], M, p, params, nullptr, ws, gw.gscore, passes, st);
  if (rc) return rc;
  group_scatter_mean_fwd_kernel<<<(unsigned)((bn + 255) / 256), 256, 0, st>>>(
      gw.gscore, gw.inv, gw.cnt, S, B, N, G, gs, logits_out);
  TFR_LAUNCH_OK();
  return TFR_OK;
}

extern "C" int tfr_group_mlp_check(const tfr_mlp_cfg* cfg, int B, int N, int G, int gs,
                                   void* workspace, void* stream) {
  // Host-synchronising diagnostic: did the last forward see a (position, slot) pair in two
  // valid groups of one shuffle block, or an index outside [0, N)?
  MlpPlan p;
  int rc = make_mlp_plan(cfg, B * G, &p);
  if (rc) return rc;
  float* ws = ws_base(workspace);
  GroupWs gw = carve_group(ws + p.ws_floats, B, N, G, gs, p.dims[1]);
  int flag = 0;
  TFR_CUDA_OK(cudaMemcpyAsync(&flag, gw.dup, sizeof(int), cudaMemcpyDeviceToHost,
                              (cudaStream_t)stream));
  TFR_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
  TFR_REQUIRE(flag != 2, "groupwise tower: a member index lies outside [0, list_size)");
  TFR_REQUIRE(flag != 1, "groupwise tower: an item occupies the same slot of two valid groups "
                         "of one shuffle (not a rolling-window grouping)");
  return TFR_OK;
}

extern "C" int tfr_group_mlp_bwd(const float* X, int B, int N, int G, int gs, const int32_t* idx,
                                 const uint8_t* gmask, const tfr_mlp_cfg* cfg,
                                 const float* params, const float* dlogits, void* workspace,
                                 float* grads, int precision, void* stream) {
  MlpPlan p;
  int rc = check_group(cfg, B, N, G, gs, precision, &p);
  if (rc) return rc;
  TFR_REQUIRE(X && idx && gmask && params && workspace && dlogits && grads, "NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int passes = precision == TFR_PREC_TF32X3 ? 3 : 1;
  float* ws = ws_base(workspace);
  const int D = p.dims[0] / gs, H = p.dims[1], M = B * G, S = G / N;
  const size_t bn = (size_t)B * N;
  GroupWs gw = carve_group(ws + p.ws_floats, B, N, G, gs, H);
  // d logits -> d member scores (the member-score buffer is reused)
  {
    const size_t t = (size_t)M * gs;
    group_scatter_mean_bwd_kernel<<<(unsigned)((t + 255) / 256), 256, 0, st>>>(
        dlogits, idx, gmask, gw.cnt, B, N, G, gs, gw.gscore);
    TFR_LAUNCH_OK();
  }
  MlpBwdTail tail{};
  rc = mlp_tc_bwd_until(1, &tail, nullptr, M, p, params, gw.gscore, nullptr, ws, grads, passes, st);
  if (rc) return rc;
  // first layer: dP_j by the inverse index, dW_1^(j) = X^T dP_j (rows split over CTAs)
  int rows_per = 0;
  int splits = dw_row_splits((int)bn, &rows_per);
  if (splits > p.splits) splits = p.splits;
  for (int j = 0; j < gs; ++j) {
    float* dP = gw.P + (size_t)j * gw.p_stride;
    const size_t t = bn * (size_t)(H >> 2);
    group_gather_bwd_kernel<<<(unsigned)((t + 255) / 256), 256, 0, st>>>(tail.dz, gw.inv, S, B, N,
                                                                         G, gs, j, H, dP);
    TFR_LAUNCH_OK();
    rc = tc::gemm(dense_dw_gemm(X, D, dP, H, (int)bn, passes, ws + p.partial_off, splits,
                                p.partial_stride), st);
    if (rc) return rc;
    const bool last = j == gs - 1;   // the bias gradient follows the last slot's block
    rc = mlp_reduce2(ws + p.partial_off, splits, p.partial_stride, (size_t)D * H,
                     last ? tail.bias_src : nullptr, last ? tail.bias_slots : 0,
                     last ? tail.bias_stride : 0, last ? (size_t)H : 0,
                     grads + p.w_off[0] + (size_t)j * D * H, st);
    if (rc) return rc;
  }
  return TFR_OK;
}
