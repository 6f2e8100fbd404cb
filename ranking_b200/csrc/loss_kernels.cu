// K1 / K2 / K3: fused forward+backward loss kernels, one CTA per list.
//
// Each list's scores, labels and weights are staged once into shared memory;
// every O(N^2) pairwise quantity the reference materialises as a [B, N, N]
// tensor (losses_impl.py:61-64) exists only in registers here.  A warp owns a
// row k and its lanes stride over the partners j; the per-item gradient is
// reduced with warp shuffles.  Each unordered pair is visited from both of its
// ends, so no scatter/atomic is needed and results are deterministic.
#include <math_constants.h>

#include "common.cuh"
#include "loss_common.cuh"

namespace tfr {

template <int PHI, int LAM>
__global__ void __launch_bounds__(kLossThreads)
pairwise_loss_kernel(const float* __restrict__ scores, const float* __restrict__ labels,
                     const float* __restrict__ item_w, int w_per_item,
                     const uint8_t* __restrict__ mask, int N, float temperature,
                     LamDev lam, float grad_scale, float* __restrict__ grad,
                     float* __restrict__ row_loss, float* __restrict__ loss_sum,
                     float* __restrict__ w_sum, float* __restrict__ nnz,
                     int32_t* __restrict__ ranks_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const ListView v = carve(smem_raw, N);
  const int b = blockIdx.x, tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;

  const float zmin = load_list(v, scores, labels, item_w, w_per_item, mask, b, N,
                               temperature);
  const bool need_rank = lam_needs_rank(LAM) || ranks_out != nullptr;
  if (need_rank) {
    compute_ranks(v, N, zmin);
    __syncthreads();
    if (ranks_out)
      for (int i = tid; i < N; i += blockDim.x) ranks_out[(size_t)b * N + i] = v.rank[i];
  }
  setup_lambda(lam, v, b, N, tid);
  const int topn = lam.topn > 0 ? lam.topn : N;
  const float inv_t = grad_scale / temperature;

  float part_l = 0.f, part_w = 0.f, part_n = 0.f;
  for (int k = warp; k < N; k += nwarps) {
    float acc_g = 0.f, acc_l = 0.f, acc_w = 0.f, acc_n = 0.f;
    if (v.mv[k]) {
      const float zk = v.z[k], lk = v.l[k], wk = v.w[k];
      for (int j = lane; j < N; j += 32) {
        if (!v.mv[j] || j == k) continue;
        const float lj = v.l[j], zj = v.z[j];
        if (PHI == TFR_PHI_MSE) {
          // all ordered valid pairs i != j (losses_impl.py:972-998)
          const float lm = pair_lambda<LAM>(lam, v, N, topn, k, j);
          const float wkj = lm * wk, wjk = lm * v.w[j];
          const float d = (zk - zj) - (lk - lj);
          acc_l += wkj * d * d;
          acc_w += wkj;
          acc_n += wkj != 0.f ? 1.f : 0.f;
          acc_g += 2.f * d * (wkj + wjk);
        } else if (lk > lj) {  // k is the preferred item of pair (k, j)
          const float W = pair_lambda<LAM>(lam, v, N, topn, k, j) * wk;
          float f, df;
          phi_eval<PHI>(zk - zj, f, df);
          acc_l += W * f;
          acc_w += W;
          acc_n += W != 0.f ? 1.f : 0.f;
          acc_g += W * df;
        } else if (lj > lk) {  // pair (j, k): k is the non-preferred item
          const float W = pair_lambda<LAM>(lam, v, N, topn, j, k) * v.w[j];
          float f, df;
          phi_eval<PHI>(zj - zk, f, df);
          acc_g -= W * df;
        }
      }
    }
    acc_g = warp_sum(acc_g);
    acc_l = warp_sum(acc_l);
    acc_w = warp_sum(acc_w);
    acc_n = warp_sum(acc_n);
    if (lane == 0) {
      if (grad) grad[(size_t)b * N + k] = acc_g * inv_t;
      if (row_loss) row_loss[(size_t)b * N + k] = acc_l;
      part_l += acc_l;
      part_w += acc_w;
      part_n += acc_n;
    }
  }
  part_l = block_sum(part_l, v.red);
  part_w = block_sum(part_w, v.red);
  part_n = block_sum(part_n, v.red);
  if (tid == 0) {
    loss_sum[b] = part_l;
    if (w_sum) w_sum[b] = part_w;
    if (nnz) nnz[b] = part_n;
  }
}

template <int LAM>
__global__ void __launch_bounds__(kLossThreads)
pair_weights_kernel(const float* __restrict__ labels, const int32_t* __restrict__ ranks,
                    int N, LamDev lam, float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const ListView v = carve(smem_raw, N);
  const int b = blockIdx.x, tid = threadIdx.x;
  for (int i = tid; i < N; i += blockDim.x) {
    const float lab = labels[(size_t)b * N + i];
    v.l[i] = lab;
    v.lv[i] = lab >= 0.f;
    v.mv[i] = lab >= 0.f;
    v.rank[i] = ranks[(size_t)b * N + i];
  }
  __syncthreads();
  setup_lambda(lam, v, b, N, tid);
  __syncthreads();
  const int topn = lam.topn > 0 ? lam.topn : N;
  for (int p = tid; p < N * N; p += blockDim.x) {
    const int i = p / N, j = p % N;
    out[(size_t)b * N * N + p] = pair_lambda<LAM>(lam, v, N, topn, i, j);
  }
}

__global__ void __launch_bounds__(kLossThreads)
sorted_ranks_kernel(const float* __restrict__ scores, const float* __restrict__ labels,
                    const uint8_t* __restrict__ mask, int N, int32_t* __restrict__ ranks) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const ListView v = carve(smem_raw, N);
  const int b = blockIdx.x;
  const float zmin = load_list(v, scores, labels, nullptr, 0, mask, b, N, 1.f);
  compute_ranks(v, N, zmin);
  __syncthreads();
  for (int i = threadIdx.x; i < N; i += blockDim.x) ranks[(size_t)b * N + i] = v.rank[i];
}

// ---------------------------------------------------------------------------
// K2  ApproxNDCG / ApproxMRR
// ---------------------------------------------------------------------------

// Each unordered pair {a < b} is evaluated ONCE (sigmoid is antisymmetric about 1/2,
// sigmoid' is even): the warp that owns row a adds the (a, b) term to its row
// accumulator and the mirrored term to a per-lane register accumulator of column b
// (lane l always sees the columns l + 32 t).  T = ceil(N / 32) column registers;
// T == 0 selects the generic both-ends loop for N > 1024.
template <int MODE, int T>
// 7 warps x 7 CTAs/SM: B = 1024 lists in one wave (224 threads measured faster than 192 or 256)
__global__ void __launch_bounds__(T > 0 && T <= 8 ? 224 : kLossThreads, T > 0 && T <= 8 ? 7 : 2)
approx_loss_kernel(const float* __restrict__ scores, const float* __restrict__ labels,
                   const float* __restrict__ item_w, int w_per_item,
                   const uint8_t* __restrict__ mask, int N, float temperature,
                   float grad_scale, int scale_by_weight, float* __restrict__ grad,
                   float* __restrict__ loss, float* __restrict__ weight) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const ListView v = carve(smem_raw, N);
  float* cl = v.g;               // cleaned labels
  float* c = v.disc;             // d loss / d r_i          (N <= N + 2)
  float* r = reinterpret_cast<float*>(v.rank);  // approx ranks
  const int b = blockIdx.x, tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;

  const float zmin = load_list(v, scores, labels, item_w, w_per_item, mask, b, N,
                               temperature);
  // invalid logits -> min - 1e3, invalid labels -> 0   (losses_impl.py:1591-1594)
  float lsum = 0.f, wl = 0.f, lvsum = 0.f;
  const float zinv = -1e3f + zmin;
  for (int i = tid; i < N; i += blockDim.x) {
    const bool mvalid = v.mv[i];
    if (!mvalid) v.z[i] = zinv;
    const float x = mvalid ? v.l[i] : 0.f;
    cl[i] = x;
    lsum += x;
    // list weight = sum(w * l) / sum(l) over label-valid items (:1004-1015)
    const float lv = v.lv[i] ? v.l[i] : 0.f;
    float wraw = 1.f;
    if (item_w) wraw = w_per_item ? item_w[(size_t)b * N + i] : item_w[b];
    wl += wraw * lv;
    lvsum += lv;
  }
  lsum = block_sum(lsum, v.red);
  wl = block_sum(wl, v.red);
  lvsum = block_sum(lvsum, v.red);
  const bool nonzero = lsum > 0.f;
  if (!nonzero) {  // labels := 1e-10 on the whole row (:1598-1599)
    for (int i = tid; i < N; i += blockDim.x) cl[i] = 1e-10f;
  }
  float list_w = item_w ? (lvsum != 0.f ? wl / lvsum : 0.f) : 1.f;
  if (!nonzero) list_w = 0.f;
  // Tail padding: an invalid item sits 1e3 (in units of z) below every valid one, so
  // sigmoid(z_invalid - z_valid) and sigmoid' across that gap are exactly 0 in fp32 and its
  // gain is 0: it changes no valid rank, no loss term and no gradient.  Tiles that lie
  // entirely behind the last valid item are therefore skipped (lists are padded at the tail
  // in every batch the input side produces; holes inside a list are walked as before).
  float lastf = -1.f;
  for (int i = tid; i < N; i += blockDim.x)
    if (v.mv[i]) lastf = fmaxf(lastf, (float)i);
  const int nv_hi = (int)block_max(lastf, v.red) + 1;   // (barrier: publishes z / cl as well)
  const int tmax = (nv_hi + 31) >> 5;

  // pass 1: approx ranks r_i = 0.5 + sum_j sigmoid(z_j - z_i)   (:102-106)
  // [nwarps][N] cross-warp column partials (T > 0), placed after the list view
  float* colpart = reinterpret_cast<float*>(smem_raw + ((list_smem_bytes(N) + 15) & ~(size_t)15));
  if (T > 0) {
    // Column operands live in registers for the whole pass: zc[t] = z'[lane + 32 t]
    // with z' = z * log2(e), so that sigmoid(d) = 1 / (1 + 2^-d') needs one ex2.
    float col[T > 0 ? T : 1], zc[T > 0 ? T : 1];
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const int j = lane + 32 * t;
      col[t] = 0.f;
      // columns past N sit at -huge: sigmoid(z_j - z_i) = 0 without a bounds test
      zc[t] = j < N ? v.z[j] * kLog2e : -3.0e38f;
    }
    // Rows are walked tile by tile (t0 compile-time), so the column loop t = t0..T-1 has
    // static bounds: no divergence bookkeeping, static register indexing, and only the
    // diagonal tile pays for the j > i mask.  2 MUFU + 9 ALU per pair: MUFU-bound.
#pragma unroll
    for (int t0 = 0; t0 < T; ++t0) {
      if (t0 >= tmax) break;
      const int iend = min(nv_hi, 32 * t0 + 32);
      for (int i = 32 * t0 + warp; i < iend; i += nwarps) {
        const float zi = v.z[i] * kLog2e;
        float acc = 0.f;
#pragma unroll
        for (int t = t0; t < T; ++t) {
          if (t >= tmax) break;
          const float d = zc[t] - zi;
          const float e = exp2f_approx(-fabsf(d));
          const float big = rcp_approx(1.f + e);      // sigmoid(|d|)
          const float small = e * big;                // sigmoid(-|d|)
          float sa = d >= 0.f ? big : small;          // sigmoid(z_j - z_i) -> r_i
          float sb = d >= 0.f ? small : big;          // sigmoid(z_i - z_j) -> r_j
          if (t == t0) {
            const bool on = lane + 32 * t0 > i;
            sa = on ? sa : 0.f;
            sb = on ? sb : 0.f;
          }
          acc += sa;
          col[t] += sb;
        }
        acc = warp_sum(acc);
        if (lane == 0) r[i] = acc;
      }
    }
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const int j = lane + 32 * t;
      if (j < N) colpart[warp * N + j] = col[t];
    }
    __syncthreads();
    for (int i = tid; i < N; i += blockDim.x) {
      // + 0.5 of the reference (:106) + sigmoid(0) = 0.5 of the skipped j == i term
      float acc = 1.0f;
      if (i < nv_hi) {
        acc += r[i];
        for (int w = 0; w < nwarps; ++w) acc += colpart[w * N + i];
      }
      r[i] = acc;   // (skipped tail: any finite rank, its gain is 0)
    }
  } else {
    for (int i = warp; i < N; i += nwarps) {
      const float zi = v.z[i];
      float acc = 0.f;
      for (int j = lane; j < N; j += 32) {
        const float d = v.z[j] - zi;
        const float e = __expf(-fabsf(d));
        const float rc = rcp_approx(1.f + e);
        acc += d >= 0.f ? rc : e * rc;
      }
      acc = warp_sum(acc);
      if (lane == 0) r[i] = acc + 0.5f;
    }
  }
  __syncthreads();

  float list_loss;
  if (MODE == 0) {
    // safe gains (:33-49), inverse max DCG with 1/ln(1+k) (:109-134), ndcg (:159-165)
    float lmax = -CUDART_INF_F;
    for (int i = tid; i < N; i += blockDim.x) lmax = fmaxf(lmax, cl[i]);
    lmax = block_max(lmax, v.red);
    const float shift = exp2f(-lmax);
    for (int i = tid; i < N; i += blockDim.x) v.w[i] = exp2f(cl[i] - lmax) - shift;  // G_i
    __syncthreads();
    const float ideal = ideal_dcg(cl, v.w, N, N, v.red,
                                  [](int k) { return 1.f / log1pf((float)k); });
    const float D = ideal > 0.f ? 1.f / ideal : 0.f;
    float dcg = 0.f;
    for (int i = tid; i < N; i += blockDim.x) {
      const float lg = log1pf(r[i]);
      dcg += v.w[i] / lg;
      c[i] = D * v.w[i] / ((1.f + r[i]) * lg * lg);
    }
    dcg = block_sum(dcg, v.red);
    list_loss = -(dcg * D);
  } else {
    // mrr = sum(l_i / r_i) / sum(l_i)   (:1629-1632)
    float s = 0.f, rr = 0.f;
    for (int i = tid; i < N; i += blockDim.x) {
      s += cl[i];
      rr += cl[i] / r[i];
    }
    s = block_sum(s, v.red);
    rr = block_sum(rr, v.red);
    for (int i = tid; i < N; i += blockDim.x) c[i] = cl[i] / (r[i] * r[i] * s);
    list_loss = -(rr / s);
  }
  __syncthreads();

  // pass 2: grad_k = (1/T) sum_i (c_i - c_k) sigmoid'(z_k - z_i)
  if (grad) {
    const float gs = grad_scale / temperature * (scale_by_weight ? list_w : 1.f);
    if (T > 0) {
      float* gacc = reinterpret_cast<float*>(v.l);   // raw labels are no longer needed
      float col[T > 0 ? T : 1], zc[T > 0 ? T : 1], cc[T > 0 ? T : 1];
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int j = lane + 32 * t;
        col[t] = 0.f;
        zc[t] = j < N ? v.z[j] * kLog2e : -3.0e38f;
        cc[t] = j < N ? c[j] : 0.f;
      }
#pragma unroll
      for (int t0 = 0; t0 < T; ++t0) {
        if (t0 >= tmax) break;
        const int kend = min(nv_hi, 32 * t0 + 32);
        for (int k = 32 * t0 + warp; k < kend; k += nwarps) {
          const float zk = v.z[k] * kLog2e, ck = c[k];
          float acc = 0.f;
#pragma unroll
          for (int t = t0; t < T; ++t) {
            if (t >= tmax) break;
            const float e = exp2f_approx(-fabsf(zk - zc[t]));   // columns past N: e = 0
            const float rc = rcp_approx(1.f + e);
            float term = (cc[t] - ck) * (e * rc * rc);           // (c_i - c_k) sigmoid'
            if (t == t0) term = lane + 32 * t0 > k ? term : 0.f;
            acc += term;        // -> grad_k
            col[t] -= term;     // -> grad_i (antisymmetric)
          }
          acc = warp_sum(acc);
          if (lane == 0) gacc[k] = acc;
        }
      }
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int j = lane + 32 * t;
        if (j < N) colpart[warp * N + j] = col[t];
      }
      __syncthreads();
      for (int k = tid; k < N; k += blockDim.x) {
        float acc = 0.f;
        if (k < nv_hi) {
          acc = gacc[k];
          for (int w = 0; w < nwarps; ++w) acc += colpart[w * N + k];
        }
        grad[(size_t)b * N + k] = v.mv[k] ? acc * gs : 0.f;
      }
    } else {
      for (int k = warp; k < N; k += nwarps) {
        float acc = 0.f;
        if (v.mv[k]) {
          const float zk = v.z[k], ck = c[k];
          for (int i = lane; i < N; i += 32) {
            const float e = __expf(-fabsf(zk - v.z[i]));
            const float rc = rcp_approx(1.f + e);
            acc += (c[i] - ck) * (e * rc * rc);
          }
        }
        acc = warp_sum(acc);
        if (lane == 0) grad[(size_t)b * N + k] = acc * gs;
      }
    }
  }
  if (tid == 0) {
    loss[b] = list_loss;
    if (weight) weight[b] = list_w;
  }
}

// ---------------------------------------------------------------------------
// K3  Softmax
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kLossThreads)
softmax_loss_kernel(const float* __restrict__ scores, const float* __restrict__ labels,
                    const float* __restrict__ item_w, int w_per_item,
                    const uint8_t* __restrict__ mask, int N, float temperature,
                    LamDev lam, float grad_scale, int scale_by_weight,
                    float* __restrict__ grad, float* __restrict__ loss,
                    float* __restrict__ weight) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const ListView v = carve(smem_raw, N);
  const int b = blockIdx.x, tid = threadIdx.x;
  const float zmin = load_list(v, scores, labels, item_w, w_per_item, mask, b, N,
                               temperature);
  const bool use_lambda = lam.kind == TFR_LAMBDA_DCG;  // isinstance(DCGLambdaWeight) :1132-1134
  if (use_lambda) {
    compute_ranks(v, N, zmin);
    __syncthreads();
    // individual_weights cleans by the mask-cleaned labels (:1129, :285-287)
    for (int i = tid; i < N; i += blockDim.x) v.lv[i] = v.mv[i] && v.lv[i];
    __syncthreads();
    setup_lambda(lam, v, b, N, tid);
  }
  float* lp = v.w;  // l' : effective labels (w no longer needed as-is)
  float lsum = 0.f;
  for (int i = tid; i < N; i += blockDim.x) {
    const bool mvalid = v.mv[i];
    float x = mvalid ? v.l[i] : 0.f;
    if (use_lambda) x = v.g[i] * v.disc[v.rank[i]];
    float wraw = 1.f;
    if (item_w) wraw = w_per_item ? item_w[(size_t)b * N + i] : item_w[b];
    x *= wraw;
    if (!mvalid) v.z[i] = kLogEpsilon;
    lp[i] = x;
    lsum += x;
  }
  lsum = block_sum(lsum, v.red);
  const bool nonzero = lsum > 0.f;
  float psum = 0.f, zmax = -CUDART_INF_F;
  for (int i = tid; i < N; i += blockDim.x) {
    float p = nonzero ? lp[i] : 1e-10f;
    if (!v.mv[i]) p = 0.f;
    lp[i] = p;
    psum += p;
    zmax = fmaxf(zmax, v.z[i]);
  }
  psum = block_sum(psum, v.red);
  zmax = block_max(zmax, v.red);
  float se = 0.f, dot = 0.f;
  const float pinv = psum != 0.f ? 1.f / psum : 0.f;
  for (int i = tid; i < N; i += blockDim.x) {
    se += expf(v.z[i] - zmax);
    dot += lp[i] * pinv * v.z[i];
  }
  se = block_sum(se, v.red);
  dot = block_sum(dot, v.red);
  const float lse = zmax + logf(se);
  const float ptot = psum != 0.f ? 1.f : 0.f;
  if (grad) {
    const float gs = grad_scale / temperature * (scale_by_weight ? lsum : 1.f);
    for (int i = tid; i < N; i += blockDim.x) {
      const float sm = expf(v.z[i] - lse);
      grad[(size_t)b * N + i] = v.mv[i] ? (sm * ptot - lp[i] * pinv) * gs : 0.f;
    }
  }
  if (tid == 0) {
    loss[b] = lse * ptot - dot;
    if (weight) weight[b] = lsum;
  }
}

__global__ void __launch_bounds__(1024)
weighted_sum_kernel(const float* __restrict__ v, const float* __restrict__ w, int n,
                    float scale, float* __restrict__ out2) {
  __shared__ float red[32];
  float a = 0.f, c = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float wi = w ? w[i] : 1.f;
    a += v[i] * wi;
    c += wi;
  }
  a = block_sum(a, red);
  c = block_sum(c, red);
  if (threadIdx.x == 0) {
    out2[0] = a * scale;
    out2[1] = c;
  }
}


// ---------------------------------------------------------------------------
// K3b  Remaining RankingLossKey members that share the one-CTA-per-list staging:
//   pointwise  SigmoidCrossEntropyLoss / MeanSquaredLoss  (losses_impl.py:1284-1469)
//   listwise   UniqueSoftmaxLoss (:1250-1281), ListMLELoss (:1541-1576)
// ---------------------------------------------------------------------------

// Exclusive prefix sums of a[0..N) in place (block-wide): every thread scans a
// contiguous chunk, chunk totals are scanned through `red`-style shuffles.
__device__ inline void block_exclusive_scan(float* a, int N, float* scratch /*[blockDim.x]*/) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const int per = (N + nt - 1) / nt;
  const int beg = min(N, tid * per), end = min(N, beg + per);
  float s = 0.f;
  for (int i = beg; i < end; ++i) s += a[i];
  scratch[tid] = s;
  __syncthreads();
  if (tid == 0) {              // nt <= 256 chunk totals: serial scan is ~0.3 us
    float run = 0.f;
    for (int t = 0; t < nt; ++t) {
      const float x = scratch[t];
      scratch[t] = run;
      run += x;
    }
  }
  __syncthreads();
  float run = scratch[tid];
  for (int i = beg; i < end; ++i) {
    const float x = a[i];
    a[i] = run;
    run += x;
  }
  __syncthreads();
}

template <int KIND>
__global__ void __launch_bounds__(kLossThreads)
misc_loss_kernel(const float* __restrict__ scores, const float* __restrict__ labels,
                 const float* __restrict__ item_w, int w_per_item,
                 const uint8_t* __restrict__ mask, int N, float temperature,
                 const float* __restrict__ rank_weight, const float* __restrict__ order_scores,
                 int topk, float grad_scale, float* __restrict__ grad, float* __restrict__ row,
                 float* __restrict__ loss, float* __restrict__ weight,
                 float* __restrict__ nonzero) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const ListView v = carve(smem_raw, N);
  float* scratch = reinterpret_cast<float*>(smem_raw + ((list_smem_bytes(N) + 15) & ~(size_t)15));
  const int b = blockIdx.x, tid = threadIdx.x;
  load_list(v, scores, labels, item_w, w_per_item, mask, b, N, temperature);
  const size_t off = (size_t)b * N;
  const float gs = grad_scale / temperature;

  if (KIND == TFR_MISC_SIGMOID_CE || KIND == TFR_MISC_MEAN_SQUARED) {
    // item weight = (label valid ? w : 0) * mask   (:1287-1293, :1443 / :1469)
    float sl = 0.f, sw = 0.f, nz = 0.f;
    for (int i = tid; i < N; i += blockDim.x) {
      const bool mvalid = v.mv[i];
      const float z = mvalid ? v.z[i] : 0.f;
      const float l = mvalid ? v.l[i] : 0.f;
      const float w = mvalid ? v.w[i] : 0.f;
      float f, df;
      if (KIND == TFR_MISC_SIGMOID_CE) {
        // max(z, 0) - z l + log1p(exp(-|z|));  d/dz = sigmoid(z) - l
        const float e = expf(-fabsf(z));
        f = fmaxf(z, 0.f) - z * l + log1pf(e);
        df = (z >= 0.f ? 1.f / (1.f + e) : e / (1.f + e)) - l;
      } else {
        const float d = z - l;
        f = d * d;
        df = 2.f * d;
      }
      if (row) row[off + i] = f * w;
      if (grad) grad[off + i] = mvalid ? df * w * gs : 0.f;
      sl += f * w;
      sw += w;
      nz += w != 0.f ? 1.f : 0.f;
    }
    sl = block_sum(sl, v.red);
    sw = block_sum(sw, v.red);
    nz = block_sum(nz, v.red);
    if (tid == 0) {
      loss[b] = sl;
      if (weight) weight[b] = sw;
      if (nonzero) nonzero[b] = nz;
    }
    return;
  }

  // ---- listwise: cleaned labels / logits and the list weight (:1004-1015) ----
  float wl = 0.f, lvsum = 0.f, lsum_clean = 0.f;
  for (int i = tid; i < N; i += blockDim.x) {
    const bool mvalid = v.mv[i];
    const float lv = v.lv[i] ? v.l[i] : 0.f;
    wl += v.w[i] * lv;              // v.w is already 0 for invalid labels
    lvsum += lv;
    lsum_clean += mvalid ? v.l[i] : 0.f;
    if (!mvalid) {
      v.z[i] = kLogEpsilon;
      v.l[i] = 0.f;
    }
  }
  wl = block_sum(wl, v.red);
  lvsum = block_sum(lvsum, v.red);
  lsum_clean = block_sum(lsum_clean, v.red);
  const float list_w = item_w ? (lvsum != 0.f ? wl / lvsum : 0.f) : 1.f;
  __syncthreads();

  if (KIND == TFR_MISC_UNIQUE_SOFTMAX) {
    // L = sum_i g_i [ -z_i + log( e^{z_i} + sum_{j: l_j < l_i, both valid} e^{z_j} ) ]
    float* g = v.g;                                   // 2^l - 1
    float* m = v.disc;                                // row maxima
    float* q = reinterpret_cast<float*>(v.rank);      // g_i / S_i
    float part = 0.f;
    for (int i = tid; i < N; i += blockDim.x) {
      const float li = v.l[i], zi = v.z[i];
      const bool vi = v.mv[i];
      float mi = zi;
      for (int j = 0; j < N; ++j)
        if (vi && v.mv[j] && li > v.l[j]) mi = fmaxf(mi, v.z[j]);
      float S = expf(zi - mi);
      for (int j = 0; j < N; ++j)
        if (vi && v.mv[j] && li > v.l[j]) S += expf(v.z[j] - mi);
      const float gi = exp2f(li) - 1.f;
      part += gi * (-zi + mi + logf(S));
      g[i] = gi;
      m[i] = mi;
      q[i] = gi / S;
    }
    part = block_sum(part, v.red);   // barrier publishes g / m / q
    if (grad) {
      for (int k = tid; k < N; k += blockDim.x) {
        const float lk = v.l[k], zk = v.z[k];
        const bool vk = v.mv[k];
        float acc = -g[k] + expf(zk - m[k]) * q[k];
        for (int i = 0; i < N; ++i)
          if (vk && v.mv[i] && v.l[i] > lk) acc += expf(zk - m[i]) * q[i];
        grad[off + k] = vk ? acc * gs : 0.f;
      }
    }
    if (tid == 0) {
      loss[b] = part;
      if (weight) weight[b] = list_w;
    }
    return;
  }

  // ---- ListMLE: order by label (valid first, ties by index; the reference shuffles
  // ties randomly and parks invalid items at min(label) - 1e-6), then
  //   L = sum_p w_p [ log sum_{m >= p} e^{z_(m)} - z_(p) ]
  float* zs = v.g;                                   // sorted logits (shifted by the max)
  float* C = v.disc;                                 // suffix sums of exp
  float* A = v.w;                                    // prefix sums of w_p / C_p
  int* pos = v.rank;                                 // position of item i
  float zmax = -CUDART_INF_F;
  const int kmax = topk > 0 ? min(topk, N) : N;     // only the first kmax positions count
  if (order_scores) {
    // CoupledRankDistilLoss (:1984-2116): the order is that of the given (sampled teacher)
    // scores, a plain descending sort with ties by index; the list weight is [sum l > 0]
    float* key = A;                                   // free until the prefix sums
    for (int i = tid; i < N; i += blockDim.x) key[i] = order_scores[off + i];
    __syncthreads();
    for (int i = tid; i < N; i += blockDim.x) {
      const float ki = key[i];
      int cnt = 0;
      for (int j = 0; j < N; ++j) cnt += (key[j] > ki) || (key[j] == ki && j < i);
      pos[i] = cnt;
      zmax = fmaxf(zmax, v.z[i]);
    }
    __syncthreads();
  } else {
    for (int i = tid; i < N; i += blockDim.x) {
      const float li = v.l[i];
      const bool vi = v.mv[i];
      int cnt = 0;
      for (int j = 0; j < N; ++j) {
        const bool vj = v.mv[j];
        const float lj = v.l[j];
        const bool before = vi == vj ? ((vi && lj > li) || ((!vi || lj == li) && j < i)) : vj;
        cnt += before;
      }
      pos[i] = cnt;
      zmax = fmaxf(zmax, v.z[i]);
    }
  }
  zmax = block_max(zmax, v.red);
  const float lead_eps = order_scores ? expf(kLogEpsilon - zmax) : 0.f;
  for (int i = tid; i < N; i += blockDim.x) zs[pos[i]] = v.z[i] - zmax;
  __syncthreads();
  // suffix sums: exclusive prefix over the reversed order, plus the own term
  for (int p = tid; p < N; p += blockDim.x) C[N - 1 - p] = expf(zs[p]);
  __syncthreads();
  block_exclusive_scan(C, N, scratch);               // C[r] = sum_{r' < r} e_rev[r']
  float part = 0.f;
  for (int p = tid; p < N; p += blockDim.x) {
    // sum_{m >= p}; RankDistil masks the p leading entries of the denominator to
    // log(1e-10) instead of dropping them (:2094-2097), i.e. adds p * 1e-10
    const float suffix = C[N - 1 - p] + expf(zs[p]) + (float)p * lead_eps;
    const float wp = p < kmax ? (rank_weight ? rank_weight[p] : 1.f) : 0.f;
    part += wp * (logf(suffix) - zs[p]);
    A[p] = wp / suffix;
  }
  part = block_sum(part, v.red);
  if (grad) {
    __syncthreads();
    block_exclusive_scan(A, N, scratch);             // A[p] = sum_{k < p} w_k / C_k
    for (int i = tid; i < N; i += blockDim.x) {
      const int p = pos[i];
      const float wp = p < kmax ? (rank_weight ? rank_weight[p] : 1.f) : 0.f;
      const float e = expf(zs[p]);
      const float suffix = C[N - 1 - p] + e + (float)p * lead_eps;
      const float gsum = A[p] + wp / suffix;          // inclusive prefix
      grad[off + i] = v.mv[i] ? (e * gsum - wp) * gs : 0.f;
    }
  }
  if (tid == 0) {
    loss[b] = part;
    // RankDistil: loss weight = [sum of the cleaned labels > 0] (:2027-2029, :2116)
    if (weight) weight[b] = order_scores ? (lsum_clean > 0.f ? list_w : 0.f) : list_w;
  }
}

// ---------------------------------------------------------------------------
// Gumbel sampler (losses_impl.py:540-649): S perturbed copies of every list,
//   out = log(softmax((s + G) / T) + 1e-20),  G = -log(-log(u + 1e-20) + 1e-20),
// invalid labels (< 0) sit at log(1e-20) before the softmax.  u is a counter hash of
// (seed, element) — see the header — so the backward pass regenerates it.
// ---------------------------------------------------------------------------
__device__ __forceinline__ float hash_uniform01(unsigned long long seed, unsigned long long idx) {
  unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (idx + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (float)(z >> 40) * (1.0f / 16777216.0f);
}

// mode 0: GumbelSampler (:540-649): z = label valid ? (score + G) / T : log(1e-20).
// mode 1: CoupledRankDistil teacher (:2031-2046): the teacher scores ARE the labels,
//         z = (label valid ? label : log(1e-10)) + G.
__device__ __forceinline__ float gumbel_logit(float score, float label, float inv_t,
                                              unsigned long long seed, unsigned long long idx,
                                              int mode) {
  const bool ok = label >= 0.f;
  if (mode == 0 && !ok) return logf(1e-20f);
  const float u = hash_uniform01(seed, idx);
  const float g = -logf(-logf(u + 1e-20f) + 1e-20f);
  if (mode == 1) return (ok ? label : logf(1e-10f)) + g;
  return (score + g) * inv_t;
}

// grid (S, B): list (b, s) -> row b * S + s of out.
__global__ void __launch_bounds__(kLossThreads)
gumbel_sample_fwd_kernel(const float* __restrict__ scores, const float* __restrict__ labels,
                         int N, int S, float inv_t, unsigned long long seed, int mode,
                         float* __restrict__ out) {
  extern __shared__ float zs[];          // [N] + red[32]
  float* red = zs + N;
  const int s = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const size_t in_off = (size_t)b * N, row = (size_t)b * S + s;
  float zmax = -CUDART_INF_F;
  for (int i = tid; i < N; i += blockDim.x) {
    const float z = gumbel_logit(scores ? scores[in_off + i] : 0.f, labels[in_off + i], inv_t,
                                 seed, row * N + i, mode);
    zs[i] = z;
    zmax = fmaxf(zmax, z);
  }
  zmax = block_max(zmax, red);
  float se = 0.f;
  for (int i = tid; i < N; i += blockDim.x) se += expf(zs[i] - zmax);
  se = block_sum(se, red);
  const float inv = 1.f / se;
  const float eps = mode == 1 ? 1e-10f : 1e-20f;
  for (int i = tid; i < N; i += blockDim.x)
    out[row * N + i] = logf(expf(zs[i] - zmax) * inv + eps);
}

// grid (B): d scores[b, i] = sum_s (1/T) (a_i - p_i sum_j a_j), a_j = gout_j p_j / (p_j + 1e-20)
__global__ void __launch_bounds__(kLossThreads)
gumbel_sample_bwd_kernel(const float* __restrict__ scores, const float* __restrict__ labels,
                         int N, int S, float inv_t, unsigned long long seed,
                         const float* __restrict__ gout, float* __restrict__ gin) {
  extern __shared__ float zs[];          // z [N], acc [N], red[32]
  float* acc = zs + N;
  float* red = acc + N;
  const int b = blockIdx.x, tid = threadIdx.x;
  const size_t in_off = (size_t)b * N;
  for (int i = tid; i < N; i += blockDim.x) acc[i] = 0.f;
  for (int s = 0; s < S; ++s) {
    const size_t row = (size_t)b * S + s;
    float zmax = -CUDART_INF_F;
    for (int i = tid; i < N; i += blockDim.x) {
      const float z = gumbel_logit(scores[in_off + i], labels[in_off + i], inv_t, seed,
                                   row * N + i, 0);
      zs[i] = z;
      zmax = fmaxf(zmax, z);
    }
    zmax = block_max(zmax, red);
    float se = 0.f;
    for (int i = tid; i < N; i += blockDim.x) se += expf(zs[i] - zmax);
    se = block_sum(se, red);
    const float inv = 1.f / se;
    float sa = 0.f;
    for (int i = tid; i < N; i += blockDim.x) {
      const float p = expf(zs[i] - zmax) * inv;
      const float a = gout[row * N + i] * (p / (p + 1e-20f));
      zs[i] = p;                 // own element only: safe without a barrier
      sa += a;
      acc[i] += a;               // a_i part
    }
    sa = block_sum(sa, red);
    for (int i = tid; i < N; i += blockDim.x) acc[i] -= zs[i] * sa;
    __syncthreads();
  }
  for (int i = tid; i < N; i += blockDim.x)
    gin[in_off + i] = labels[in_off + i] >= 0.f ? acc[i] * inv_t : 0.f;
}

// ---------------------------------------------------------------------------
// OrdinalLoss (losses_impl.py:1850-1918): K ordinal heads per item, head k trained
// with sigmoid cross entropy against [label >= k + 1] (plus the fraction when asked).
// Pointwise weights / outputs as in K3b.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kLossThreads)
ordinal_loss_kernel(const float* __restrict__ scores, const float* __restrict__ labels,
                    const float* __restrict__ item_w, int w_per_item,
                    const uint8_t* __restrict__ mask, int N, int K, float temperature,
                    int use_fraction, float grad_scale, float* __restrict__ grad,
                    float* __restrict__ row, float* __restrict__ loss,
                    float* __restrict__ weight, float* __restrict__ nonzero) {
  __shared__ float red[32];
  const int b = blockIdx.x, tid = threadIdx.x;
  const size_t off = (size_t)b * N;
  const float gs = grad_scale / temperature;
  float sl = 0.f, sw = 0.f, nz = 0.f;
  for (int i = tid; i < N; i += blockDim.x) {
    const float lab = labels[off + i];
    const bool lvalid = lab >= 0.f;
    const bool mvalid = mask ? (mask[off + i] != 0) : lvalid;
    float wv = 1.f;
    if (item_w) wv = w_per_item ? item_w[off + i] : item_w[b];
    const float w = (lvalid && mvalid) ? wv : 0.f;
    const float l = mvalid ? lab : 0.f;
    float f = 0.f;
    for (int k = 0; k < K; ++k) {
      const float z = mvalid ? scores[(off + i) * K + k] / temperature : 0.f;
      float o = l >= (float)(k + 1) ? 1.f : 0.f;
      if (use_fraction) {
        const float fr = l - (float)k;            // labels - one_to_n + 1
        if (fr > 0.f && fr < 1.f) o += fr;
      }
      if (!mvalid) o = 0.f;
      const float e = expf(-fabsf(z));
      const float ce = fmaxf(z, 0.f) - z * o + log1pf(e);
      f += mvalid ? ce : 0.f;
      if (grad) {
        const float sg = z >= 0.f ? 1.f / (1.f + e) : e / (1.f + e);
        grad[(off + i) * K + k] = mvalid ? (sg - o) * w * gs : 0.f;
      }
    }
    if (row) row[off + i] = f * w;
    sl += f * w;
    sw += w;
    nz += w != 0.f ? 1.f : 0.f;
  }
  sl = block_sum(sl, red);
  sw = block_sum(sw, red);
  nz = block_sum(nz, red);
  if (tid == 0) {
    loss[b] = sl;
    if (weight) weight[b] = sw;
    if (nonzero) nonzero[b] = nz;
  }
}

// ---------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------
template <typename K>
static int prep_smem(K kernel, size_t bytes) {
  if (bytes > 48 * 1024) {
    TFR_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)bytes));
  }
  return TFR_OK;
}

static int check_list_args(const void* scores, const void* labels, int B, int N,
                           float temperature) {
  TFR_REQUIRE(scores != nullptr && labels != nullptr, "scores/labels must not be NULL");
  TFR_REQUIRE(B >= 0 && N >= 1, "need batch_size >= 0 and list_size >= 1 (got B=%d N=%d)", B, N);
  TFR_REQUIRE(N <= kMaxListSize, "list_size %d exceeds the supported maximum %d", N, kMaxListSize);
  TFR_REQUIRE(temperature != 0.f, "temperature must be non-zero");
  return TFR_OK;
}

template <int PHI>
static int launch_pairwise(int lamkind, dim3 grid, size_t smem, cudaStream_t st,
                           const float* scores, const float* labels, const float* item_w,
                           int w_per_item, const uint8_t* mask, int N, float temperature,
                           LamDev lam, float grad_scale, float* grad, float* row_loss,
                           float* loss_sum, float* w_sum, float* nnz, int32_t* ranks_out) {
#define TFR_CASE(L)                                                                      \
  case L: {                                                                              \
    int rc = prep_smem(pairwise_loss_kernel<PHI, L>, smem);                              \
    if (rc) return rc;                                                                   \
    pairwise_loss_kernel<PHI, L><<<grid, kLossThreads, smem, st>>>(                      \
        scores, labels, item_w, w_per_item, mask, N, temperature, lam, grad_scale, grad, \
        row_loss, loss_sum, w_sum, nnz, ranks_out);                                      \
    break;                                                                               \
  }
  switch (lamkind) {
    TFR_CASE(TFR_LAMBDA_NONE)
    TFR_CASE(TFR_LAMBDA_LABEL_DIFF)
    TFR_CASE(TFR_LAMBDA_DCG)
    TFR_CASE(TFR_LAMBDA_DCG_V2)
    TFR_CASE(TFR_LAMBDA_YETI)
    TFR_CASE(TFR_LAMBDA_PRECISION)
    default:
      set_error("bad lambda kind %d", lamkind);
      return TFR_INVALID_ARGUMENT;
  }
#undef TFR_CASE
  TFR_LAUNCH_OK();
  return TFR_OK;
}

// pairwise_tri.cu
int launch_pairwise_tri(int phi, cudaStream_t st, const float* scores, const float* labels,
                        const float* item_w, int w_per_item, const uint8_t* mask, int B, int N,
                        float temperature, const LamDev& lam, float grad_scale, float* grad,
                        float* row_loss, float* loss_sum, float* w_sum, float* nnz,
                        int32_t* ranks_out);

}  // namespace tfr

using namespace tfr;

extern "C" int tfr_pairwise_loss_fwd_bwd(const float* scores, const float* labels,
                                         const float* item_w, int w_per_item,
                                         const uint8_t* mask, int B, int N,
                                         float temperature, int phi,
                                         const tfr_lambda_cfg* lam_host, float grad_scale,
                                         float* grad, float* row_loss, float* loss_sum,
                                         float* w_sum, float* nnz, int32_t* ranks_out,
                                         void* stream) {
  int rc = check_list_args(scores, labels, B, N, temperature);
  if (rc) return rc;
  TFR_REQUIRE(loss_sum != nullptr, "loss_sum must not be NULL");
  TFR_REQUIRE(phi >= TFR_PHI_LOGISTIC && phi <= TFR_PHI_MSE, "phi %d is not a tfr_phi", phi);
  rc = check_lam(lam_host);
  if (rc) return rc;
  if (B == 0) return TFR_OK;
  const LamDev lam = make_lam(lam_host);
  const size_t smem = list_smem_bytes(N);
  cudaStream_t st = (cudaStream_t)stream;
  // One phi evaluation per unordered pair (pairwise_tri.cu); the both-ends kernel below
  // keeps PairwiseMSELoss and N > 1024.
  if (phi != TFR_PHI_MSE && N <= 1024)
    return launch_pairwise_tri(phi, st, scores, labels, item_w, w_per_item, mask, B, N,
                               temperature, lam, grad_scale, grad, row_loss, loss_sum, w_sum,
                               nnz, ranks_out);
  dim3 grid(B);
#define TFR_PHI_CASE(P)                                                                   \
  case P:                                                                                 \
    return launch_pairwise<P>(lam.kind, grid, smem, st, scores, labels, item_w, w_per_item, \
                              mask, N, temperature, lam, grad_scale, grad, row_loss,      \
                              loss_sum, w_sum, nnz, ranks_out);
  switch (phi) {
    TFR_PHI_CASE(TFR_PHI_LOGISTIC)
    TFR_PHI_CASE(TFR_PHI_HINGE)
    TFR_PHI_CASE(TFR_PHI_SOFT_ZERO_ONE)
    TFR_PHI_CASE(TFR_PHI_MSE)
  }
#undef TFR_PHI_CASE
  return TFR_INVALID_ARGUMENT;
}

extern "C" int tfr_lambda_pair_weights(const float* labels, const int32_t* ranks, int B,
                                       int N, const tfr_lambda_cfg* lam_host, float* out,
                                       void* stream) {
  TFR_REQUIRE(labels && ranks && out && lam_host, "NULL argument");
  TFR_REQUIRE(B >= 0 && N >= 1 && N <= 1024, "pair weights helper needs 1 <= N <= 1024");
  int rc = check_lam(lam_host);
  if (rc) return rc;
  if (B == 0) return TFR_OK;
  const LamDev lam = make_lam(lam_host);
  const size_t smem = list_smem_bytes(N);
  cudaStream_t st = (cudaStream_t)stream;
#define TFR_CASE(L)                                                                   \
  case L: {                                                                           \
    rc = prep_smem(pair_weights_kernel<L>, smem);                                     \
    if (rc) return rc;                                                                \
    pair_weights_kernel<L><<<B, kLossThreads, smem, st>>>(labels, ranks, N, lam, out); \
    break;                                                                            \
  }
  switch (lam.kind) {
    TFR_CASE(TFR_LAMBDA_NONE)
    TFR_CASE(TFR_LAMBDA_LABEL_DIFF)
    TFR_CASE(TFR_LAMBDA_DCG)
    TFR_CASE(TFR_LAMBDA_DCG_V2)
    TFR_CASE(TFR_LAMBDA_YETI)
    TFR_CASE(TFR_LAMBDA_PRECISION)
  }
#undef TFR_CASE
  TFR_LAUNCH_OK();
  return TFR_OK;
}

extern "C" int tfr_sorted_ranks(const float* scores, const float* labels,
                                const uint8_t* mask, int B, int N, int32_t* ranks,
                                void* stream) {
  int rc = check_list_args(scores, labels, B, N, 1.f);
  if (rc) return rc;
  TFR_REQUIRE(ranks != nullptr, "ranks must not be NULL");
  if (B == 0) return TFR_OK;
  const size_t smem = list_smem_bytes(N);
  rc = prep_smem(sorted_ranks_kernel, smem);
  if (rc) return rc;
  sorted_ranks_kernel<<<B, kLossThreads, smem, (cudaStream_t)stream>>>(scores, labels, mask,
                                                                      N, ranks);
  TFR_LAUNCH_OK();
  return TFR_OK;
}

extern "C" int tfr_approx_loss_fwd_bwd(const float* scores, const float* labels,
                                       const float* item_w, int w_per_item,
                                       const uint8_t* mask, int B, int N, float temperature,
                                       int mode, float grad_scale, int scale_by_weight,
                                       float* grad, float* loss, float* weight,
                                       void* stream) {
  int rc = check_list_args(scores, labels, B, N, temperature);
  if (rc) return rc;
  TFR_REQUIRE(loss != nullptr, "loss must not be NULL");
  TFR_REQUIRE(mode == 0 || mode == 1, "mode must be 0 (NDCG) or 1 (MRR)");
  if (B == 0) return TFR_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int T = N <= 1024 ? (N + 31) / 32 : 0;
  // column partials of the triangular loop: [kLossThreads / 32][N] floats after `red`
  const size_t smem = ((list_smem_bytes(N) + 15) & ~(size_t)15) +
                      (T > 0 ? (size_t)(kLossThreads / 32) * N * 4 : 0);
#define TFR_APPROX_CASE(MODE_, T_)                                                          \
  {                                                                                         \
    rc = prep_smem(approx_loss_kernel<MODE_, T_>, smem);                                    \
    if (rc) return rc;                                                                      \
    approx_loss_kernel<MODE_, T_><<<B, (T_ > 0 && T_ <= 8) ? 224 : kLossThreads, smem, st>>>(                           \
        scores, labels, item_w, w_per_item, mask, N, temperature, grad_scale,               \
        scale_by_weight, grad, loss, weight);                                               \
  }
#define TFR_APPROX_T(MODE_)                                   \
  if (T == 0) TFR_APPROX_CASE(MODE_, 0)                       \
  else if (T <= 1) TFR_APPROX_CASE(MODE_, 1)                  \
  else if (T <= 2) TFR_APPROX_CASE(MODE_, 2)                  \
  else if (T <= 4) TFR_APPROX_CASE(MODE_, 4)                  \
  else if (T <= 7) TFR_APPROX_CASE(MODE_, 7)                  \
  else if (T <= 8) TFR_APPROX_CASE(MODE_, 8)                  \
  else if (T <= 16) TFR_APPROX_CASE(MODE_, 16)                \
  else TFR_APPROX_CASE(MODE_, 32)
  if (mode == 0) {
    TFR_APPROX_T(0)
  } else {
    TFR_APPROX_T(1)
  }
#undef TFR_APPROX_T
#undef TFR_APPROX_CASE
  TFR_LAUNCH_OK();
  return TFR_OK;
}

extern "C" int tfr_softmax_loss_fwd_bwd(const float* scores, const float* labels,
                                        const float* item_w, int w_per_item,
                                        const uint8_t* mask, int B, int N, float temperature,
                                        const tfr_lambda_cfg* lam_host, float grad_scale,
                                        int scale_by_weight, float* grad, float* loss,
                                        float* weight, void* stream) {
  int rc = check_list_args(scores, labels, B, N, temperature);
  if (rc) return rc;
  TFR_REQUIRE(loss != nullptr, "loss must not be NULL");
  rc = check_lam(lam_host);
  if (rc) return rc;
  if (B == 0) return TFR_OK;
  const LamDev lam = make_lam(lam_host);
  const size_t smem = list_smem_bytes(N);
  rc = prep_smem(softmax_loss_kernel, smem);
  if (rc) return rc;
  softmax_loss_kernel<<<B, kLossThreads, smem, (cudaStream_t)stream>>>(
      scores, labels, item_w, w_per_item, mask, N, temperature, lam, grad_scale,
      scale_by_weight, grad, loss, weight);
  TFR_LAUNCH_OK();
  return TFR_OK;
}

extern "C" int tfr_misc_loss_fwd_bwd(const float* scores, const float* labels,
                                     const float* item_w, int w_per_item, const uint8_t* mask,
                                     int B, int N, float temperature, int kind,
                                     const float* rank_weight, const float* order_scores,
                                     int topk, float grad_scale, float* grad, float* row,
                                     float* loss, float* weight, float* nonzero,
                                     void* stream) {
  int rc = check_list_args(scores, labels, B, N, temperature);
  if (rc) return rc;
  TFR_REQUIRE(loss != nullptr, "loss must not be NULL");
  TFR_REQUIRE(kind >= TFR_MISC_SIGMOID_CE && kind <= TFR_MISC_LIST_MLE,
              "kind %d is not a tfr_misc_loss", kind);
  TFR_REQUIRE((order_scores == nullptr && topk <= 0) || kind == TFR_MISC_LIST_MLE,
              "order_scores / topk apply to TFR_MISC_LIST_MLE only");
  if (B == 0) return TFR_OK;
  const size_t smem = ((list_smem_bytes(N) + 15) & ~(size_t)15) + kLossThreads * sizeof(float);
  cudaStream_t st = (cudaStream_t)stream;
#define TFR_MISC_CASE(K_)                                                                    \
  case K_:                                                                                   \
    rc = prep_smem(misc_loss_kernel<K_>, smem);                                              \
    if (rc) return rc;                                                                       \
    misc_loss_kernel<K_><<<B, kLossThreads, smem, st>>>(scores, labels, item_w, w_per_item,   \
                                                        mask, N, temperature, rank_weight,   \
                                                        order_scores, topk, grad_scale,      \
                                                        grad, row, loss, weight, nonzero);   \
    break;
  switch (kind) {
    TFR_MISC_CASE(TFR_MISC_SIGMOID_CE)
    TFR_MISC_CASE(TFR_MISC_MEAN_SQUARED)
    TFR_MISC_CASE(TFR_MISC_UNIQUE_SOFTMAX)
    TFR_MISC_CASE(TFR_MISC_LIST_MLE)
  }
#undef TFR_MISC_CASE
  TFR_LAUNCH_OK();
  return TFR_OK;
}

extern "C" int tfr_gumbel_sample(const float* scores, const float* labels, int B, int N,
                                 int sample_size, float temperature, uint64_t seed, int mode,
                                 float* out_logits, const float* grad_out, float* grad_scores,
                                 void* stream) {
  TFR_REQUIRE(mode == 0 || mode == 1, "mode must be 0 (GumbelSampler) or 1 (teacher labels)");
  TFR_REQUIRE(mode == 0 || !(grad_out || grad_scores),
              "the teacher mode has no gradient (labels are constants)");
  int rc = check_list_args(mode == 1 ? labels : scores, labels, B, N, temperature);
  if (rc) return rc;
  TFR_REQUIRE(sample_size >= 1 && sample_size <= 65535, "sample_size %d out of range", sample_size);
  TFR_REQUIRE(out_logits || (grad_out && grad_scores),
              "need out_logits (forward) or grad_out + grad_scores (backward)");
  if (B == 0) return TFR_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const float inv_t = 1.f / temperature;
  if (out_logits) {
    const size_t smem = (size_t)(N + 32) * 4;
    rc = prep_smem(gumbel_sample_fwd_kernel, smem);
    if (rc) return rc;
    gumbel_sample_fwd_kernel<<<dim3(sample_size, B), kLossThreads, smem, st>>>(
        scores, labels, N, sample_size, inv_t, seed, mode, out_logits);
    TFR_LAUNCH_OK();
  }
  if (grad_out && grad_scores) {
    const size_t smem = (size_t)(2 * N + 32) * 4;
    rc = prep_smem(gumbel_sample_bwd_kernel, smem);
    if (rc) return rc;
    gumbel_sample_bwd_kernel<<<B, kLossThreads, smem, st>>>(scores, labels, N, sample_size, inv_t,
                                                            seed, grad_out, grad_scores);
    TFR_LAUNCH_OK();
  }
  return TFR_OK;
}

extern "C" int tfr_ordinal_loss_fwd_bwd(const float* scores, const float* labels,
                                        const float* item_w, int w_per_item,
                                        const uint8_t* mask, int B, int N, int K,
                                        float temperature, int use_fraction_label,
                                        float grad_scale, float* grad, float* row, float* loss,
                                        float* weight, float* nonzero, void* stream) {
  int rc = check_list_args(scores, labels, B, N, temperature);
  if (rc) return rc;
  TFR_REQUIRE(K >= 1, "ordinal_size %d must be >= 1", K);
  TFR_REQUIRE(loss != nullptr, "loss must not be NULL");
  if (B == 0) return TFR_OK;
  ordinal_loss_kernel<<<B, kLossThreads, 0, (cudaStream_t)stream>>>(
      scores, labels, item_w, w_per_item, mask, N, K, temperature, use_fraction_label,
      grad_scale, grad, row, loss, weight, nonzero);
  TFR_LAUNCH_OK();
  return TFR_OK;
}

extern "C" int tfr_weighted_sum(const float* v, const float* w, int n, float scale,
                                float* out2, void* stream) {
  TFR_REQUIRE(v != nullptr && out2 != nullptr && n >= 0, "bad arguments");
  weighted_sum_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(v, w, n, scale, out2);
  TFR_LAUNCH_OK();
  return TFR_OK;
}
