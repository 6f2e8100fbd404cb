// tcgen05 (UMMA) bf16 GEMM engine for the scorer tower (TFR_PREC_BF16, BASELINE config 3).
//
//   * operands are staged global -> shared by TMA (cp.async.bulk.tensor.2d, 128-byte
//     swizzle: 64 bf16 per row) into a ring of stages guarded by mbarriers;
//   * one converged warp issues tcgen05.mma.cta_group::1.kind::f16 (bf16 x bf16 -> fp32,
//     M = 128, N <= 256, K = 16 per instruction); accumulators live in tensor memory;
//   * eight epilogue warps (two per TMEM lane quarter) drain the accumulators with
//     tcgen05.ld: bias / ReLU / 1-bit ReLU masks / column sums in registers, bf16 packing,
//     a 128B-swizzled staging tile and a TMA store; nothing else touches global memory.
//
// Two operand layouts (tc_gemm_bf16.cuh):
//   mn = 0  forward and dZ GEMMs: both operands K-major; one 128 x N output tile per work
//           item, accumulator double-buffered so the epilogue of tile i overlaps the main
//           loop of tile i + 1;
//   mn = 1  dW GEMMs (A^T B over the M = B*N rows of the batch): both operands MN-major
//           straight from their row-major storage; a work item owns a k range and ALL
//           (<= 2) 128-row blocks of the small output, so every A / dZ element is loaded
//           exactly once; fp32 partials per k range are reduced by mlp_reduce2.
// The kernel is persistent: one CTA per SM walks a static list of work items.
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2..9 = epilogue.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "tc_gemm_bf16.cuh"
#include "tc_host.h"
#include "tc_ptx.cuh"

namespace tfr {
namespace tcb {

using namespace tfr::tc;   // PTX helpers

constexpr int kEpiWarps = 8;
constexpr int kThreads = (2 + kEpiWarps) * 32;   // 320
constexpr int BM = 128;
constexpr int BK = 64;                 // bf16 elements per 128-byte swizzle span
constexpr int kATileBytes = BM * BK * 2;   // 16 KB per 128-row block
constexpr int kMaxStages = 6;
constexpr int kStagingBytes = 4096;    // per epilogue warp: 32 rows x 128 B

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// lane = row, x[j] = column j  ->  sum over the 32 rows of column `lane` (x is destroyed).
// Recursive halving: after the step with offset o a lane keeps the columns c with
// (c & o) == (lane & o); 31 shuffles in total.
__device__ __forceinline__ float colsum32(float (&x)[32], int lane) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int c = 0; c < o; ++c) {
      const float keep = up ? x[c + o] : x[c];
      const float send = up ? x[c] : x[c + o];
      x[c] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  return x[0];
}

struct KArgs {
  int GM, GN, GK;
  int n_umma, n_tiles, m_tiles, MT, m_groups, splits;
  int kb_per_split, nkb_total;
  int stages, b_tile_bytes;
  uint32_t acc_cols, nbuf, tmem_alloc_cols;
  int epi, act;
  const float* bias;
  int bias_cols;
  uint32_t* bits_out;
  const uint32_t* bits_in;
  float* colsum;
  int colsum_stride, colsum_cols;
  int c_rows_per_split;
};

template <bool MN>
__global__ void __launch_bounds__(kThreads, 1)
bf16_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmC, const KArgs args) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int MT = args.MT;
  const int a_bytes = MT * kATileBytes;
  const int stage_bytes = a_bytes + args.b_tile_bytes;
  const int S = args.stages;
  unsigned char* epi_smem = smem + static_cast<size_t>(S) * stage_bytes;
  float* cacc_base = reinterpret_cast<float*>(epi_smem + kEpiWarps * kStagingBytes);
  float* sbias = cacc_base + kEpiWarps * args.colsum_cols;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sbias + args.bias_cols);
  uint64_t* full = bars;
  uint64_t* empty = bars + kMaxStages;
  uint64_t* acc_full = bars + 2 * kMaxStages;
  uint64_t* acc_empty = bars + 2 * kMaxStages + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int items_per_z = args.m_groups * args.n_tiles;
  const int total_items = items_per_z * args.splits;
  const int item0 = (int)blockIdx.x;
  const int istep = (int)gridDim.x;

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmC);
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], kEpiWarps);   // one arrival per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, args.tmem_alloc_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto sA = [&](int s) { return smem + static_cast<size_t>(s) * stage_bytes; };
  auto sB = [&](int s) { return sA(s) + a_bytes; };
  auto decode = [&](int item, int& m0, int& n0, int& z, int& kb_begin, int& nkb) {
    z = item / items_per_z;
    const int r = item - z * items_per_z;
    m0 = (r / args.n_tiles) * MT * BM;
    n0 = (r % args.n_tiles) * args.n_umma;
    kb_begin = z * args.kb_per_split;
    const int kb_end = min(args.nkb_total, kb_begin + args.kb_per_split);
    nkb = max(kb_end - kb_begin, 0);
  };

  if (warp == 0) {
    // ------------------------------------------------------- TMA producer ----
    // Converged warp: lane 0 arms the stage barrier, every box of the stage is issued by its
    // own lane in one warp instruction (the dW layout has 2 MT + N / 64 boxes of 8 KB).
    {
      const uint32_t tx_bytes = a_bytes + args.b_tile_bytes;
      const int nA = MN ? 2 * MT : 1;
      const int nB = MN ? args.b_tile_bytes / 8192 : 1;
      uint32_t it = 0;
      for (int item = item0; item < total_items; item += istep) {
        int m0, n0, z, kb_begin, nkb;
        decode(item, m0, n0, z, kb_begin, nkb);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % S;
          const uint32_t ph = (it / S) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          if (lane == 0) mbar_expect_tx(&full[s], tx_bytes);
          __syncwarp();
          const int k0 = (kb_begin + kb) * BK;
          if (lane < nA) {
            if (!MN) tma_load_2d(sA(s), &tmA, &full[s], k0, m0);     // box {64 k, 128 rows}
            else tma_load_2d(sA(s) + lane * 8192, &tmA, &full[s], m0 + 64 * lane, k0);   // {64 m, 64 k}
          } else if (lane < nA + nB) {
            const int j = lane - nA;
            if (!MN) tma_load_2d(sB(s), &tmB, &full[s], k0, n0);     // box {64 k, n_umma rows}
            else tma_load_2d(sB(s) + j * 8192, &tmB, &full[s], n0 + 64 * j, k0);         // {64 n, 64 k}
          }
        }
      }
    }
  } else if (warp == 1) {
    // --------------------------------------------------------- MMA issuer ----
    // instruction descriptor: D fp32, A / B bf16, majorness, N >> 3, M >> 4
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) |
                           (static_cast<uint32_t>(MN) << 15) | (static_cast<uint32_t>(MN) << 16) |
                           (static_cast<uint32_t>(args.n_umma >> 3) << 17) |
                           (static_cast<uint32_t>(BM >> 4) << 24);
    // K-major: 128 B rows, 8-row atoms every 1024 B, a k step (16 bf16) = 32 B.
    // MN-major: rows = k (128 B = 64 m / n), 8-k atoms every 1024 B, the next 64 m / n at
    // LBO = 8192 B (the next TMA box), a k step (16 rows) = 2048 B.
    const uint32_t lbo = MN ? 8192u : 16u, sbo = 1024u;
    const uint32_t step16 = MN ? (2048u >> 4) : (32u >> 4);
    uint32_t it = 0, tcount = 0;
    for (int item = item0; item < total_items; item += istep, ++tcount) {
      int m0, n0, z, kb_begin, nkb;
      decode(item, m0, n0, z, kb_begin, nkb);
      const uint32_t ab = tcount % args.nbuf, aph = (tcount / args.nbuf) & 1;
      mbar_wait(&acc_empty[ab], aph ^ 1);
      tc_fence_after();
      const uint32_t tmem_d0 = tmem_base + ab * MT * args.acc_cols;
      for (int kb = 0; kb < nkb; ++kb, ++it) {
        const int s = it % S;
        const uint32_t ph = (it / S) & 1;
        mbar_wait(&full[s], ph);
        tc_fence_after();
        const int krem = args.GK - (kb_begin + kb) * BK;
        const int ksteps = krem >= BK ? BK / 16 : (krem + 15) / 16;
        const uint64_t db0 = make_smem_desc(smem_u32(sB(s)), lbo, sbo, 2u);
        for (int mt = 0; mt < MT; ++mt) {
          const uint64_t da0 = make_smem_desc(smem_u32(sA(s) + mt * kATileBytes), lbo, sbo, 2u);
          const uint32_t tmem_d = tmem_d0 + mt * args.acc_cols;
#pragma unroll 4
          for (int ks = 0; ks < ksteps; ++ks)
            umma_bf16(tmem_d, da0 + static_cast<uint64_t>(ks * step16),
                      db0 + static_cast<uint64_t>(ks * step16), idesc, (kb | ks) != 0 ? 1u : 0u);
        }
        umma_commit(&empty[s]);
      }
      if (nkb > 0) umma_commit(&acc_full[ab]);
      else if (lane == 0) mbar_arrive(&acc_full[ab]);
      __syncwarp();
    }
  } else {
    // ---------------------------------------------------- epilogue (warps 2..9)
    const int q = warp & 3;           // TMEM lane quarter this warp may access
    const int ew = warp - 2;          // 0..7
    // "accumulator drained" (all lanes call it at a warp-uniform point; one lane arrives)
    auto arrive_acc_empty = [&](uint32_t ab) {
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[ab]);
    };
    const int half = ew >> 2;         // which of the two warps of the quarter
    unsigned char* stg = epi_smem + ew * kStagingBytes;
    float* cacc = cacc_base + ew * args.colsum_cols;
    for (int c = lane; c < args.colsum_cols; c += 32) cacc[c] = 0.f;
    if (args.bias_cols) {
      for (int c = ew * 32 + lane; c < args.bias_cols; c += kEpiWarps * 32)
        sbias[c] = c < args.GN ? __ldg(args.bias + c) : 0.f;
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiWarps * 32) : "memory");
    }
    __syncwarp();
    uint32_t tcount = 0;
    for (int item = item0; item < total_items; item += istep, ++tcount) {
      int m0, n0, z, kb_begin, nkb;
      decode(item, m0, n0, z, kb_begin, nkb);
      const uint32_t ab = tcount % args.nbuf, aph = (tcount / args.nbuf) & 1;
      const uint32_t tmem_d0 = tmem_base + ab * MT * args.acc_cols +
                               (static_cast<uint32_t>(q * 32) << 16);
      if (!MN) {
        // bf16 row-major output: this warp owns rows m0 + 32 q .. + 31 and the 64-column
        // chunks c0 = 64 half, 64 half + 128, ...
        const int row0 = m0 + q * 32, row = row0 + lane;
        const bool warp_live = row0 < args.GM;
        int my_last = -1;
        for (int c0 = half * 64; c0 < args.n_umma && n0 + c0 < args.GN; c0 += 128) my_last = c0;
        auto load_bits = [&](int c0, int hh) -> uint32_t {
          const int col = n0 + c0 + 32 * hh;
          return (c0 <= my_last && col < args.GN && row < args.GM)
                     ? __ldg(args.bits_in + static_cast<size_t>(col >> 5) * args.GM + row)
                     : 0u;
        };
        uint32_t mw0 = 0, mw1 = 0;
        if (args.epi == EPI_MASK_BITS) {
          mw0 = load_bits(half * 64, 0);
          mw1 = load_bits(half * 64, 1);
        }
        mbar_wait(&acc_full[ab], aph);
        tc_fence_after();
        if (my_last < 0) {
          tc_fence_before();
          arrive_acc_empty(ab);
          continue;
        }
#pragma unroll 1
        for (int c0 = half * 64; c0 <= my_last; c0 += 128) {
          const int colb = n0 + c0;
          uint32_t v0[32], v1[32];
          tmem_ld32(tmem_d0 + c0, v0);
          tmem_ld32(tmem_d0 + c0 + 32, v1);
          uint32_t nw0 = 0, nw1 = 0;
          if (args.epi == EPI_MASK_BITS) {   // next chunk's words while the loads fly
            nw0 = load_bits(c0 + 128, 0);
            nw1 = load_bits(c0 + 128, 1);
          }
          tmem_ld_wait();
          if (c0 == my_last) {   // accumulator drained: the MMA warp may refill it
            tc_fence_before();
            arrive_acc_empty(ab);
          }
          float x0[32], x1[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            x0[j] = nkb > 0 ? __uint_as_float(v0[j]) : 0.f;
            x1[j] = nkb > 0 ? __uint_as_float(v1[j]) : 0.f;
          }
          uint32_t packed[32];
          if (args.epi == EPI_BIAS_ACT) {
            uint32_t w0 = 0, w1 = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 b0 = *reinterpret_cast<const float4*>(sbias + colb + 4 * j);
              const float4 b1 = *reinterpret_cast<const float4*>(sbias + colb + 32 + 4 * j);
              x0[4 * j + 0] += b0.x; x0[4 * j + 1] += b0.y;
              x0[4 * j + 2] += b0.z; x0[4 * j + 3] += b0.w;
              x1[4 * j + 0] += b1.x; x1[4 * j + 1] += b1.y;
              x1[4 * j + 2] += b1.z; x1[4 * j + 3] += b1.w;
            }
            if (args.act == TFR_ACT_RELU) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                x0[j] = fmaxf(x0[j], 0.f);
                x1[j] = fmaxf(x1[j], 0.f);
              }
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              packed[j] = pack_bf16(x0[2 * j], x0[2 * j + 1]);
              packed[16 + j] = pack_bf16(x1[2 * j], x1[2 * j + 1]);
            }
            if (args.bits_out) {
              // sign bits of the STORED bf16 values (post-ReLU: never negative; an fp32
              // denormal may round to 0, so the test is on the packed halves)
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                w0 |= ((packed[j] & 0x7FFFu) != 0 ? 1u : 0u) << (2 * j);
                w0 |= ((packed[j] & 0x7FFF0000u) != 0 ? 1u : 0u) << (2 * j + 1);
                w1 |= ((packed[16 + j] & 0x7FFFu) != 0 ? 1u : 0u) << (2 * j);
                w1 |= ((packed[16 + j] & 0x7FFF0000u) != 0 ? 1u : 0u) << (2 * j + 1);
              }
              if (args.GN - colb < 32) w0 &= (1u << (args.GN - colb)) - 1u;
              if (args.GN - colb - 32 < 32)
                w1 &= args.GN - colb - 32 > 0 ? (1u << (args.GN - colb - 32)) - 1u : 0u;
              if (row < args.GM) {
                args.bits_out[static_cast<size_t>(colb >> 5) * args.GM + row] = w0;
                if (colb + 32 < args.GN)
                  args.bits_out[static_cast<size_t>((colb >> 5) + 1) * args.GM + row] = w1;
              }
            }
          } else {
            if (args.epi == EPI_MASK_BITS) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                int m0b, m1b;
                asm("bfe.s32 %0, %1, %2, 1;" : "=r"(m0b) : "r"(mw0), "r"(j));
                asm("bfe.s32 %0, %1, %2, 1;" : "=r"(m1b) : "r"(mw1), "r"(j));
                x0[j] = __uint_as_float(__float_as_uint(x0[j]) & static_cast<uint32_t>(m0b));
                x1[j] = __uint_as_float(__float_as_uint(x1[j]) & static_cast<uint32_t>(m1b));
              }
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              packed[j] = pack_bf16(x0[2 * j], x0[2 * j + 1]);
              packed[16 + j] = pack_bf16(x1[2 * j], x1[2 * j + 1]);
            }
          }
          // the previous TMA store of this warp must have finished reading the tile
          if (lane == 0) bulk_wait_read0();
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<uint4*>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
          fence_proxy_async();
          __syncwarp();
          if (warp_live && lane == 0) {
            tma_store_2d(&tmC, stg, colb, row0);   // box {64 cols, 32 rows}; clipped at GN / GM
            bulk_commit();
          }
          if (args.colsum) {
            // fp32 column sums of what was stored (rows past GM hold zeros)
            const float s0 = colsum32(x0, lane);
            const float s1 = colsum32(x1, lane);
            if (colb + lane < args.colsum_cols) cacc[colb + lane] += s0;
            if (colb + 32 + lane < args.colsum_cols) cacc[colb + 32 + lane] += s1;
          }
          mw0 = nw0;
          mw1 = nw1;
        }
      } else {
        // fp32 partial output of a dW GEMM: 32-column chunks of every 128-row block,
        // alternating between the two warps of the quarter
        mbar_wait(&acc_full[ab], aph);
        tc_fence_after();
        const int nchunk = (args.n_umma + 31) >> 5;
        int my_last = -1;
        // (128-row blocks past GM — the second block of the last pair — are not stored: the
        // partial of a split is roundup(GM, 128) rows)
        for (int idx = half; idx < MT * nchunk; idx += 2)
          if (n0 + (idx % nchunk) * 32 < args.GN && m0 + (idx / nchunk) * BM < args.GM)
            my_last = idx;
        if (my_last < 0) {
          tc_fence_before();
          arrive_acc_empty(ab);
          continue;
        }
#pragma unroll 1
        for (int idx = half; idx <= my_last; idx += 2) {
          const int mt = idx / nchunk, c0 = (idx % nchunk) * 32;
          if (n0 + c0 >= args.GN || m0 + mt * BM >= args.GM) continue;
          uint32_t v[32];
          tmem_ld32(tmem_d0 + mt * args.acc_cols + c0, v);
          tmem_ld_wait();
          if (idx == my_last) {
            tc_fence_before();
            arrive_acc_empty(ab);
          }
          if (nkb == 0) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = 0u;
          }
          if (lane == 0) bulk_wait_read0();
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<uint4*>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tmC, stg, n0 + c0,
                         z * args.c_rows_per_split + m0 + mt * BM + q * 32);   // box {32, 32}
            bulk_commit();
          }
        }
      }
    }
    if (lane == 0) bulk_wait_all();
    if (args.colsum) {
      __syncwarp();
      float* dst = args.colsum + static_cast<size_t>(blockIdx.x * kEpiWarps + ew) * args.colsum_stride;
      for (int c = lane; c < args.GN; c += 32) dst[c] = cacc[c];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, args.tmem_alloc_cols);
}

// ------------------------------------------------------------------ host -------
// 2D tensor [outer rows][inner cols] of `esize`-byte elements (bf16 or fp32), 128B swizzle,
// box {box_inner (= 128 B), box_outer}.
static int encode_2d(CUtensorMap* tm, const void* ptr, int esize, uint64_t inner, uint64_t outer,
                     uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer) {
  return encode_tmap_2d(
      tm, esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, ptr,
      inner, outer, ld_elems * (uint64_t)esize, box_inner, box_outer, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <bool MN>
static int launch(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC,
                  const KArgs& ka, dim3 grid, size_t smem, cudaStream_t st) {
  auto kern = bf16_gemm_kernel<MN>;
  TFR_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, kThreads, smem, st>>>(tmA, tmB, tmC, ka);
  TFR_LAUNCH_OK();
  return TFR_OK;
}

int gemm(const GemmDesc& g, cudaStream_t st) {
  TFR_REQUIRE(g.A && g.B && g.C, "bf16 gemm: NULL operand");
  TFR_REQUIRE(g.GM >= 1 && g.GN >= 1 && g.GK >= 1, "bf16 gemm: empty problem");
  TFR_REQUIRE(g.lda % 8 == 0 && g.ldb % 8 == 0,
              "bf16 gemm: leading dimensions must be multiples of 8 elements");
  TFR_REQUIRE((reinterpret_cast<uintptr_t>(g.A) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(g.B) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(g.C) & 15) == 0,
              "bf16 gemm: operands must be 16-byte aligned");
  const bool mn = g.mn != 0;
  TFR_REQUIRE(mn ? g.ldc % 4 == 0 : g.ldc % 8 == 0, "bf16 gemm: ldc alignment");
  TFR_REQUIRE(g.epi == EPI_STORE || g.epi == EPI_BIAS_ACT || g.epi == EPI_MASK_BITS,
              "bf16 gemm: bad epilogue %d", g.epi);
  TFR_REQUIRE(!mn || g.epi == EPI_STORE, "bf16 gemm: dW layout only stores");
  TFR_REQUIRE(g.epi != EPI_BIAS_ACT || g.bias, "bf16 gemm: bias required");
  TFR_REQUIRE(g.epi != EPI_MASK_BITS || g.mask_bits_in, "bf16 gemm: mask_bits_in required");
  TFR_REQUIRE(!g.colsum || (!mn && g.GN <= 1024), "bf16 gemm: colsum needs mn = 0, GN <= 1024");
  TFR_REQUIRE(!g.mask_bits_out || (g.epi == EPI_BIAS_ACT && g.act == TFR_ACT_RELU),
              "bf16 gemm: sign bits are written by the bias + ReLU epilogue only");

  KArgs ka{};
  ka.GM = g.GM; ka.GN = g.GN; ka.GK = g.GK;
  const int n16 = (g.GN + 15) / 16 * 16;
  ka.n_umma = n16 <= 256 ? n16 : 256;
  ka.n_tiles = (g.GN + ka.n_umma - 1) / ka.n_umma;
  ka.m_tiles = (g.GM + BM - 1) / BM;
  ka.MT = mn ? (ka.m_tiles < 2 ? ka.m_tiles : 2) : 1;
  ka.m_groups = (ka.m_tiles + ka.MT - 1) / ka.MT;
  ka.splits = mn ? (g.splits < 1 ? 1 : g.splits) : 1;
  uint32_t acc_cols = 64;
  while ((int)acc_cols < ka.n_umma) acc_cols <<= 1;
  ka.acc_cols = acc_cols;
  ka.nbuf = (2u * ka.MT * acc_cols <= 512u) ? 2u : 1u;
  {
    uint32_t need = ka.nbuf * ka.MT * acc_cols, alloc = 32;
    while (alloc < need) alloc <<= 1;
    ka.tmem_alloc_cols = alloc;
  }
  ka.nkb_total = (g.GK + BK - 1) / BK;
  ka.kb_per_split = (ka.nkb_total + ka.splits - 1) / ka.splits;
  ka.b_tile_bytes = mn ? ((ka.n_umma + 63) / 64) * 8192 : ka.n_umma * 128;
  ka.epi = g.epi; ka.act = g.act; ka.bias = g.bias;
  ka.bias_cols = g.epi == EPI_BIAS_ACT ? ((ka.n_tiles * ka.n_umma + 63) / 64) * 64 + 64 : 0;
  ka.bits_out = g.mask_bits_out; ka.bits_in = g.mask_bits_in;
  ka.colsum = g.colsum; ka.colsum_stride = g.colsum_stride;
  ka.colsum_cols = g.colsum ? ((g.GN + 3) / 4) * 4 : 0;
  ka.c_rows_per_split = ka.m_tiles * BM;
  TFR_REQUIRE(!mn || g.splits <= 1 || g.split_stride >= (size_t)ka.c_rows_per_split * g.ldc,
              "bf16 gemm: split_stride must cover the padded partial (%d rows)",
              ka.c_rows_per_split);
  TFR_REQUIRE(!mn || g.splits <= 1 || g.split_stride == (size_t)ka.c_rows_per_split * g.ldc,
              "bf16 gemm: split_stride must equal roundup(GM, 128) * ldc");

  const int stage_bytes = ka.MT * kATileBytes + ka.b_tile_bytes;
  const size_t fixed = (size_t)kEpiWarps * kStagingBytes +
                       ((size_t)kEpiWarps * ka.colsum_cols + ka.bias_cols) * sizeof(float) +
                       256 /*barriers*/ + 1024 /*align*/;
  const size_t budget = 227 * 1024;
  int stages = (int)((budget - fixed) / stage_bytes);
  if (stages > kMaxStages) stages = kMaxStages;
  TFR_REQUIRE(stages >= 2, "bf16 gemm: tile does not fit shared memory");
  ka.stages = stages;

  CUtensorMap tmA, tmB, tmC;
  int rc;
  if (!mn) {
    rc = encode_2d(&tmA, g.A, 2, (uint64_t)g.GK, (uint64_t)g.GM, (uint64_t)g.lda, BK, BM);
    if (rc) return rc;
    rc = encode_2d(&tmB, g.B, 2, (uint64_t)g.GK, (uint64_t)g.GN, (uint64_t)g.ldb, BK,
                   (uint32_t)ka.n_umma);
    if (rc) return rc;
    rc = encode_2d(&tmC, g.C, 2, (uint64_t)g.GN, (uint64_t)g.GM, (uint64_t)g.ldc, 64, 32);
    if (rc) return rc;
  } else {
    rc = encode_2d(&tmA, g.A, 2, (uint64_t)g.GM, (uint64_t)g.GK, (uint64_t)g.lda, 64, BK);
    if (rc) return rc;
    rc = encode_2d(&tmB, g.B, 2, (uint64_t)g.GN, (uint64_t)g.GK, (uint64_t)g.ldb, 64, BK);
    if (rc) return rc;
    rc = encode_2d(&tmC, g.C, 4, (uint64_t)g.GN, (uint64_t)ka.splits * ka.c_rows_per_split,
                   (uint64_t)g.ldc, 32, 32);
    if (rc) return rc;
  }

  const int total_items = ka.m_groups * ka.n_tiles * ka.splits;
  const int sms = num_sms();
  dim3 grid(total_items < sms ? total_items : sms);
  const size_t smem = (size_t)stages * stage_bytes + fixed;
  if (g.colsum_slots_out) *g.colsum_slots_out = kEpiWarps * (int)grid.x;
  return mn ? launch<true>(tmA, tmB, tmC, ka, grid, smem, st)
            : launch<false>(tmA, tmB, tmC, ka, grid, smem, st);
}

}  // namespace tcb
}  // namespace tfr

// Test / parity entry: raw GEMM through the bf16 tensor-core engine (see tc_gemm_bf16.cuh).
extern "C" int tfr_tc_gemm_bf16(const void* A, int lda, const void* B, int ldb, void* C, int ldc,
                                int GM, int GN, int GK, int mn, int epi, const float* bias,
                                int act, uint32_t* mask_bits_out, const uint32_t* mask_bits_in,
                                float* colsum, int colsum_stride, int* colsum_slots_out,
                                int splits, size_t split_stride, void* stream) {
  tfr::tcb::GemmDesc g{};
  g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.C = C; g.ldc = ldc;
  g.GM = GM; g.GN = GN; g.GK = GK; g.mn = mn; g.epi = epi; g.bias = bias; g.act = act;
  g.mask_bits_out = mask_bits_out; g.mask_bits_in = mask_bits_in;
  g.colsum = colsum; g.colsum_stride = colsum_stride; g.colsum_slots_out = colsum_slots_out;
  g.splits = splits; g.split_stride = split_stride;
  return tfr::tcb::gemm(g, (cudaStream_t)stream);
}
