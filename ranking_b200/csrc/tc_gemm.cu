// tcgen05 (UMMA) TF32 GEMM engine for the scorer tower (sm_100a).
//
//   * operands are staged global -> shared by TMA (cp.async.bulk.tensor, 128-byte
//     swizzle) into a ring of stages guarded by mbarriers;
//   * one converged warp issues tcgen05.mma.kind::tf32 (elect.sync picks the lane) with the
//     fp32 accumulator tile [128 x N] living in TMEM;
//   * for the fp32-faithful mode (3xTF32) eight "splitter" warps turn each landed fp32 tile
//     into a round-to-nearest TF32 hi part and an fp32 lo residual, so that
//     D = Ahi*Bhi + Alo*Bhi + Ahi*Blo carries ~22 mantissa bits.  K-major A operands are
//     written straight into tensor memory (tcgen05.st) and read from there by the MMAs;
//     MN-major operands are split in place in shared memory;
//   * eight epilogue warps (two per TMEM lane quarter) drain the accumulators with
//     tcgen05.ld: bias / ReLU / 1-bit ReLU masks / column sums in registers, a swizzled
//     staging tile and a TMA store for row-major outputs; STG paths for the transposed and
//     split-K partial stores of the dW GEMMs.
//
// The kernel is persistent: one CTA per SM walks a static list of output tiles.
// Warp roles (576 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA
// issuer, warps 2..9 = hi/lo splitters, warps 10..17 = epilogue.  The accumulator is
// double-buffered in TMEM, so the epilogue of tile i overlaps the main loop of
// tile i+1 and the prologue (barrier init, TMEM allocation) is paid once per SM.
#include <cuda.h>

#include "common.cuh"
#include "tc_gemm.cuh"
#include "tc_host.h"
#include "tc_ptx.cuh"

namespace tfr {
namespace tc {

constexpr int kSplitWarps = 8;
constexpr int kSplitThreads = kSplitWarps * 32;
constexpr int kEpiWarp0 = 2 + kSplitWarps;          // first epilogue warp
constexpr int kEpiWarps = 8;                        // two per TMEM lane quarter
constexpr int kThreads = (kEpiWarp0 + kEpiWarps) * 32;   // 576
constexpr int kEpiSmemBytes = 4 * 32 * 37 * 4;   // fallback stores (4 warps): transpose buffers
constexpr int kEpiSmemBytes2 = kEpiWarps * 4096; // TMA-store path: one staging tile per warp
constexpr int BM = 128;       // UMMA M (cta_group::1)
constexpr int BK = 32;        // fp32 elements per 128-byte swizzle span = k of one stage
constexpr int kATileBytes = BM * BK * 4;   // 16 KB
constexpr int kBoxBytes = BK * 128;        // one MN-major TMA box: [32 k rows][128 B]
constexpr int kMaxStages = 4;
constexpr int kMaxN = 256;    // widest UMMA N: wider outputs are cut into tiles of 256

struct KernelArgs {
  float* C;
  int ldc;
  int GM, GN, GK;
  int n_umma;          // UMMA N of one tile (multiple of 16, <= 256)
  int a_tile_bytes;    // bytes of one A stage tile (hi part) = 128 * BK * 4
  int b_tile_bytes;    // bytes of one B stage tile (hi part)
  int stages;
  int epi, act, store_transposed;
  const float* bias;
  const float* aux;
  int kb_per_split;    // k-blocks (of 32) handled by one k split
  int m_tiles, n_tiles, splits;
  size_t split_stride;
  uint32_t tmem_cols;
  float* colsum;       // optional [4 * gridDim.x][colsum_stride]: column sums of everything
  int colsum_stride;   //   this CTA stored, per 32-row quarter (bias gradients)
  int colsum_cols;     // GN rounded up to 4 (0 when colsum is off): smem accumulators
  long long* dbg;      // optional [gridDim.x][12] wait-cycle counters per warp role
  int vec_ok;          // C / aux / bias / colsum allow 16-byte vector access
  int tma_store;       // row-major unsplit output: epilogue stores 32x32 blocks by TMA
  int epi_smem_bytes;  // bytes of the epilogue staging region
  int colsum_regs;     // column sums kept in registers (single n tile, tma_store)
  int bias_cols;       // floats of the bias copy staged in smem (tma_store + EPI_BIAS_ACT)
  int a_tmem;          // 3xTF32, K-major A: the splitters write A_hi / A_lo to tensor memory
                       //   and the MMAs read A from there (halves the smem operand traffic)
  uint32_t a_col0;     // first TMEM column of the A region: stage s at a_col0 + 64 s
  uint32_t acc_bufs;   // accumulator buffers in TMEM (2: epilogue overlaps the next tile;
                       //   1: long split-K tiles whose A stages need the columns)
  uint32_t tmem_alloc_cols;   // power of two >= 2 * tmem_cols (+ 64 * stages with a_tmem)
  uint32_t* bits_out;        // optional (tma_store): ReLU sign bits of the stored values,
  const uint32_t* bits_in;   //   word [(col / 32) * GM + row]; EPI_MASK_BITS reads them
};

// CG2: CTA pairs (cluster of 2, tcgen05 cta_group::2).  Only for K-major A through tensor
// memory with pre-split K-major B (the forward and dZ GEMMs): the pair owns 256 rows, each
// CTA stages its 128 rows of A and its HALF of the B tile, so the bytes a CTA pulls per k
// block drop from 16 + 2 * 128 N to 16 + 128 N KB (the per-SM ingest rate, ~35-40 B / cycle,
// is what bounds these kernels: profiles/r02_tc_gemm_wait_cycles.txt) and the stage shrinks
// enough for a 4-deep ring at N = 256.
// FAST_EPI >= 0 fixes the epilogue at compile time (row-major TMA-store path only): 1 = bias +
// ReLU (+ sign bits), 3 = ReLU mask from sign bits (+ column sums).  The generic kernel keeps
// every store path alive in one function, which costs the hot loop registers (96 per thread
// with 18 warps) — the forward / dZ GEMMs are bound by exactly that loop.
template <bool A_MN, bool B_MN, int PASSES, bool SPLIT_B, bool CG2 = false, int FAST_EPI = -1>
// (18 warps: ptxas grants 96 registers per thread; 112 was tried with __maxnreg__ and the
//  launch fails with "too many resources" — the per-warp allocation step does not fit)
__global__ void __launch_bounds__(kThreads, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmBlo, const __grid_constant__ CUtensorMap tmC,
               const KernelArgs args) {
  constexpr bool kFastOuter = FAST_EPI >= 0;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // 1024-byte alignment is required by the 128B swizzle atoms.
  // (pointer arithmetic, not an integer round trip: keeps the shared address space so
  // the compiler emits LDS/STS and knows these never alias global memory)
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int kACopies = (PASSES == 3 && !args.a_tmem) ? 2 : 1;
  constexpr int kBCopies = PASSES == 3 ? 2 : 1;
  const int a_bytes = args.a_tile_bytes * kACopies;
  const int stage_bytes = a_bytes + args.b_tile_bytes * kBCopies;
  const int S = args.stages;
  unsigned char* epi_smem = smem + static_cast<size_t>(S) * stage_bytes;   // 4 x [32][33] floats
  float* cacc_base = reinterpret_cast<float*>(epi_smem + args.epi_smem_bytes);   // [4][colsum_cols]
  float* sbias = cacc_base + kEpiWarps * args.colsum_cols;                       // [bias_cols]
  uint64_t* bars = reinterpret_cast<uint64_t*>(
      epi_smem + args.epi_smem_bytes +
      (kEpiWarps * args.colsum_cols + args.bias_cols) * sizeof(float));
  uint64_t* full = bars;                         // TMA landed
  uint64_t* split = bars + kMaxStages;           // hi/lo split done
  uint64_t* empty = bars + 2 * kMaxStages;       // MMAs that read the stage retired
  uint64_t* acc_full = bars + 3 * kMaxStages;    // [2] accumulator buffer complete
  uint64_t* acc_empty = bars + 3 * kMaxStages + 2;   // [2] accumulator buffer drained
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * kMaxStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb_total = (args.GK + BK - 1) / BK;
  const uint32_t rank = CG2 ? cluster_ctarank() : 0u;
  const int tiles_mn = (CG2 ? (args.m_tiles + 1) / 2 : args.m_tiles) * args.n_tiles;
  const int total_tiles = tiles_mn * args.splits;
  const int tile0 = CG2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;   // pairs share a tile list
  const int tstep = CG2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if (PASSES == 3 && !SPLIT_B) prefetch_tmap(&tmBlo);
    if (args.tma_store) prefetch_tmap(&tmC);
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      // pairs: the leader's barrier collects the splitter warps of both CTAs
      mbar_init(&split[s], CG2 ? 2 * kSplitWarps : kSplitWarps);
      mbar_init(&empty[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], (CG2 ? 2 : 1) * kEpiWarps);   // one arrival per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    if (CG2) {
      tmem_alloc2(tmem_slot, args.tmem_alloc_cols);
      tmem_relinquish2();
    } else {
      tmem_alloc(tmem_slot, args.tmem_alloc_cols);   // two accumulator buffers (+ A stages)
      tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CG2) cluster_sync_all();   // the peer's barriers are initialised before anyone arrives
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto sA_hi = [&](int s) { return smem + static_cast<size_t>(s) * stage_bytes; };
  auto sA_lo = [&](int s) { return sA_hi(s) + args.a_tile_bytes; };
  auto sB_hi = [&](int s) { return sA_hi(s) + a_bytes; };
  auto sB_lo = [&](int s) { return sB_hi(s) + args.b_tile_bytes; };
  // tile -> (split z, m tile, n tile): consecutive CTAs work on neighbouring rows.
  auto decode = [&](int tile, int& m0, int& n0, int& z, int& kb_begin, int& nkb) {
    z = tile / tiles_mn;
    const int r = tile - z * tiles_mn;
    m0 = CG2 ? (r / args.n_tiles) * 2 * BM + (int)rank * BM : (r / args.n_tiles) * BM;
    n0 = (r % args.n_tiles) * args.n_umma;
    kb_begin = z * args.kb_per_split;
    const int kb_end = min(nkb_total, kb_begin + args.kb_per_split);
    nkb = max(kb_end - kb_begin, 0);
  };

  if (warp == 0) {
    // ------------------------------------------------------- TMA producer ----
    // The warp stays converged: lane 0 arms the stage barrier, then every TMA box of the
    // stage is issued by its own lane in ONE warp instruction (a K-major tile is a single
    // box; an MN-major tile is one 4 KB box per 32 columns, up to 4 + 8 + 8 boxes per stage).
    // Issued one after the other by a single thread the boxes cost ~120-140 cycles each,
    // which made the producer the bottleneck of every GEMM with an MN-major operand.
    {
      const uint32_t tx_bytes =
          args.a_tile_bytes + args.b_tile_bytes * ((PASSES == 3 && !SPLIT_B) ? 2 : 1);
      const int nA = A_MN ? BM / 32 : 1;
      const int nB = B_MN ? args.b_tile_bytes / kBoxBytes : 1;
      const int nBlo = (PASSES == 3 && !SPLIT_B) ? nB : 0;
      uint32_t it = 0;
      long long w_empty = 0;
      const long long t_start = clock64();
      for (int tile = tile0; tile < total_tiles; tile += tstep) {
        int m0, n0, z, kb_begin, nkb;
        decode(tile, m0, n0, z, kb_begin, nkb);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % S;
          const uint32_t ph = (it / S) & 1;
          w_empty += mbar_wait(&empty[s], ph ^ 1);
          if (lane == 0) mbar_expect_tx(&full[s], tx_bytes);
          __syncwarp();
          const int k0 = (kb_begin + kb) * BK;
          if (lane < nA) {
            if (!A_MN) tma_load_2d(sA_hi(s), &tmA, &full[s], k0, m0);      // box [128 rows][32 k]
            else tma_load_2d(sA_hi(s) + lane * kBoxBytes, &tmA, &full[s], m0 + 32 * lane, k0);
          } else if (lane < nA + nB) {
            const int j = lane - nA;
            // (pairs: box [N / 2 rows][32 k], this CTA's half of the tile)
            if (!B_MN) tma_load_2d(sB_hi(s), &tmB, &full[s], k0,
                                   n0 + (CG2 ? (int)rank * (args.n_umma >> 1) : 0));
            else tma_load_2d(sB_hi(s) + j * kBoxBytes, &tmB, &full[s],
                             n0 + (CG2 ? (int)rank * (args.n_umma >> 1) : 0) + 32 * j, k0);
          } else if (lane < nA + nB + nBlo) {
            const int j = lane - nA - nB;
            if (!B_MN) tma_load_2d(sB_lo(s), &tmBlo, &full[s], k0,
                                   n0 + (CG2 ? (int)rank * (args.n_umma >> 1) : 0));
            else tma_load_2d(sB_lo(s) + j * kBoxBytes, &tmBlo, &full[s], n0 + 32 * j, k0);
          }
        }
      }
      if (args.dbg && lane == 0) {
        args.dbg[blockIdx.x * 12 + 0] = w_empty;
        args.dbg[blockIdx.x * 12 + 1] = clock64() - t_start;
      }
    }
  } else if (warp == 1) {
    // --------------------------------------------------------- MMA issuer ----
    if (!CG2 || rank == 0) {   // pairs: the leader issues for both CTAs
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) |
                             (static_cast<uint32_t>(A_MN && !args.a_tmem) << 15) |
                             (static_cast<uint32_t>(B_MN) << 16) |
                             (static_cast<uint32_t>(args.n_umma >> 3) << 17) |
                             (static_cast<uint32_t>((CG2 ? 2 * BM : BM) >> 4) << 24);
      const uint32_t a_step = A_MN ? 1024u : 32u;   // bytes per UMMA K step (8 fp32)
      const uint32_t b_step = B_MN ? 1024u : 32u;
      const uint32_t a_lbo = A_MN ? (uint32_t)kBoxBytes : 16u;
      const uint32_t b_lbo = B_MN ? (uint32_t)kBoxBytes : 16u;
      const uint32_t a_sbo = A_MN ? 512u : 1024u, b_sbo = B_MN ? 512u : 1024u;
      const uint32_t a_lt = A_MN ? 1u : 2u, b_lt = B_MN ? 1u : 2u;
      uint32_t it = 0, tcount = 0;
      long long w_acc = 0, w_full = 0;
      const long long t_start = clock64();
      for (int tile = tile0; tile < total_tiles; tile += tstep, ++tcount) {
        int m0, n0, z, kb_begin, nkb;
        decode(tile, m0, n0, z, kb_begin, nkb);
        const uint32_t ab = tcount % args.acc_bufs, aph = (tcount / args.acc_bufs) & 1;
        const long long th0 = args.dbg ? clock64() : 0;
        mbar_wait(&acc_empty[ab], aph ^ 1);   // epilogue has drained this buffer
        tc_fence_after();
        if (args.dbg) w_acc += clock64() - th0;
        const uint32_t tmem_d = tmem_base + ab * args.tmem_cols;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % S;
          const uint32_t ph = (it / S) & 1;
          const long long tw0 = args.dbg ? clock64() : 0;
          mbar_wait(PASSES == 3 ? &split[s] : &full[s], ph);
          tc_fence_after();
          if (args.dbg) w_full += clock64() - tw0;
          const uint32_t a_hi = smem_u32(sA_hi(s)), a_lo = smem_u32(sA_lo(s));
          const uint32_t b_hi = smem_u32(sB_hi(s)), b_lo = smem_u32(sB_lo(s));
          // descriptors of the stage once; a k step only adds (bytes >> 4) to the address field
          const uint64_t da_hi0 = make_smem_desc(a_hi, a_lbo, a_sbo, a_lt);
          const uint64_t da_lo0 = make_smem_desc(a_lo, a_lbo, a_sbo, a_lt);
          const uint64_t db_hi0 = make_smem_desc(b_hi, b_lbo, b_sbo, b_lt);
          const uint64_t db_lo0 = make_smem_desc(b_lo, b_lbo, b_sbo, b_lt);
          // the last k block of a K that is no multiple of 32 holds zeros past K (TMA fill):
          // skip the all-zero k steps
          const int krem = args.GK - (kb_begin + kb) * BK;
          const int ksteps = krem >= BK ? BK / 8 : (krem + 7) / 8;
          if (PASSES == 3 && args.a_tmem) {
            // A_hi / A_lo sit in tensor memory (written by the splitters)
            const uint32_t ta_hi = tmem_base + args.a_col0 + static_cast<uint32_t>(s) * 64u;
            const uint32_t ta_lo = ta_hi + 32u;
#pragma unroll 4
            for (int ks = 0; ks < ksteps; ++ks) {
              const uint64_t db_hi = db_hi0 + static_cast<uint64_t>(ks * (b_step >> 4));
              const uint64_t db_lo = db_lo0 + static_cast<uint64_t>(ks * (b_step >> 4));
              if (CG2) {
                umma_tf32_ts_cg2(tmem_d, ta_hi + ks * 8, db_hi, idesc, (kb | ks) != 0 ? 1u : 0u);
                umma_tf32_ts_cg2(tmem_d, ta_lo + ks * 8, db_hi, idesc, 1u);
                umma_tf32_ts_cg2(tmem_d, ta_hi + ks * 8, db_lo, idesc, 1u);
              } else {
                umma_tf32_ts(tmem_d, ta_hi + ks * 8, db_hi, idesc, (kb | ks) != 0 ? 1u : 0u);
                umma_tf32_ts(tmem_d, ta_lo + ks * 8, db_hi, idesc, 1u);
                umma_tf32_ts(tmem_d, ta_hi + ks * 8, db_lo, idesc, 1u);
              }
            }
            if (CG2) umma_commit_cg2(&empty[s]);   // frees the stage in both CTAs
            else umma_commit(&empty[s]);
            continue;
          }
#pragma unroll 4
          for (int ks = 0; ks < ksteps; ++ks) {
            const uint64_t da_hi = da_hi0 + static_cast<uint64_t>(ks * (a_step >> 4));
            const uint64_t db_hi = db_hi0 + static_cast<uint64_t>(ks * (b_step >> 4));
            if (CG2) umma_tf32_cg2(tmem_d, da_hi, db_hi, idesc, (kb | ks) != 0 ? 1u : 0u);
            else umma_tf32(tmem_d, da_hi, db_hi, idesc, (kb | ks) != 0 ? 1u : 0u);
            if (PASSES == 3) {
              const uint64_t da_lo = da_lo0 + static_cast<uint64_t>(ks * (a_step >> 4));
              const uint64_t db_lo = db_lo0 + static_cast<uint64_t>(ks * (b_step >> 4));
              if (CG2) {
                umma_tf32_cg2(tmem_d, da_lo, db_hi, idesc, 1u);
                umma_tf32_cg2(tmem_d, da_hi, db_lo, idesc, 1u);
              } else {
                umma_tf32(tmem_d, da_lo, db_hi, idesc, 1u);
                umma_tf32(tmem_d, da_hi, db_lo, idesc, 1u);
              }
            }
          }
          if (CG2) umma_commit_cg2(&empty[s]);
          else umma_commit(&empty[s]);   // frees the stage once these MMAs have read it
        }
        if (CG2) umma_commit_cg2(&acc_full[ab]);          // (pairs never see an empty k range)
        else if (nkb > 0) umma_commit(&acc_full[ab]);
        else if (lane == 0) mbar_arrive(&acc_full[ab]);   // empty k range: epilogue stores zeros
        __syncwarp();
      }
      if (args.dbg && lane == 0) {
        args.dbg[blockIdx.x * 12 + 2] = w_acc;
        args.dbg[blockIdx.x * 12 + 3] = w_full;
        args.dbg[blockIdx.x * 12 + 4] = clock64() - t_start;
      }
    }
  } else if (warp < kEpiWarp0) {
    // ------------------------------------------------ hi/lo splitters (warps 2..9)
    if (PASSES == 3) {
      const int t = threadIdx.x - 64;   // 0 .. kSplitThreads - 1
      const int b_chunks = SPLIT_B ? args.b_tile_bytes / 16 : 0;
      uint32_t it = 0;
      long long w_tma = 0;
      for (int tile = tile0; tile < total_tiles; tile += tstep) {
        int m0, n0, z, kb_begin, nkb;
        decode(tile, m0, n0, z, kb_begin, nkb);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % S;
          const uint32_t ph = (it / S) & 1;
          w_tma += mbar_wait(&full[s], ph);
          if (!A_MN && !SPLIT_B && args.a_tmem) {
            // lane = row of the K-major tile; the two warps of a TMEM lane quarter take
            // 16 of the 32 k columns each: 4 swizzled LDS.128 -> hi/lo -> 2 tcgen05.st.x16
            const int q = warp & 3, hsel = (warp - 2) >> 2;
            const int row = q * 32 + lane;
            const unsigned char* src = sA_hi(s) + row * 128;
            uint32_t h[16], l[16];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
              const int j = hsel * 4 + jj;
              const float4 v4 = *reinterpret_cast<const float4*>(src + ((j ^ (row & 7)) << 4));
              const float xs[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float hh = tf32_rn(xs[e]);
                h[jj * 4 + e] = __float_as_uint(hh);
                l[jj * 4 + e] = __float_as_uint(xs[e] - hh);
              }
            }
            const uint32_t ta = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + args.a_col0 +
                                static_cast<uint32_t>(s) * 64u + hsel * 16u;
            tmem_st16(ta, h);
            tmem_st16(ta + 32u, l);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (CG2) mbar_arrive_cluster(mapa_u32(&split[s], 0));   // the leader's barrier
              else mbar_arrive(&split[s]);
            }
            continue;
          }
          if (A_MN && args.a_tmem) {
            // MN-major A (rows = k, 128 B = 32 m per box): the warps of TMEM lane quarter q
            // own box q; lane = m, so the transpose into tensor memory (lane = row of A^T,
            // column = k) is free.  32 B chunks are XOR-ed with (k % 4) by the 32 B-atom
            // swizzle.  Each of the two warps of a quarter takes 16 of the 32 k rows.
            const int q = warp & 3, hsel = (warp - 2) >> 2;
            const unsigned char* box = sA_hi(s) + q * kBoxBytes + ((lane & 7) << 2);
            const int c32 = lane >> 3;
            uint32_t h[16], l[16];
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
              const int k = hsel * 16 + jj;
              const float x = *reinterpret_cast<const float*>(box + k * 128 + ((c32 ^ (k & 3)) << 5));
              const float hh = tf32_rn(x);
              h[jj] = __float_as_uint(hh);
              l[jj] = __float_as_uint(x - hh);
            }
            const uint32_t ta = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + args.a_col0 +
                                static_cast<uint32_t>(s) * 64u + hsel * 16u;
            tmem_st16(ta, h);
            tmem_st16(ta + 32u, l);
          }
          float4* __restrict__ hi = reinterpret_cast<float4*>(sA_hi(s));
          float4* __restrict__ lo = reinterpret_cast<float4*>(sA_lo(s));
          for (int pass = (A_MN && args.a_tmem) ? 1 : 0; pass < (SPLIT_B ? 2 : 1); ++pass) {
            const int chunks = pass == 0 ? args.a_tile_bytes / 16 : b_chunks;
            if (pass == 1) {
              hi = reinterpret_cast<float4*>(sB_hi(s));
              lo = reinterpret_cast<float4*>(sB_lo(s));
            }
            // 4 independent 16-byte loads in flight per thread, then convert + store
            for (int c = t; c < chunks; c += 4 * kSplitThreads) {
              float4 v[4];
#pragma unroll
              for (int u = 0; u < 4; ++u)
                if (c + u * kSplitThreads < chunks) v[u] = hi[c + u * kSplitThreads];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                if (c + u * kSplitThreads < chunks) {
                  float4 h, l;
                  h.x = tf32_rn(v[u].x);
                  h.y = tf32_rn(v[u].y);
                  h.z = tf32_rn(v[u].z);
                  h.w = tf32_rn(v[u].w);
                  l.x = v[u].x - h.x;
                  l.y = v[u].y - h.y;
                  l.z = v[u].z - h.z;
                  l.w = v[u].w - h.w;
                  hi[c + u * kSplitThreads] = h;
                  lo[c + u * kSplitThreads] = l;
                }
              }
            }
          }
          if (A_MN && args.a_tmem) {
            tmem_st_wait();
            tc_fence_before();
          }
          fence_proxy_async();       // generic-proxy writes -> visible to the tensor core
          __syncwarp();
          if (lane == 0) {                          // one arrival per splitter warp
            if (CG2) mbar_arrive_cluster(mapa_u32(&split[s], 0));
            else mbar_arrive(&split[s]);
          }
        }
      }
      if (args.dbg && t == 0) args.dbg[blockIdx.x * 12 + 5] = w_tma;
    }
  } else {
    // ---------------------------------------------------- epilogue (warps 10..17)
    // TMEM lane quarter is fixed by warp id % 4; the two warps of a quarter take
    // alternate 32-column chunks (TMA-store mode; the single-warp epilogue is
    // instruction/latency-bound at ~2k cycles per chunk).  The fallback stores
    // (transposed / split-K partials: one store per long k loop) use warps 0..3 only.
    // While these warps drain buffer `ab`, the MMA warp already fills the other one.
    const int q = warp & 3;
    const int ew = warp - kEpiWarp0;          // 0..7
    // "accumulator drained": to the MMA issuer's barrier — the leader's in a pair
    // (called by all lanes at a warp-uniform point, after their tcgen05.wait::ld and
    //  tcgen05.fence::before_thread_sync; one lane arrives for the warp.  A remote arrival
    //  per THREAD cost the peer ~5 k cycles per tile: profiles/README.md, round 2.)
    auto arrive_acc_empty = [&](uint32_t ab) {
      __syncwarp();
      if (lane == 0) {
        if (CG2) mbar_arrive_cluster(mapa_u32(&acc_empty[ab], 0));
        else mbar_arrive(&acc_empty[ab]);
      }
    };
    const int half = ew >> 2;                 // which of the two warps of the quarter
    constexpr bool kFast = FAST_EPI >= 0;
    // FAST_EPI 0 / 1 / 3: TMA-store path with that epilogue; 4: the other store paths only
    // (transposed / split-K partials of the dW GEMMs), plain store
    const bool tma_store = kFast ? (FAST_EPI != 4) : (args.tma_store != 0);
    const int epi = kFast ? (FAST_EPI == 4 ? (int)EPI_STORE : FAST_EPI) : args.epi;
    const int act = FAST_EPI == 1 ? (int)TFR_ACT_RELU : args.act;
    float* tb = reinterpret_cast<float*>(epi_smem) + (ew & 3) * (32 * 37);
    // per-warp running column sums over all tiles of this CTA (one slot per CTA and
    // quarter instead of one per tile: 592 slots to reduce instead of 6400)
    float* cacc = cacc_base + ew * args.colsum_cols;
    for (int c = lane; c < args.colsum_cols; c += 32) cacc[c] = 0.f;
    __syncwarp();
    if (args.bias_cols) {   // bias copy, zero past GN; named barrier over the epilogue warps
      for (int c = ew * 32 + lane; c < args.bias_cols; c += kEpiWarps * 32)
        sbias[c] = c < args.GN ? __ldg(args.bias + c) : 0.f;
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiWarps * 32) : "memory");
    }
    uint32_t tcount = 0;
    // register column sums (colsum_regs mode): this warp only sees the chunks of its
    // parity, so slot j holds chunk 2 j + half; lane = column within the chunk
    float ccol[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) ccol[k] = 0.f;
    // wait-cycle counters of the profiling build live in shared memory: as registers they
    // stayed live across the whole epilogue loop and pushed its operands onto the stack
    long long* s_dbg = reinterpret_cast<long long*>(bars + 3 * kMaxStages + 6);   // [5]
    const bool dbg_me = args.dbg != nullptr && threadIdx.x == kEpiWarp0 * 32;
    if (dbg_me) {
#pragma unroll
      for (int i = 0; i < 5; ++i) s_dbg[i] = 0;
    }
    const long long t_start = args.dbg ? clock64() : 0;
    for (int tile = tile0; tile < total_tiles; tile += tstep, ++tcount) {
      int m0, n0, z, kb_begin, nkb;
      decode(tile, m0, n0, z, kb_begin, nkb);
      const uint32_t ab = tcount % args.acc_bufs, aph = (tcount / args.acc_bufs) & 1;
      // ReLU sign bits of this warp's 32 rows (one word per row and 32-column chunk);
      // the first chunk's word is fetched before the accumulator is even complete, the
      // following ones one chunk ahead.
      auto load_bits = [&](int c0) -> uint32_t {
        const int col = n0 + c0, row = m0 + q * 32 + lane;
        return (c0 < args.n_umma && col < args.GN && row < args.GM)
                   ? __ldg(args.bits_in + static_cast<size_t>(col >> 5) * args.GM + row)
                   : 0u;
      };
      uint32_t mword = 0, mword_next = 0;
      if (tma_store && epi == EPI_MASK_BITS) mword = load_bits(half * 32);
      {
        const long long wcy = mbar_wait(&acc_full[ab], aph);
        if (dbg_me) s_dbg[0] += wcy;
      }
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + ab * args.tmem_cols +
                              (static_cast<uint32_t>(q * 32) << 16);
      float* C = args.C + static_cast<size_t>(z) * args.split_stride;
      if (tma_store) {
        // Row-major output through TMA: lane = row; each 32-column chunk is drained in two
        // 16-column halves (register budget: 96/thread with 18 warps).  Bias / ReLU / mask
        // run in registers, the block goes to a 128B-swizzled [32][32] staging tile
        // (conflict-free STS.128) and one elected lane hands it to the async proxy, so
        // the warp never waits on global stores.
        unsigned char* stg = epi_smem + ew * 4096;
        const int row = m0 + q * 32 + lane;
        const bool warp_live = m0 + q * 32 < args.GM;
        int last_c0 = 0;
        for (int c = 0; c < args.n_umma && n0 + c < args.GN; c += 32) last_c0 = c;
        if (half * 32 > last_c0) {      // nothing for this warp in a one-chunk tile
          tc_fence_before();
          arrive_acc_empty(ab);
          continue;
        }
        const int my_last = last_c0 - (((last_c0 >> 5) & 1) != half ? 32 : 0);
#pragma unroll 1
        for (int c0 = half * 32; c0 <= last_c0; c0 += 64) {
          const int colb = n0 + c0;
          if (epi == EPI_MASK_BITS) mword_next = load_bits(c0 + 64);
          uint32_t word_out = 0;
#pragma unroll 1
          for (int hf = 0; hf < 2; ++hf) {
            const long long tp0 = args.dbg ? clock64() : 0;
            uint32_t v[16];
            tmem_ld16(tmem_d + c0 + hf * 16, v);
            const int colh = colb + hf * 16;
            tmem_ld_wait();
            if (hf == 1 && c0 == my_last) {   // accumulator drained: the MMA warp may refill it
              tc_fence_before();
              arrive_acc_empty(ab);
            }
            const long long tp1 = args.dbg ? clock64() : 0;
            float x[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = __uint_as_float(v[j]);
            if (nkb == 0) {            // empty k range: the accumulator was never written
#pragma unroll
              for (int j = 0; j < 16; ++j) x[j] = 0.f;
            }
            if (epi == EPI_BIAS_ACT) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float4 b4 = *reinterpret_cast<const float4*>(sbias + colh + 4 * j);
                x[4 * j + 0] += b4.x; x[4 * j + 1] += b4.y;
                x[4 * j + 2] += b4.z; x[4 * j + 3] += b4.w;
              }
              if (act == TFR_ACT_RELU) {
#pragma unroll
                for (int j = 0; j < 16; ++j) x[j] = fmaxf(x[j], 0.f);
              }
              if (args.bits_out) {
                uint32_t w16 = 0;
#pragma unroll
                for (int j = 0; j < 16; ++j) w16 |= (x[j] > 0.f ? 1u : 0u) << j;
                word_out |= w16 << (hf * 16);
              }
            } else if (epi == EPI_MASK_BITS) {
              const uint32_t w16 = mword >> (hf * 16);
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                // bfe.s32 of a 1-bit field: 0 or 0xffffffff
                int m;
                asm("bfe.s32 %0, %1, %2, 1;" : "=r"(m) : "r"(w16), "r"(j));
                x[j] = __uint_as_float(__float_as_uint(x[j]) & static_cast<uint32_t>(m));
              }
            }
            const long long tpa = args.dbg ? clock64() : 0;
            if (hf == 0) {
              // the previous TMA store of this warp must have finished reading the tile
              if (lane == 0) bulk_wait_read0();
              __syncwarp();
            }
            const long long tpb = args.dbg ? clock64() : 0;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              *reinterpret_cast<float4*>(stg + lane * 128 + (((hf * 4 + j) ^ (lane & 7)) << 4)) =
                  make_float4(x[4 * j + 0], x[4 * j + 1], x[4 * j + 2], x[4 * j + 3]);
            if (dbg_me) {
              s_dbg[1] += tp1 - tp0;
              s_dbg[2] += tpa - tp1;    // register math
              s_dbg[3] += tpb - tpa;    // wait for the staging tile
            }
          }
          const long long tpc = args.dbg ? clock64() : 0;
          if (epi == EPI_BIAS_ACT && args.bits_out) {
            if (args.GN - colb < 32) word_out &= (1u << (args.GN - colb)) - 1u;   // columns >= GN
            if (row < args.GM)
              args.bits_out[static_cast<size_t>(colb >> 5) * args.GM + row] = word_out;
          }
          mword = mword_next;
          fence_proxy_async();
          __syncwarp();
          if (warp_live && lane == 0) {
            tma_store_2d(&tmC, stg, colb, m0 + q * 32);
            bulk_commit();
          }
          if (args.colsum) {
            // lane = column: sum the 32 rows of the staged block (rows past GM are zero)
            const float* tbf = reinterpret_cast<const float*>(stg);
            float cs4[4] = {0.f, 0.f, 0.f, 0.f};   // four chains: the adds are latency-bound
#pragma unroll
            for (int r = 0; r < 32; ++r)
              cs4[r & 3] += tbf[r * 32 + ((((lane >> 2) ^ (r & 7)) << 2) | (lane & 3))];
            const float cs = (cs4[0] + cs4[1]) + (cs4[2] + cs4[3]);
            if (args.colsum_regs) {
              const int ci = c0 >> 5;
#pragma unroll
              for (int k = 0; k < 4; ++k) ccol[k] += (ci >> 1) == k ? cs : 0.f;
            } else if (colb + lane < args.colsum_cols) {
              cacc[colb + lane] += cs;
            }
          }
          if (dbg_me) s_dbg[4] += clock64() - tpc;   // fence + store issue + column sums
        }
        continue;   // acc_empty already signalled
      }
      if (ew >= 4) {                   // fallback stores are done by warps 0..3
        tc_fence_before();
        arrive_acc_empty(ab);
        continue;
      }
      if (args.store_transposed) {
        // lane = row: consecutive lanes hit consecutive addresses of C^T.
        const int row = m0 + q * 32 + lane;
        for (int c0 = 0; c0 < args.n_umma; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(tmem_d + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int col = n0 + c0 + j;
            if (c0 + j >= args.n_umma || col >= args.GN || row >= args.GM) continue;
            const float x = nkb > 0 ? __uint_as_float(v[j]) : 0.f;
            C[static_cast<size_t>(col) * args.ldc + row] = x;
          }
        }
      } else if (args.vec_ok) {
        // Row-major store, vectorised: each 32x32 block goes through shared memory
        // ([32][36] floats, 16-byte rows) so that one warp instruction stores
        // 4 rows x 128 contiguous bytes (STG.128); bias / ReLU mask / column sums
        // ride along.  8 STS.128 + 8 LDS.128 + 8 STG.128 per block.
        float4* tb4 = reinterpret_cast<float4*>(tb);
        const int rows_here = min(32, args.GM - (m0 + q * 32));
        const int r4 = lane >> 3, c4 = lane & 7;
        const bool masked = epi == EPI_MASK_POS && act == TFR_ACT_RELU;
        const size_t rstep = static_cast<size_t>(4) * args.ldc;
        const size_t row_off = static_cast<size_t>(m0 + q * 32 + r4) * args.ldc;
        // ReLU mask source for one 32x32 block: 8 independent 16-byte loads.
        auto load_keep = [&](int c0, float4 (&k)[8]) {
          const int col = n0 + c0 + c4 * 4;
          const bool ok = (c0 + c4 * 4 < args.n_umma) && col < args.GN;
#pragma unroll
          for (int i = 0; i < 8; ++i)
            k[i] = (ok && i * 4 + r4 < rows_here)
                       ? __ldg(reinterpret_cast<const float4*>(args.aux + row_off + col + i * rstep))
                       : make_float4(1.f, 1.f, 1.f, 1.f);
        };
        float4 keep[8], keep_next[8];
        if (masked) load_keep(0, keep);
        for (int c0 = 0; c0 < args.n_umma; c0 += 32) {
          uint32_t v[32];
          const long long tp0 = args.dbg ? clock64() : 0;
          tmem_ld32(tmem_d + c0, v);
          // prefetch the next block's mask while this one is transposed and stored
          if (masked && c0 + 32 < args.n_umma) load_keep(c0 + 32, keep_next);
          const int col = n0 + c0 + c4 * 4;
          const bool col_ok = (c0 + c4 * 4 < args.n_umma) && col < args.GN;
          float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
          if (epi == EPI_BIAS_ACT && col_ok)
            bv = __ldg(reinterpret_cast<const float4*>(args.bias + col));
          tmem_ld_wait();
          const long long tp1 = args.dbg ? clock64() : 0;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float4 t4;
            t4.x = nkb > 0 ? __uint_as_float(v[4 * j + 0]) : 0.f;
            t4.y = nkb > 0 ? __uint_as_float(v[4 * j + 1]) : 0.f;
            t4.z = nkb > 0 ? __uint_as_float(v[4 * j + 2]) : 0.f;
            t4.w = nkb > 0 ? __uint_as_float(v[4 * j + 3]) : 0.f;
            tb4[lane * 9 + j] = t4;
          }
          __syncwarp();
          const size_t off0 = row_off + col;
          float4 xs[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) xs[i] = tb4[(i * 4 + r4) * 9 + c4];
          const long long tp2 = args.dbg ? clock64() : 0;
          float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float4 x = xs[i];
            if (epi == EPI_BIAS_ACT) {
              x.x += bv.x; x.y += bv.y; x.z += bv.z; x.w += bv.w;
              if (act == TFR_ACT_RELU) {
                x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f);
                x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f);
              }
            } else if (masked) {
              if (!(keep[i].x > 0.f)) x.x = 0.f;
              if (!(keep[i].y > 0.f)) x.y = 0.f;
              if (!(keep[i].z > 0.f)) x.z = 0.f;
              if (!(keep[i].w > 0.f)) x.w = 0.f;
            }
            if (col_ok && i * 4 + r4 < rows_here) {
              *reinterpret_cast<float4*>(C + off0 + i * rstep) = x;
              cs.x += x.x; cs.y += x.y; cs.z += x.z; cs.w += x.w;
            }
          }
          if (args.colsum) {
#pragma unroll
            for (int o = 8; o <= 16; o <<= 1) {
              cs.x += __shfl_xor_sync(0xffffffffu, cs.x, o);
              cs.y += __shfl_xor_sync(0xffffffffu, cs.y, o);
              cs.z += __shfl_xor_sync(0xffffffffu, cs.z, o);
              cs.w += __shfl_xor_sync(0xffffffffu, cs.w, o);
            }
            if (r4 == 0 && col_ok) {   // lanes 0..7 own disjoint 4-column groups
              float4* a4 = reinterpret_cast<float4*>(cacc + col);
              float4 a = *a4;
              a.x += cs.x; a.y += cs.y; a.z += cs.z; a.w += cs.w;
              *a4 = a;
            }
          }
          if (masked) {
#pragma unroll
            for (int i = 0; i < 8; ++i) keep[i] = keep_next[i];
          }
          __syncwarp();
          if (dbg_me) {
            const long long tp3 = clock64();
            s_dbg[1] += tp1 - tp0;
            s_dbg[2] += tp2 - tp1;
            s_dbg[3] += tp3 - tp2;
          }
        }
      } else {
        // Row-major store, scalar fallback (unaligned leading dimension / width).
        const int rows_here = min(32, args.GM - (m0 + q * 32));
        for (int c0 = 0; c0 < args.n_umma; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(tmem_d + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) tb[lane * 37 + j] = nkb > 0 ? __uint_as_float(v[j]) : 0.f;
          __syncwarp();
          const int col = n0 + c0 + lane;
          const bool col_ok = (c0 + lane < args.n_umma) && col < args.GN;
          const float bv = (epi == EPI_BIAS_ACT && col_ok) ? __ldg(args.bias + col) : 0.f;
          const size_t off0 = static_cast<size_t>(m0 + q * 32) * args.ldc + col;
          float csum = 0.f;
          for (int rr = 0; rr < rows_here; ++rr) {
            float x = tb[rr * 37 + lane];
            if (epi == EPI_BIAS_ACT) {
              x += bv;
              if (act == TFR_ACT_RELU) x = fmaxf(x, 0.f);
            } else if (epi == EPI_MASK_POS && act == TFR_ACT_RELU && col_ok) {
              if (!(__ldg(args.aux + off0 + static_cast<size_t>(rr) * args.ldc) > 0.f)) x = 0.f;
            }
            if (col_ok) {
              C[off0 + static_cast<size_t>(rr) * args.ldc] = x;
              csum += x;
            }
          }
          if (args.colsum && col_ok) cacc[col] += csum;
          __syncwarp();
        }
      }
      tc_fence_before();
      arrive_acc_empty(ab);   // all epilogue threads arrive: buffer is free
    }
    if ((kFastOuter ? (FAST_EPI != 4) : (args.tma_store != 0)) && lane == 0) bulk_wait_all();
    if (args.colsum) {
      __syncwarp();
      float* dst = args.colsum + static_cast<size_t>(blockIdx.x * kEpiWarps + ew) * args.colsum_stride;
      if (args.colsum_regs) {
        // every warp writes a full row of its slot: its own chunks, zeros elsewhere
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k * 32 + lane < args.GN)
            dst[k * 32 + lane] = (k & 1) == half ? ccol[k >> 1] : 0.f;
      } else {
        for (int c = lane; c < args.GN; c += 32) dst[c] = cacc[c];
      }
    }
    if (dbg_me) {
      args.dbg[blockIdx.x * 12 + 6] = s_dbg[0];
      args.dbg[blockIdx.x * 12 + 7] = clock64() - t_start;
      args.dbg[blockIdx.x * 12 + 8] = s_dbg[1];
      args.dbg[blockIdx.x * 12 + 9] = s_dbg[2];
      args.dbg[blockIdx.x * 12 + 10] = s_dbg[3];
      args.dbg[blockIdx.x * 12 + 11] = s_dbg[4];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CG2) cluster_sync_all();   // no CTA leaves (or frees tensor memory) while its peer works
  if (warp == 1) {
    if (CG2) tmem_dealloc2(tmem_base, args.tmem_alloc_cols);
    else tmem_dealloc(tmem_base, args.tmem_alloc_cols);
  }
}

// ------------------------------------------------------------------ host -------
// 2D fp32 tensor [outer rows][inner cols], box [box_outer][32 cols], 128B swizzle (the 32 B
// atom variant for MN-major operands).
static int encode_2d(CUtensorMap* tm, const float* ptr, uint64_t inner, uint64_t outer,
                     uint64_t ld_floats, uint32_t box_outer, bool mn_major) {
  return encode_tmap_2d(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, ptr, inner, outer,
                        ld_floats * sizeof(float), BK, box_outer,
                        mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B);
}

bool shape_supported(int lda, int ldb) { return lda % 4 == 0 && ldb % 4 == 0; }

static long long* g_dbg = nullptr;   // set by tfr_tc_set_debug (profiling aid)

template <bool A_MN, bool B_MN, int PASSES, bool SPLIT_B>
static int launch(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmBlo,
                  const CUtensorMap& tmC, const KernelArgs& ka, dim3 grid, size_t smem,
                  cudaStream_t st) {
  auto kern = tc_gemm_kernel<A_MN, B_MN, PASSES, SPLIT_B>;
  TFR_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, kThreads, smem, st>>>(tmA, tmB, tmBlo, tmC, ka);
  TFR_LAUNCH_OK();
  return TFR_OK;
}

// CTA pairs: cluster of 2 along x (one TPC), cta_group::2 MMAs.
// MN = false: forward / dZ (K-major, pre-split B); true: dW (MN-major, split B).
// FE: compile-time epilogue (see FAST_EPI), -1 = generic.
template <bool MN, int FE>
static int launch_pairs(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmBlo,
                        const CUtensorMap& tmC, const KernelArgs& ka, dim3 grid, size_t smem,
                        cudaStream_t st) {
  auto kern = tc_gemm_kernel<MN, MN, 3, MN, true, FE>;
  TFR_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  TFR_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmBlo, tmC, ka));
  TFR_LAUNCH_OK();
  return TFR_OK;
}

int gemm(const GemmDesc& g, cudaStream_t st) {
  TFR_REQUIRE(g.A && g.B && g.C, "tc gemm: NULL operand");
  TFR_REQUIRE(g.GM >= 1 && g.GN >= 1 && g.GK >= 1, "tc gemm: empty problem");
  TFR_REQUIRE(g.passes == 1 || g.passes == 3, "tc gemm: passes must be 1 or 3");
  TFR_REQUIRE(g.lda % 4 == 0 && g.ldb % 4 == 0, "tc gemm: leading dimensions must be multiples of 4");
  TFR_REQUIRE((reinterpret_cast<uintptr_t>(g.A) & 15) == 0 && (reinterpret_cast<uintptr_t>(g.B) & 15) == 0,
              "tc gemm: operands must be 16-byte aligned");
  const bool pre_split_b = g.passes == 3 && !g.split_b;
  TFR_REQUIRE(!pre_split_b || g.B_lo != nullptr, "tc gemm: B_lo required for pre-split B");
  TFR_REQUIRE(!pre_split_b || (reinterpret_cast<uintptr_t>(g.B_lo) & 15) == 0, "tc gemm: B_lo alignment");

  // N tiling: one tile if it fits a single UMMA (N <= 256), else tiles of 256.
  // dW GEMMs as CTA pairs: each CTA stages its 128 rows of the M side and HALF of the N side
  // (whole 32-column boxes), so N is rounded up to a multiple of 64.
  const bool want_pairs_mn = g.passes == 3 && g.a_mn && g.b_mn && g.split_b && g.GM > BM &&
                             (g.GN + 63) / 64 * 64 <= kMaxN;
  const int n_umma = want_pairs_mn ? (g.GN + 63) / 64 * 64
                                   : (g.GN <= kMaxN ? ((g.GN + 15) / 16) * 16 : kMaxN);
  const int n_tiles = (g.GN + n_umma - 1) / n_umma;
  // Stage depth in k is BK for both majornesses (16-row MN-major stages, which would deepen
  // the ring of the dW GEMMs, were measured slower: more TMA boxes per byte).
  const int a_tile_bytes = g.a_mn ? (BM / 32) * kBoxBytes : kATileBytes;
  int b_tile_bytes = g.b_mn ? ((n_umma + 31) / 32) * kBoxBytes : n_umma * 128;
  const int copies = g.passes == 3 ? 2 : 1;
  uint32_t acc_cols = 32;
  while ((int)acc_cols < n_umma) acc_cols <<= 1;
  // A in tensor memory: needs 64 columns per stage next to the two accumulators
  // (K-major A with pre-split B: forward / dZ GEMMs.  MN-major A with B split on the fly: the
  //  dW GEMMs, whose tiles are long split-K loops — one accumulator buffer is enough there,
  //  which leaves the columns for the A stages even at N = 256.)
  const bool a_tmem_k = !g.a_mn && !g.split_b;
  const bool a_tmem_mn = g.a_mn && g.split_b;
  uint32_t acc_bufs = 2;
  if (a_tmem_mn && 2 * acc_cols + 3 * 64 > 512) acc_bufs = 1;
  bool a_tmem = g.passes == 3 && (a_tmem_k || a_tmem_mn) && acc_bufs * acc_cols + 2 * 64 <= 512;
  if (!a_tmem) acc_bufs = 2;
  // CTA pairs (see the kernel's CG2 note): forward / dZ GEMMs with one n tile.
  const int m_tiles_all = (g.GM + BM - 1) / BM;
  const bool cg2_k = g.passes == 3 && a_tmem_k && !g.b_mn && n_tiles == 1 && (g.splits <= 1) &&
                     n_umma % 32 == 0 && m_tiles_all >= 4;
  const bool cg2_mn = want_pairs_mn && a_tmem && n_tiles == 1;
  const bool cg2 = cg2_k || cg2_mn;
  if (cg2_k) b_tile_bytes = (n_umma / 2) * 128;         // this CTA's half of the B tile
  if (cg2_mn) b_tile_bytes = (n_umma / 64) * kBoxBytes; // ... as whole [32 k][32 n] boxes
  const int stage_bytes = a_tmem ? a_tile_bytes + b_tile_bytes * copies
                                 : (a_tile_bytes + b_tile_bytes) * copies;
  int splits = g.splits < 1 ? 1 : g.splits;
  // TMA-store epilogue: row-major, unsplit output with 16-byte aligned rows.
  const bool tma_store =
      g.epi != EPI_MASK_POS && !g.store_transposed && splits == 1 &&
      g.ldc % 4 == 0 && g.GN % 4 == 0 && (reinterpret_cast<uintptr_t>(g.C) & 15) == 0 &&
      (!g.bias || (reinterpret_cast<uintptr_t>(g.bias) & 15) == 0) &&
      (n_tiles == 1 || n_umma % 32 == 0);
  const bool colsum_regs = tma_store && g.colsum && n_tiles == 1;
  const int colsum_cols = (g.colsum && !colsum_regs) ? ((g.GN + 3) / 4) * 4 : 0;
  TFR_REQUIRE(colsum_cols <= 1024, "tc gemm: colsum output supports GN <= 1024");
  const int bias_cols = (tma_store && g.epi == EPI_BIAS_ACT) ? ((n_tiles * n_umma + 31) / 32) * 32 : 0;
  const size_t fixed1 = kEpiSmemBytes + kEpiWarps * colsum_cols * sizeof(float);
  const size_t fixed2 = kEpiSmemBytes2 + (kEpiWarps * colsum_cols + bias_cols) * sizeof(float);
  const size_t budget = 227 * 1024 - 1024 /*align*/ - 256 /*barriers*/;
  const int epi_smem_bytes = tma_store ? kEpiSmemBytes2 : kEpiSmemBytes;
  int stages = (int)((budget - (tma_store ? fixed2 : fixed1)) / stage_bytes);
  if (stages > kMaxStages) stages = kMaxStages;
  if (a_tmem) {
    const int room = (512 - (int)(acc_bufs * acc_cols)) / 64;   // A stages that fit tensor memory
    if (stages > room) stages = room;
  }
  TFR_REQUIRE(stages >= 1, "tc gemm: tile does not fit shared memory");
  const int nkb_total = (g.GK + BK - 1) / BK;
  int kb_per_split = (nkb_total + splits - 1) / splits;
  // (a split whose k range is empty stores zeros, so any split count is legal)

  CUtensorMap tmA, tmB, tmBlo;
  int rc;
  if (!g.a_mn) rc = encode_2d(&tmA, g.A, (uint64_t)g.GK, (uint64_t)g.GM, (uint64_t)g.lda, BM, false);
  else rc = encode_2d(&tmA, g.A, (uint64_t)g.GM, (uint64_t)g.GK, (uint64_t)g.lda, (uint32_t)BK, true);
  if (rc) return rc;
  const uint32_t b_box_rows = cg2 ? (uint32_t)n_umma / 2 : (uint32_t)n_umma;
  if (!g.b_mn) rc = encode_2d(&tmB, g.B, (uint64_t)g.GK, (uint64_t)g.GN, (uint64_t)g.ldb, b_box_rows, false);
  else rc = encode_2d(&tmB, g.B, (uint64_t)g.GN, (uint64_t)g.GK, (uint64_t)g.ldb, (uint32_t)BK, true);
  if (rc) return rc;
  tmBlo = tmB;
  if (pre_split_b) {
    if (!g.b_mn) rc = encode_2d(&tmBlo, g.B_lo, (uint64_t)g.GK, (uint64_t)g.GN, (uint64_t)g.ldb, b_box_rows, false);
    else rc = encode_2d(&tmBlo, g.B_lo, (uint64_t)g.GN, (uint64_t)g.GK, (uint64_t)g.ldb, (uint32_t)BK, true);
    if (rc) return rc;
  }

  KernelArgs ka;
  ka.C = g.C; ka.ldc = g.ldc;
  ka.GM = g.GM; ka.GN = g.GN; ka.GK = g.GK;
  ka.n_umma = n_umma;
  ka.b_tile_bytes = b_tile_bytes;
  ka.a_tile_bytes = a_tile_bytes;
  ka.stages = stages;
  ka.epi = g.epi; ka.act = g.act; ka.store_transposed = g.store_transposed;
  ka.bias = g.bias; ka.aux = g.aux;
  ka.kb_per_split = kb_per_split;
  ka.split_stride = g.split_stride;
  ka.tmem_cols = acc_cols;     // per accumulator buffer; the kernel allocates two
  ka.a_tmem = a_tmem ? 1 : 0;
  ka.acc_bufs = acc_bufs;
  ka.a_col0 = acc_bufs * acc_cols;
  {
    uint32_t need = acc_bufs * acc_cols + (a_tmem ? 64u * (uint32_t)stages : 0u), alloc = 32;
    while (alloc < need) alloc <<= 1;
    ka.tmem_alloc_cols = cg2 ? 512u : alloc;   // pairs: all of it, same base in both CTAs
  }
  ka.dbg = g_dbg;
  ka.vec_ok = (g.ldc % 4 == 0) && (g.GN % 4 == 0) && (g.split_stride % 4 == 0) &&
              ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0) &&
              (!g.aux || (reinterpret_cast<uintptr_t>(g.aux) & 15) == 0) &&
              (!g.bias || (reinterpret_cast<uintptr_t>(g.bias) & 15) == 0) &&
              (!g.colsum || ((reinterpret_cast<uintptr_t>(g.colsum) & 15) == 0 &&
                             g.colsum_stride % 4 == 0));
  ka.colsum = g.colsum;
  ka.colsum_stride = g.colsum_stride;
  ka.colsum_cols = colsum_cols;
  TFR_REQUIRE(!g.colsum || (!g.store_transposed && splits == 1),
              "tc gemm: colsum output needs a row-major, unsplit store");
  TFR_REQUIRE(g.epi != EPI_BIAS_ACT || g.bias, "tc gemm: bias required");
  TFR_REQUIRE(g.epi != EPI_MASK_POS || g.aux, "tc gemm: aux required");
  ka.tma_store = tma_store;
  ka.epi_smem_bytes = epi_smem_bytes;
  ka.colsum_regs = colsum_regs;
  ka.bias_cols = bias_cols;
  ka.bits_out = g.mask_bits_out;
  ka.bits_in = g.mask_bits_in;
  TFR_REQUIRE(!(g.mask_bits_out || g.epi == EPI_MASK_BITS) || ka.tma_store,
              "tc gemm: ReLU sign bits need the row-major TMA-store epilogue");
  TFR_REQUIRE(g.epi != EPI_MASK_BITS || g.mask_bits_in, "tc gemm: mask_bits_in required");
  CUtensorMap tmC = tmA;
  if (ka.tma_store) {
    rc = encode_2d(&tmC, g.C, (uint64_t)g.GN, (uint64_t)g.GM, (uint64_t)g.ldc, 32, false);
    if (rc) return rc;
  }

  ka.m_tiles = (g.GM + BM - 1) / BM;
  ka.n_tiles = n_tiles;
  ka.splits = splits;
  const int total_tiles = ka.m_tiles * ka.n_tiles * splits;
  const int sms = num_sms();
  dim3 grid(total_tiles < sms ? total_tiles : sms);
  if (cg2) {
    const int pair_tiles = (ka.m_tiles + 1) / 2 * ka.n_tiles * splits;
    const int pairs = pair_tiles < sms / 2 ? pair_tiles : sms / 2;
    grid = dim3(2 * pairs);
  }
  const size_t smem = (size_t)stages * stage_bytes + epi_smem_bytes +
                      (kEpiWarps * colsum_cols + bias_cols) * sizeof(float) + 1024 /*align*/ +
                      256 /*barriers*/;
  if (g.colsum_slots_out) *g.colsum_slots_out = kEpiWarps * (int)grid.x;

  if (cg2) {
    if (cg2_mn) {
      if (!ka.tma_store && g.epi == EPI_STORE)
        return launch_pairs<true, 4>(tmA, tmB, tmBlo, tmC, ka, grid, smem, st);
      return launch_pairs<true, -1>(tmA, tmB, tmBlo, tmC, ka, grid, smem, st);
    }
    if (ka.tma_store && g.epi == EPI_STORE)
      return launch_pairs<false, 0>(tmA, tmB, tmBlo, tmC, ka, grid, smem, st);
    if (ka.tma_store && g.epi == EPI_BIAS_ACT && g.act == TFR_ACT_RELU)
      return launch_pairs<false, 1>(tmA, tmB, tmBlo, tmC, ka, grid, smem, st);
    if (ka.tma_store && g.epi == EPI_MASK_BITS)
      return launch_pairs<false, 3>(tmA, tmB, tmBlo, tmC, ka, grid, smem, st);
    return launch_pairs<false, -1>(tmA, tmB, tmBlo, tmC, ka, grid, smem, st);
  }
  if (g.a_mn && g.b_mn && g.passes == 3 && g.split_b && !ka.tma_store &&
      g.epi == EPI_STORE) {   // single-CTA dW GEMM (one 128-row block): plain-store kernel
    auto kern = tc_gemm_kernel<true, true, 3, true, false, 4>;
    TFR_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kThreads, smem, st>>>(tmA, tmB, tmBlo, tmC, ka);
    TFR_LAUNCH_OK();
    return TFR_OK;
  }
#define TFR_TC_LAUNCH(AMN, BMN, P, SB) \
  return launch<AMN, BMN, P, SB>(tmA, tmB, tmBlo, tmC, ka, grid, smem, st)
  const int key = (g.a_mn ? 8 : 0) | (g.b_mn ? 4 : 0) | (g.passes == 3 ? 2 : 0) |
                  ((g.passes == 3 && g.split_b) ? 1 : 0);
  switch (key) {
    case 0: TFR_TC_LAUNCH(false, false, 1, false);
    case 2: TFR_TC_LAUNCH(false, false, 3, false);
    case 3: TFR_TC_LAUNCH(false, false, 3, true);
    case 4: TFR_TC_LAUNCH(false, true, 1, false);
    case 6: TFR_TC_LAUNCH(false, true, 3, false);
    case 7: TFR_TC_LAUNCH(false, true, 3, true);
    case 8: TFR_TC_LAUNCH(true, false, 1, false);
    case 10: TFR_TC_LAUNCH(true, false, 3, false);
    case 11: TFR_TC_LAUNCH(true, false, 3, true);
    case 12: TFR_TC_LAUNCH(true, true, 1, false);
    case 14: TFR_TC_LAUNCH(true, true, 3, false);
    case 15: TFR_TC_LAUNCH(true, true, 3, true);
  }
#undef TFR_TC_LAUNCH
  set_error("tc gemm: unsupported variant %d", key);
  return TFR_UNSUPPORTED;
}

}  // namespace tc
}  // namespace tfr

// Profiling aid: [num_ctas][8] int64 wait-cycle counters written by each launch
// {producer wait-empty, producer total, mma wait-acc-empty, mma wait-operands, mma total,
//  splitter wait-tma, epilogue wait-acc-full, epilogue total}.  NULL disables.
extern "C" int tfr_tc_set_debug(long long* buf) {
  tfr::tc::g_dbg = buf;
  return 0;
}

// Test / parity entry: raw GEMM through the tensor-core engine.
extern "C" int tfr_tc_gemm(const float* A, int lda, const float* B, int ldb, const float* B_lo,
                           float* C, int ldc, int GM, int GN, int GK, int a_mn, int b_mn,
                           int passes, int split_b, int epi, const float* bias, const float* aux,
                           int act, int store_transposed, int splits, size_t split_stride,
                           uint32_t* mask_bits_out, const uint32_t* mask_bits_in,
                           void* stream) {
  tfr::tc::GemmDesc g{};
  g.mask_bits_out = mask_bits_out; g.mask_bits_in = mask_bits_in;
  g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.B_lo = B_lo; g.C = C; g.ldc = ldc;
  g.GM = GM; g.GN = GN; g.GK = GK; g.a_mn = a_mn; g.b_mn = b_mn; g.passes = passes;
  g.split_b = split_b; g.epi = epi; g.bias = bias; g.aux = aux; g.act = act;
  g.store_transposed = store_transposed; g.splits = splits; g.split_stride = split_stride;
  return tfr::tc::gemm(g, (cudaStream_t)stream);
}
