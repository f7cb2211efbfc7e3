// Dense layers of the PropMLP / NerfMLP on 5th-gen tensor cores (sm_100a): persistent,
// warp-specialised GEMM with TMA-staged operands, tcgen05.mma accumulating in TMEM and a fused
// epilogue.  Replaces nn.Dense (+ReLU, + skip-concat as a wider K) of models.py:436-437,455-460,
// 527,577 and the dgrad / wgrad GEMMs jax.value_and_grad derives from them
// (train_utils.py:316-317).
//
//   warp 0   : TMA producer (one elected lane) -- cp.async.bulk.tensor.2d into an operand ring
//   warp 1   : MMA issuer  (one elected lane) -- tcgen05.mma.kind::f16, N<=256
//   warp 2   : TMEM allocator (512 columns = two 256-column accumulator stages)
//   warps 4-11: epilogue -- two warps per TMEM lane quadrant (each takes half of the tile's
//              columns): tcgen05.ld 32x32b, bias/ReLU | mask/rank-1/column sums | fp32 reduction,
//              swizzled smem staging + TMA bulk stores
//
// Two variants of the same kernel (template CTAS):
//   CTAS=1 : one CTA per 128 x block_n tile, tcgen05.mma.cta_group::1 (M=128); any shape.
//   CTAS=2 : a two-CTA cluster (one TPC) per 256 x 256 tile, tcgen05.mma.cta_group::2 (M=256) issued by
//            the leader CTA; each CTA stages its own 128 A rows and HALF of the B tile, so operand
//            shared-memory traffic per SM drops by a third and the ring holds 6 stages.  The leader's
//            "full" barriers collect both CTAs' TMA bytes; "empty"/"accumulator full" arrivals are
//            multicast to both CTAs by tcgen05.commit; both epilogues release the accumulator on the
//            leader's barrier.  Used when M % 256 == 0 and block_n == 256 (all 360-config layers).
//
// Operand layouts (all bf16, 128-byte swizzle):
//   FWD / DGRAD : A[M,K] and B[N,K] are K-major (reduction index contiguous);
//   WGRAD       : A = X[R,Mo] and B = dY[R,N] are "MN-major" (reduction index R on rows):
//                 out[Mo,N] += X^T dY, split over R with fp32 vector reductions.
#include <cuda.h>

#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "tc_common.cuh"

namespace mnrf {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;          // 64 bf16 = one 128-byte swizzle span
constexpr int MAX_BLOCK_N = 256;
constexpr int NUM_ACC = 2;
constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;        // 16 KiB
constexpr int B_STAGE_BYTES = MAX_BLOCK_N * BLOCK_K * 2;    // 32 KiB
constexpr int NUM_EPI_WARPS = 8;
constexpr int OUT_STAGE_BYTES = NUM_EPI_WARPS * 32 * 128;    // one 32-row x 128-byte slab per epilogue warp
// Operand ring depth: a CTA of a pair stages half of each B tile, so its ring holds 6 stages where a single CTA's
// holds 4.  A K = 1024 tile spends 8k cycles in the main loop, so the deepest ring that fits next to one output
// staging slab per epilogue warp wins (fewer stages with 2 or 3 slabs measured no faster even on K = 256 tiles).
constexpr int num_stages(int ctas) { return ctas == 2 ? 6 : 4; }
constexpr int smem_bytes(int ctas) {
  return num_stages(ctas) * (A_STAGE_BYTES + B_STAGE_BYTES / ctas) + OUT_STAGE_BYTES + 1024 /*align*/ + 256;
}

constexpr int NUM_THREADS = 128 + NUM_EPI_WARPS * 32;

struct GemmParams {
  int mode, act;
  int64_t m;                  // output rows
  int n, k;                   // output cols, reduction length
  int block_n;                // N tile (<= 256, multiple of 16, divides n)
  int num_m_blocks, num_n_blocks, num_splits, kblocks_per_split, num_k_blocks;
  int64_t ldc, ldmask;
  const float* bias;
  const float* rowv;
  const float* colv;
  const __nv_bfloat16* mask;
  uint32_t* maskbits;         // FWD+ReLU: written (1 bit per output, word = 32 columns); DGRAD: read
  int64_t ldmaskbits;         // in 32-bit words
  int64_t mask_mod;           // > 0: mask row = output row mod mask_mod
  const __nv_bfloat16* addend;  // DGRAD: out += addend[M, ldadd] (second contribution to a shared input)
  int64_t ldadd;
  int use_tma_store;
  int debug;                  // MNRF_GEMM_DEBUG (timing experiments only): 1 = skip the epilogue, 2 = skip stores
  float* colsum;              // DGRAD: colsum[N] += column sums of the output (bias gradient of the
                              // layer that produced the masking activation), from the epilogue registers
  // WGRAD side sums, computed by the (otherwise idle) epilogue warps from the operand tiles the main loop stages:
  float* side_bsum;           //   side_bsum[n] += sum_r B[r, n]            (bias gradient: column sums of dY)
  const float* side_w;        //   side_aw[m]  += sum_r side_w[r] * A[r, m] (weight gradient of a Dense(1) head
  float* side_aw;             //                                             that reads the same activation X)
  void* out;
};

template <int MODE, int CTAS>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ CUtensorMap tmap_c, const GemmParams p) {
  constexpr int NUM_STAGES = num_stages(CTAS);
  constexpr int B_STAGE = B_STAGE_BYTES / CTAS;    // each CTA of a pair stages half of the B tile
  extern __shared__ uint8_t smem_dyn[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + NUM_STAGES * A_STAGE_BYTES;
  uint8_t* smem_out = smem + NUM_STAGES * (A_STAGE_BYTES + B_STAGE);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_out + OUT_STAGE_BYTES);
  uint64_t* full_bar = bars;                       // [NUM_STAGES]  (CTAS=2: the leader's are used)
  uint64_t* empty_bar = bars + NUM_STAGES;         // [NUM_STAGES]
  uint64_t* tfull_bar = bars + 2 * NUM_STAGES;     // [NUM_ACC]
  uint64_t* tempty_bar = tfull_bar + NUM_ACC;      // [NUM_ACC]     (CTAS=2: the leader's are used)
  uint64_t* mdone_bar = tempty_bar + NUM_ACC;      // [NUM_STAGES]  WGRAD side sums: the MMAs of this stage have retired
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(mdone_bar + NUM_STAGES);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int rank = CTAS == 1 ? 0 : (int)cluster_ctarank();     // CTA within its pair; 0 = leader
  const int worker = blockIdx.x / CTAS;                        // tile owner (CTA or CTA pair)
  const int num_workers = gridDim.x / CTAS;
  const int num_m_units = p.num_m_blocks / CTAS;               // 128*CTAS-row units
  const int total_tiles = num_m_units * p.num_n_blocks * p.num_splits;
  constexpr bool kWgrad = (MODE == MNRF_GEMM_WGRAD);
  // WGRAD side sums: the epilogue warps also consume every operand stage, after the MMAs that read it
  const bool side = kWgrad && (p.side_bsum != nullptr || p.side_aw != nullptr);

  if (warp == 0 && elect_one()) {
    prefetch_tmap(&tmap_a);
    prefetch_tmap(&tmap_b);
    if (MODE != MNRF_GEMM_WGRAD) prefetch_tmap(&tmap_c);
  }
  if (warp == 1 && elect_one()) {
    for (int i = 0; i < NUM_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], side ? 1 + NUM_EPI_WARPS : 1);
      mbar_init(&mdone_bar[i], 1);
    }
    for (int i = 0; i < NUM_ACC; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], CTAS * NUM_EPI_WARPS * 32); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<CTAS>(tmem_ptr, 512);
  tc_fence_before();
  if (CTAS == 1) __syncthreads(); else cluster_sync_all();    // peers must see initialised barriers
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  const int b_rows = p.block_n / CTAS;             // B-tile rows this CTA stages
  const uint32_t stage_bytes = A_STAGE_BYTES + (uint32_t)b_rows * BLOCK_K * 2;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      uint32_t stage = 0, phase = 0;
      for (int tile = worker; tile < total_tiles; tile += num_workers) {
        const int n_blk = tile % p.num_n_blocks;
        const int rest = tile / p.num_n_blocks;
        const int m_blk = (rest % num_m_units) * CTAS + rank;
        const int split = rest / num_m_units;
        const int kb0 = split * p.kblocks_per_split;
        const int kb1 = min(p.num_k_blocks, kb0 + p.kblocks_per_split);
        const int b_row0 = n_blk * p.block_n + rank * b_rows;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1, 1);
          if (rank == 0) mbar_expect_tx(&full_bar[stage], stage_bytes * CTAS);
          uint8_t* sa = smem_a + stage * A_STAGE_BYTES;
          uint8_t* sb = smem_b + stage * B_STAGE;
          if (!kWgrad) {
            // K-major: box = [64 k][rows]
            if (CTAS == 1) {
              tma_load_2d(sa, &tmap_a, &full_bar[stage], kb * BLOCK_K, m_blk * BLOCK_M);
              tma_load_2d(sb, &tmap_b, &full_bar[stage], kb * BLOCK_K, b_row0);
            } else {
              tma_load_2d_pair(sa, &tmap_a, &full_bar[stage], kb * BLOCK_K, m_blk * BLOCK_M);
              tma_load_2d_pair(sb, &tmap_b, &full_bar[stage], kb * BLOCK_K, b_row0);
            }
          } else {
            // MN-major: one box per 64-wide MN atom = [64 mn][64 r], atoms BLOCK_K*128 bytes apart
            for (int a = 0; a < BLOCK_M / 64; ++a) {
              if (CTAS == 1) tma_load_2d(sa + a * (BLOCK_K * 128), &tmap_a, &full_bar[stage], m_blk * BLOCK_M + a * 64, kb * BLOCK_K);
              else tma_load_2d_pair(sa + a * (BLOCK_K * 128), &tmap_a, &full_bar[stage], m_blk * BLOCK_M + a * 64, kb * BLOCK_K);
            }
            for (int a = 0; a < b_rows / 64; ++a) {
              if (CTAS == 1) tma_load_2d(sb + a * (BLOCK_K * 128), &tmap_b, &full_bar[stage], b_row0 + a * 64, kb * BLOCK_K);
              else tma_load_2d_pair(sb + a * (BLOCK_K * 128), &tmap_b, &full_bar[stage], b_row0 + a * 64, kb * BLOCK_K);
            }
          }
          if (++stage == NUM_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (CTAS=2: leader CTA only) =====================
    if (rank == 0) {
    const uint32_t idesc = make_idesc(BLOCK_M * CTAS, p.block_n, kWgrad ? 1 : 0, kWgrad ? 1 : 0);
    uint32_t stage = 0, phase = 0;
    int it = 0;
    for (int tile = worker; tile < total_tiles; tile += num_workers, ++it) {
      const int rest = tile / p.num_n_blocks;
      const int split = rest / num_m_units;
      const int kb0 = split * p.kblocks_per_split;
      const int kb1 = min(p.num_k_blocks, kb0 + p.kblocks_per_split);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1, 2);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * MAX_BLOCK_N;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full_bar[stage], phase, 3);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem_a + stage * A_STAGE_BYTES);
          const uint32_t sb = smem_u32(smem_b + stage * B_STAGE);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            uint64_t adesc, bdesc;
            if (!kWgrad) {
              // K-major, SW128: 8-row groups 1024 B apart; advance 32 B per UMMA_K inside the span
              adesc = make_smem_desc(sa + k * (UMMA_K * 2), 0, 1024);
              bdesc = make_smem_desc(sb + k * (UMMA_K * 2), 0, 1024);
            } else {
              // MN-major, SW128: LBO = stride between 64-wide MN atoms, SBO = stride between
              // 8-row k groups; advance 16 k rows = 2048 B per UMMA_K
              adesc = make_smem_desc(sa + k * (UMMA_K * 128), BLOCK_K * 128, 1024);
              bdesc = make_smem_desc(sb + k * (UMMA_K * 128), BLOCK_K * 128, 1024);
            }
            umma_bf16<CTAS>(tmem_d, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit<CTAS>(&empty_bar[stage]);               // frees the smem slot when the MMAs retire
          if (side) umma_commit<CTAS>(&mdone_bar[stage]);     // ... after the side sums have read it too
          if (kb == kb1 - 1) umma_commit<CTAS>(&tfull_bar[acc]);  // accumulator complete
        }
        __syncwarp();
        if (++stage == NUM_STAGES) { stage = 0; phase ^= 1; }
      }
    }
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int q = warp & 3;                 // TMEM lane quadrant this warp may touch
    const int ew = warp - 4;                // epilogue warp index 0..7
    // the two warps of a quadrant split the tile's columns (tiles narrower than 128: warp-half 0 only)
    const int cols_per_half = p.block_n >= 128 ? p.block_n / 2 : p.block_n;
    const int c_begin = (ew >> 2) * cols_per_half;
    const int ncols = max(0, min(p.block_n, c_begin + cols_per_half) - c_begin);   // <= 128
    const int w_begin = c_begin >> 5;       // first 32-column mask word of this warp's columns
    const int nwords = (ncols + 31) >> 5;   // <= 4
    // Column sums stay in registers across this CTA's tiles when their n_blk repeats with period 1
    // or 2 (a worker's tiles are num_workers apart): one atomic per column per CTA instead of per tile.
    const int cs_step = num_workers % p.num_n_blocks;
    const int cs_period = cs_step == 0 ? 1 : (2 * cs_step == p.num_n_blocks ? 2 : 0);
    const bool cs_resident = cs_period != 0;
    float csacc[4] = {0.f, 0.f, 0.f, 0.f};     // tiles 0, 2, 4, ... of this CTA (all tiles for period 1)
    float csodd[4] = {0.f, 0.f, 0.f, 0.f};     // tiles 1, 3, 5, ... (period 2)
    int cs_ncol0 = -1, cs_ncol1 = -1;
    uint32_t sstage = 0, sphase = 0;        // WGRAD side sums: this warp's position in the operand ring

    // per-row inputs of a tile (DGRAD): fetched one tile ahead so their latency hides behind the
    // previous tile's epilogue
    float rv_next = 0.f;
    uint32_t mb_next[4] = {0u, 0u, 0u, 0u};
    auto fetch_row_inputs = [&](int tile) {
      rv_next = 0.f;
#pragma unroll
      for (int w = 0; w < 4; ++w) mb_next[w] = 0u;
      if (MODE != MNRF_GEMM_DGRAD || tile >= total_tiles) return;
      const int n_blk = tile % p.num_n_blocks;
      const int m_blk = ((tile / p.num_n_blocks) % num_m_units) * CTAS + rank;
      const int64_t row = (int64_t)m_blk * BLOCK_M + q * 32 + lane;
      if (row >= p.m) return;
      if (p.rowv) rv_next = p.rowv[row];
      if (p.maskbits && ncols > 0) {
        const int64_t mrow = p.mask_mod > 0 ? row % p.mask_mod : row;
        const uint32_t* mp = p.maskbits + mrow * p.ldmaskbits + ((n_blk * p.block_n) >> 5) + w_begin;
        if (nwords == 4) {
          const uint4 t = *reinterpret_cast<const uint4*>(mp);
          mb_next[0] = t.x; mb_next[1] = t.y; mb_next[2] = t.z; mb_next[3] = t.w;
        } else {
#pragma unroll
          for (int w = 0; w < 4; ++w)
            if (w < nwords) mb_next[w] = mp[w];
        }
      }
    };
    fetch_row_inputs(worker);

    int it = 0;
    for (int tile = worker; tile < total_tiles; tile += num_workers, ++it) {
      const int n_blk = tile % p.num_n_blocks;
      const int rest = tile / p.num_n_blocks;
      const int m_blk = (rest % num_m_units) * CTAS + rank;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int64_t row = (int64_t)m_blk * BLOCK_M + q * 32 + lane;
      const bool row_ok = row < p.m;
      const int ncol0 = n_blk * p.block_n;
      const float rv = rv_next;
      uint32_t mbits[4];
#pragma unroll
      for (int w = 0; w < 4; ++w) mbits[w] = mb_next[w];
      fetch_row_inputs(tile + num_workers);
      if (kWgrad && side) {
        // Consume this tile's operand stages right behind the MMAs: column sums of the B tile (dY -> bias
        // gradient; one output-row unit per column block does it) and row-weighted column sums of the A tile
        // (X -> gradient of a Dense(1) head on the same activation; the first column block does it).
        // MN-major stage layout: 64-wide atoms of [64 reduction rows x 128 B], SWIZZLE_128B.
        const int split = rest / num_m_units;
        const int kb0 = split * p.kblocks_per_split;
        const int kb1 = min(p.num_k_blocks, kb0 + p.kblocks_per_split);
        const bool do_b = p.side_bsum != nullptr && (rest % num_m_units) == 0;
        const bool do_a = p.side_aw != nullptr && n_blk == 0;
        const int t = ew * 32 + lane;
        const int b_rows_ = p.block_n / CTAS;
        const int b_pairs = b_rows_ >> 1, b_rpg = 64 / (256 / b_pairs);
        const int bp = t % b_pairs, bg = t / b_pairs;
        const int ap = t & 63, ag = t >> 6;                    // A: 128 columns = 64 pairs x 4 row groups of 16
        const uint32_t b_off = (uint32_t)((bp >> 5) * (BLOCK_K * 128) + ((bp & 3) << 2));
        const uint32_t a_off = (uint32_t)((ap >> 5) * (BLOCK_K * 128) + ((ap & 3) << 2));
        const int b_chunk = (bp & 31) >> 2, a_chunk = (ap & 31) >> 2;
        float bs0 = 0.f, bs1 = 0.f, as0 = 0.f, as1 = 0.f;
        // side_w rows of a k-block are a fresh 64-byte segment of global memory per warp: fetched kSidePf k-blocks
        // ahead (lane i < 16 holds row i of this warp's 16-row group), or every k-block would expose one cold DRAM
        // round trip on the path that releases the operand ring (measured: 2.1k cycles per k-block against 512 of
        // MMA work on the bottleneck layer's weight gradient)
        constexpr int kSidePf = 4;
        float wq[kSidePf];
        auto side_w_fetch = [&](int kbx) -> float {
          const int64_t rr = (int64_t)kbx * BLOCK_K + ag * 16 + lane;
          return (do_a && kbx < kb1 && lane < 16 && rr < p.k) ? __ldg(p.side_w + rr) : 0.f;
        };
#pragma unroll
        for (int j = 0; j < kSidePf; ++j) wq[j] = side_w_fetch(kb0 + j);
        for (int kbq = kb0; kbq < kb1; kbq += kSidePf) {
#pragma unroll
        for (int jq = 0; jq < kSidePf; ++jq) {
          const int kb = kbq + jq;
          if (kb >= kb1) break;
          const float wcur = wq[jq];
          wq[jq] = side_w_fetch(kb + kSidePf);
          mbar_wait(&mdone_bar[sstage], sphase, 6);
          if (do_b) {
            const uint32_t sbp = smem_u32(smem_b) + sstage * B_STAGE + b_off;
#pragma unroll 8
            for (int i = 0; i < b_rpg; ++i) {
              const int r = bg * b_rpg + i;
              const uint32_t w = ld_shared_u32(sbp + r * 128 + ((b_chunk ^ (r & 7)) << 4));
              bs0 += bf16_lo(w);
              bs1 += bf16_hi(w);
            }
          }
          if (do_a) {
            const uint32_t sap = smem_u32(smem_a) + sstage * A_STAGE_BYTES + a_off;
#pragma unroll 8
            for (int i = 0; i < 16; ++i) {
              const int r = ag * 16 + i;
              const float wr = __shfl_sync(0xffffffffu, wcur, i);
              const uint32_t w = ld_shared_u32(sap + r * 128 + ((a_chunk ^ (r & 7)) << 4));
              as0 += wr * bf16_lo(w);
              as1 += wr * bf16_hi(w);
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty_bar[sstage]);
          if (++sstage == NUM_STAGES) { sstage = 0; sphase ^= 1; }
        }
        }
        if (do_b) {
          float* dst = p.side_bsum + n_blk * p.block_n + rank * b_rows_ + (bp >> 5) * 64 + ((bp & 31) << 1);
          atomicAdd(dst, bs0);
          atomicAdd(dst + 1, bs1);
        }
        if (do_a) {
          const int64_t mo = (int64_t)m_blk * BLOCK_M + (ap >> 5) * 64 + ((ap & 31) << 1);
          if (mo < p.m) atomicAdd(p.side_aw + mo, as0);
          if (mo + 1 < p.m) atomicAdd(p.side_aw + mo + 1, as1);
        }
      }
      mbar_wait(&tfull_bar[acc], acc_phase, 4);
      tc_fence_after();
      const uint32_t taddr0 = tmem_base + ((uint32_t)(q * 32) << 16) + acc * MAX_BLOCK_N;
      if (!(p.debug & 1)) {
#pragma unroll
      for (int ci = 0; ci < 4; ++ci) {
        if (ci * 32 >= ncols) break;
        const int c0 = c_begin + ci * 32;
        uint32_t r[32];
        tmem_ld32(taddr0 + c0, r);
        const int col = ncol0 + c0;
        float4 cvec[8];
        const bool have_cvec = (MODE == MNRF_GEMM_FWD && p.bias) || (MODE == MNRF_GEMM_DGRAD && p.rowv);
        if (have_cvec && c0 + 32 <= p.block_n) {
          const float4* cp = reinterpret_cast<const float4*>((MODE == MNRF_GEMM_FWD ? p.bias : p.colv) + col);
#pragma unroll
          for (int j = 0; j < 8; ++j) cvec[j] = __ldg(cp + j);
        }
        tmem_ld_wait();
        if (MODE == MNRF_GEMM_WGRAD) {
          if (row_ok) {
            float* dst = reinterpret_cast<float*>(p.out) + row * p.ldc + col;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              if (c0 + j < p.block_n)
                red_add_v4(dst + j, __uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                           __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
            }
          }
          continue;
        }
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        if (MODE == MNRF_GEMM_FWD) {
          if (p.bias) {
            if (c0 + 32 <= p.block_n) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                v[4 * j] += cvec[j].x; v[4 * j + 1] += cvec[j].y; v[4 * j + 2] += cvec[j].z; v[4 * j + 3] += cvec[j].w;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] += __ldg(p.bias + min(col + j, p.n - 1));
            }
          }
          if (p.act == MNRF_ACT_RELU) {
            uint32_t bits = 0u;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              v[j] = fmaxf(v[j], 0.f);
              bits |= (v[j] > 0.f ? 1u : 0u) << j;
            }
            mbits[ci] = bits;
          }
        } else {
          if (p.rowv) {
            if (c0 + 32 <= p.block_n) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                v[4 * j] += rv * cvec[j].x; v[4 * j + 1] += rv * cvec[j].y;
                v[4 * j + 2] += rv * cvec[j].z; v[4 * j + 3] += rv * cvec[j].w;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] += rv * __ldg(p.colv + min(col + j, p.n - 1));
            }
          }
          if (p.maskbits) {
            const uint32_t bits = mbits[ci];
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = (bits >> j) & 1u ? v[j] : 0.f;
          } else if (p.mask && row_ok) {
            const uint4* mp = reinterpret_cast<const uint4*>(p.mask + row * p.ldmask + col);
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              if (c0 + g * 8 < p.block_n) {
                uint4 mv = mp[g];
                uint32_t mm[4] = {mv.x, mv.y, mv.z, mv.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  if (!(bf16_lo(mm[e]) > 0.f)) v[g * 8 + 2 * e] = 0.f;
                  if (!(bf16_hi(mm[e]) > 0.f)) v[g * 8 + 2 * e + 1] = 0.f;
                }
              }
            }
          }
        }
        if (MODE == MNRF_GEMM_DGRAD && p.addend && row_ok) {
          const uint4* ap = reinterpret_cast<const uint4*>(p.addend + row * p.ldadd + col);
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            if (c0 + g * 8 < p.block_n) {
              uint4 av = ap[g];
              uint32_t aa[4] = {av.x, av.y, av.z, av.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) { v[g * 8 + 2 * e] += bf16_lo(aa[e]); v[g * 8 + 2 * e + 1] += bf16_hi(aa[e]); }
            }
          }
        }
        if (MODE == MNRF_GEMM_DGRAD && p.colsum && c0 + 32 <= p.block_n) {
          // Column sums over this warp's 32 rows by a shuffle transpose-reduce: each stage halves
          // the values a lane holds; after 5 stages lane j owns column j.  Rows past M hold zeros
          // (TMA zero-fills the A tile, rv = 0).
          float t[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) t[j] = v[j];
#pragma unroll
          for (int sh = 16, n = 32; sh >= 1; sh >>= 1, n >>= 1) {
            const bool up = (lane & sh) != 0;
#pragma unroll
            for (int i = 0; i < n / 2; ++i) {
              const float send = up ? t[i] : t[i + n / 2];
              const float keep = up ? t[i + n / 2] : t[i];
              t[i] = keep + __shfl_xor_sync(0xffffffffu, send, sh);
            }
          }
          if (!cs_resident) atomicAdd(p.colsum + col + lane, t[0]);
          else if (cs_period == 2 && (it & 1)) csodd[ci] += t[0];
          else csacc[ci] += t[0];
        }
        uint4 o[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          o[g].x = pack_bf16(v[g * 8 + 0], v[g * 8 + 1]);
          o[g].y = pack_bf16(v[g * 8 + 2], v[g * 8 + 3]);
          o[g].z = pack_bf16(v[g * 8 + 4], v[g * 8 + 5]);
          o[g].w = pack_bf16(v[g * 8 + 6], v[g * 8 + 7]);
        }
        if (p.debug & 2) continue;
        if (p.use_tma_store) {
          // 64-column groups: two 32-column halves share one 32x128-byte swizzled staging slab
          const int half = ci & 1;
          uint8_t* slab = smem_out + ew * (32 * 128);
          const uint32_t slab_s = smem_u32(slab) + lane * 128;
          if (half == 0) {
            // the bulk store previously issued from this slab must have finished reading it
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
          }
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const int chunk = half * 4 + g;
            st_shared_v4(slab_s + ((chunk ^ (lane & 7)) << 4), o[g].x, o[g].y, o[g].z, o[g].w);
          }
          if (half == 1) {
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              tma_store_2d(&tmap_c, slab, ncol0 + c0 - 32, m_blk * BLOCK_M + q * 32);
              tma_store_commit();
            }
          }
        } else if (row_ok) {
          uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + row * p.ldc + col);
#pragma unroll
          for (int g = 0; g < 4; ++g)
            if (c0 + g * 8 < p.block_n) dst[g] = o[g];
        }
      }
      }
      tc_fence_before();
      if (CTAS == 1) mbar_arrive(&tempty_bar[acc]); else mbar_arrive_leader(&tempty_bar[acc]);
      if (cs_period == 2 && (it & 1)) cs_ncol1 = ncol0; else cs_ncol0 = ncol0;
      if (MODE == MNRF_GEMM_FWD && p.act == MNRF_ACT_RELU && p.maskbits && row_ok && ncols > 0) {
        uint32_t* mp = p.maskbits + row * p.ldmaskbits + (ncol0 >> 5) + w_begin;
        if (nwords == 4) {
          *reinterpret_cast<uint4*>(mp) = make_uint4(mbits[0], mbits[1], mbits[2], mbits[3]);
        } else {
#pragma unroll
          for (int w = 0; w < 4; ++w)
            if (w < nwords) mp[w] = mbits[w];
        }
      }
    }
    if (MODE == MNRF_GEMM_DGRAD && p.colsum && cs_resident) {
#pragma unroll
      for (int ci = 0; ci < 4; ++ci) {
        if (ci * 32 + 32 > ncols) continue;
        if (cs_ncol0 >= 0) atomicAdd(p.colsum + cs_ncol0 + c_begin + ci * 32 + lane, csacc[ci]);
        if (cs_ncol1 >= 0) atomicAdd(p.colsum + cs_ncol1 + c_begin + ci * 32 + lane, csodd[ci]);
      }
    }
    if (p.use_tma_store && lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  if (CTAS == 1) __syncthreads(); else cluster_sync_all();    // no peer may still signal this CTA's barriers
  if (warp == 2) tmem_dealloc<CTAS>(tmem_base, 512);
}

// ------------------------------------------------------------------------------------ host
static int pick_block_n(int n) {
  const int cands[] = {256, 128, 64, 32, 16};
  for (int c : cands)
    if (n % c == 0) return c;
  return 0;
}

int gemm_tc_launch(const mnrf_gemm_desc* d, const mnrf_bf16* a, const mnrf_bf16* b, const float* bias,
                   const float* rowv, const float* colv, const mnrf_bf16* mask, uint32_t* maskbits,
                   float* colsum, const mnrf_bf16* addend, float* side_bsum, const float* side_w, float* side_aw,
                   void* out, cudaStream_t stream) {
  // K-major modes: the reduction index is the contiguous one and layers are padded to 64.  WGRAD reduces
  // over the sample rows, any count: the last 64-row block is zero-filled by TMA past the tensor's end.
  MNRF_CHECK(d->mode == MNRF_GEMM_WGRAD || d->k % BLOCK_K == 0,
             "mnrf_gemm(tc): reduction length %d must be a multiple of %d", d->k, BLOCK_K);
  MNRF_CHECK(d->lda % 8 == 0 && d->ldb % 8 == 0 && ((uintptr_t)a % 16) == 0 && ((uintptr_t)b % 16) == 0,
             "mnrf_gemm(tc): operands must be 16-byte aligned with ld %% 8 == 0");
  GemmParams p{};
  p.mode = d->mode; p.act = d->act; p.m = d->m; p.n = d->n; p.k = d->k;
  p.block_n = pick_block_n(d->n);
  MNRF_CHECK(p.block_n > 0, "mnrf_gemm(tc): N=%d must be a multiple of 16", d->n);
  if (d->mode == MNRF_GEMM_WGRAD)
    MNRF_CHECK(p.block_n >= 64, "mnrf_gemm(tc): WGRAD needs N %% 64 == 0 (MN-major 128-byte atoms), N=%d", d->n);
  p.num_m_blocks = (int)((d->m + BLOCK_M - 1) / BLOCK_M);
  p.num_n_blocks = d->n / p.block_n;
  p.num_k_blocks = (d->k + BLOCK_K - 1) / BLOCK_K;
  p.ldc = d->ldc; p.ldmask = d->ldmask;
  p.bias = bias; p.rowv = rowv; p.colv = colv;
  p.mask = reinterpret_cast<const __nv_bfloat16*>(mask);
  p.out = out;
  p.maskbits = maskbits;
  p.ldmaskbits = d->ldmaskbits;
  p.mask_mod = d->mask_mod;
  p.addend = reinterpret_cast<const __nv_bfloat16*>(addend);
  p.ldadd = d->ldadd;
  if (addend) MNRF_CHECK(d->mode == MNRF_GEMM_DGRAD && d->ldadd % 8 == 0 && ((uintptr_t)addend % 16) == 0,
                         "mnrf_gemm(tc): addend is a DGRAD input with 16-byte aligned rows");
  p.side_bsum = side_bsum; p.side_w = side_w; p.side_aw = side_aw;
  if (side_bsum || side_aw) MNRF_CHECK(d->mode == MNRF_GEMM_WGRAD, "mnrf_gemm(tc): side sums belong to WGRAD");
  p.colsum = colsum;
  if (colsum) MNRF_CHECK(d->mode == MNRF_GEMM_DGRAD && p.block_n % 32 == 0,
                         "mnrf_gemm(tc): colsum is a DGRAD output and needs N %% 32 == 0");
  if (maskbits) {
    MNRF_CHECK(d->mode != MNRF_GEMM_WGRAD, "mnrf_gemm(tc): maskbits make no sense for WGRAD");
    MNRF_CHECK(d->n % 32 == 0 && p.block_n % 32 == 0 && d->ldmaskbits * 32 >= d->n,
               "mnrf_gemm(tc): maskbits need N %% 32 == 0 and ldmaskbits >= N/32");
    MNRF_CHECK(p.block_n != MAX_BLOCK_N || (d->ldmaskbits % 4 == 0 && ((uintptr_t)maskbits % 16) == 0),
               "mnrf_gemm(tc): maskbits rows must be 16-byte aligned");
  }
  if (bias) MNRF_CHECK(((uintptr_t)bias % 16) == 0, "mnrf_gemm(tc): bias must be 16-byte aligned");
  if (colv) MNRF_CHECK(((uintptr_t)colv % 16) == 0, "mnrf_gemm(tc): colv must be 16-byte aligned");
  p.use_tma_store = (d->mode != MNRF_GEMM_WGRAD && p.block_n % 64 == 0) ? 1 : 0;
#ifdef MNRF_TIMING_KNOBS
  // timing experiments only (results are wrong by construction): compiled in only on request
  static const int cfg_debug = getenv("MNRF_GEMM_DEBUG") ? atoi(getenv("MNRF_GEMM_DEBUG")) : 0;
#else
  static const int cfg_debug = 0;
#endif
  p.debug = cfg_debug;
  const int sms = mnrf_num_sms();
  // CTA pairs (tcgen05 cta_group::2) whenever the tile grid is made of whole 256 x 256 tiles
  const int ctas = (p.block_n == MAX_BLOCK_N && d->m % (2 * BLOCK_M) == 0 && sms % 2 == 0) ? 2 : 1;
  const int workers = sms / ctas;
  p.num_splits = 1;
  if (d->mode == MNRF_GEMM_WGRAD) {
    // Split the reduction over the sample rows so that (output tiles x splits) work items fill whole rounds of the
    // workers -- with the FEWEST splits that do: every work item ends in a 256 x 256 fp32 red.add pass over its
    // output tile, and for a one-tile weight gradient (PropMLP 256 x 256) those passes all hit the same 256 KB of
    // L2.  (148 splits there cost a fixed ~25 us per launch -- ncu, 2048-ray shard: 48 us against 21 us of streaming.)
    const int out_tiles = (p.num_m_blocks / ctas) * p.num_n_blocks;
    const int max_splits = std::min(std::max(1, (2 * workers) / out_tiles), p.num_k_blocks);
    int splits = max_splits;
    for (int sp = 1; sp <= max_splits; ++sp) {
      const int items = out_tiles * sp;
      const int rounds = (items + workers - 1) / workers;
      if (items * 100 >= rounds * workers * 95) { splits = sp; break; }
    }
    p.num_splits = splits;
  }
  p.kblocks_per_split = (p.num_k_blocks + p.num_splits - 1) / p.num_splits;
  p.num_splits = (p.num_k_blocks + p.kblocks_per_split - 1) / p.kblocks_per_split;
  if (d->mode != MNRF_GEMM_WGRAD) {
    MNRF_CHECK(d->ldc % 8 == 0 && ((uintptr_t)out % 16) == 0, "mnrf_gemm(tc): bf16 output must be 16-byte aligned");
    if (mask) MNRF_CHECK(d->ldmask % 8 == 0 && ((uintptr_t)mask % 16) == 0, "mnrf_gemm(tc): mask must be 16-byte aligned");
  } else {
    MNRF_CHECK(d->ldc % 4 == 0 && ((uintptr_t)out % 16) == 0, "mnrf_gemm(tc): fp32 output must be 16-byte aligned");
  }

  CUtensorMap ta, tb, tc;
  memset(&tc, 0, sizeof(tc));
  if (d->mode != MNRF_GEMM_WGRAD) {
    if (make_tmap(&ta, a, d->m, d->k, d->lda, BLOCK_K, BLOCK_M)) return 1;
    if (make_tmap(&tb, b, d->n, d->k, d->ldb, BLOCK_K, p.block_n / ctas)) return 1;
    if (p.use_tma_store && make_tmap(&tc, out, d->m, d->n, d->ldc, 64, 32)) return 1;
  } else {
    // A = X[R, Mo], B = dY[R, N]; reduction index on rows
    if (make_tmap(&ta, a, d->k, d->m, d->lda, 64, BLOCK_K)) return 1;
    if (make_tmap(&tb, b, d->k, d->n, d->ldb, 64, BLOCK_K)) return 1;
  }
  const int total_tiles = (p.num_m_blocks / ctas) * p.num_n_blocks * p.num_splits;
  const int grid = std::min(total_tiles, workers) * ctas;
  if (grid == 0) return 0;
#define MNRF_LAUNCH_TC(MODE_, CTAS_)                                                                  \
  do {                                                                                                \
    static bool attr_set = false;                                                                     \
    constexpr int kSmem = smem_bytes(CTAS_);                                                          \
    static_assert(kSmem <= 232448, "shared memory budget");                                           \
    auto kern = gemm_tc_kernel<MODE_, CTAS_>;                                                         \
    if (!attr_set) {                                                                                  \
      MNRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));      \
      attr_set = true;                                                                                \
    }                                                                                                 \
    cudaLaunchConfig_t cfg = {};                                                                      \
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(NUM_THREADS);                                       \
    cfg.dynamicSmemBytes = kSmem; cfg.stream = stream;                                                \
    cudaLaunchAttribute attr[1];                                                                      \
    attr[0].id = cudaLaunchAttributeClusterDimension;                                                 \
    attr[0].val.clusterDim.x = CTAS_; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;     \
    cfg.attrs = attr; cfg.numAttrs = 1;                                                               \
    MNRF_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tc, p));                                         \
  } while (0)
  if (ctas == 2) {
    if (d->mode == MNRF_GEMM_FWD) MNRF_LAUNCH_TC(MNRF_GEMM_FWD, 2);
    else if (d->mode == MNRF_GEMM_DGRAD) MNRF_LAUNCH_TC(MNRF_GEMM_DGRAD, 2);
    else MNRF_LAUNCH_TC(MNRF_GEMM_WGRAD, 2);
  } else {
    if (d->mode == MNRF_GEMM_FWD) MNRF_LAUNCH_TC(MNRF_GEMM_FWD, 1);
    else if (d->mode == MNRF_GEMM_DGRAD) MNRF_LAUNCH_TC(MNRF_GEMM_DGRAD, 1);
    else MNRF_LAUNCH_TC(MNRF_GEMM_WGRAD, 1);
  }
  MNRF_LAUNCH_CHECK();
  return 0;
}

}  // namespace mnrf
