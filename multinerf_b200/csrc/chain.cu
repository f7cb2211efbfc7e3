// Layer-chained 256-wide MLP trunk on 5th-gen tensor cores (sm_100a): ONE persistent launch walks
// row blocks of samples through ALL Dense layers of a trunk (forward) or through its whole
// input-gradient chain (backward).  Replaces the per-layer launches of models.py:441-465
// (`x = dense_layer(net_width)(x); x = net_activation(x)`, skip-concat as extra K blocks) and of the
// matching reverse-mode chain, for the 256-wide MLPs (PropMLP of 360.gin; PropMLP/NerfMLP of the
// blender / llff / Ref-NeRF / RawNeRF configs).
//
// Why: a 256-wide layer has 128 FLOP per byte of activation traffic when every layer reads its input
// from HBM and writes its output back -- below the machine balance (~225 FLOP/B) -- so the per-layer
// kernels are HBM-bound (profiles/r01_final_gemm_traffic.txt: 29-41 % tensor pipe).  Here the
// activations of a row block stay in shared memory between layers (they are written out ONCE, for
// the weight-gradient pass), accumulators live in TMEM, weights stream from L2 through a TMA ring.
//
// Work decomposition (per two-CTA cluster = one TPC, tcgen05 cta_group::2):
//   unit    = 512 sample rows = two row blocks X in {A, B} of 256 rows (128 per CTA);
//   phase   = one layer of one row block: MMA 256 x 256 x K into the TMEM accumulator of X
//             (columns X*256 .. X*256+255 in both CTAs), then an epilogue that turns the accumulator
//             into the next layer's A operand in shared memory (SWIZZLE_128B K-major, 4 k-blocks);
//   ping-pong: MMA(B, l) runs while the epilogue warps work on (A, l); MMA(A, l+1) while they work on
//             (B, l): the tensor pipe only waits when an epilogue is slower than a phase of MMAs.
//   weights : k-blocks [128 N-rows of this CTA x 64 K] stream through a ring of six 16 KB slots.  The four
//             k-blocks that multiply the RESIDENT operand are loaded once per layer and used by both
//             row blocks (held during A's phase, released during B's); k-blocks that multiply a
//             STREAMED operand (IPE features of layer 0 / of a skip layer, or the incoming gradient of
//             the backward chain) travel in (weight, operand) slot pairs and are released at once.
//             To keep the ring's release order FIFO, A's phase runs streamed-then-resident and B's phase
//             resident-then-streamed.
//
//   warp 0   : TMA producer (one elected lane per CTA)
//   warp 1   : MMA issuer (leader CTA, one elected lane)
//   warp 2   : TMEM allocator (512 columns = the two accumulators)
//   warp 3   : store warp: once the epilogue threads have written an activation block it issues the bulk stores
//              of that block (TMA) and tells the epilogue when the block may be overwritten
//   warps 4-11: epilogue (two warps per TMEM lane quadrant, 128 columns each)
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "tc_common.cuh"

namespace mnrf {

constexpr int CH_W = 256;                   // layer width: N of every MMA, K of the resident operand
constexpr int CH_SLOT = 16384;              // one [128 rows x 64 bf16] k-block, SWIZZLE_128B
constexpr int CH_SLOTS = 6;
constexpr int CH_ACT = 4 * CH_SLOT;         // a 128 x 256 bf16 activation block = 4 k-blocks
constexpr int CH_EPI_WARPS = 8;
constexpr int CH_EPI_THREADS = CH_EPI_WARPS * 32;
constexpr int CH_THREADS = 128 + CH_EPI_THREADS;
constexpr int CH_MAX_LAYERS = MNRF_CHAIN_MAX_LAYERS;
constexpr int CH_UNIT_ROWS = 512;
constexpr int CH_SMEM = 2 * CH_ACT + CH_SLOTS * CH_SLOT + 1024 /*head partials*/ + 256 /*barriers*/ + 1024 /*align*/;
static_assert(CH_SMEM <= 232448, "shared memory budget");

struct alignas(64) ChainMaps {
  CUtensorMap stream;
  CUtensorMap w[CH_MAX_LAYERS];
  CUtensorMap out[CH_MAX_LAYERS];
};

struct ChainLayer {
  int n_stream, stream_col0, stream_kb0;
  int n_res, res_kb0;
  int store;
  const float* bias;
  uint32_t* maskbits;
  int64_t ldmaskbits;
  float* colsum;
};

struct ChainParams {
  int num_layers;
  int64_t m;
  int64_t num_units;
  ChainLayer layer[CH_MAX_LAYERS];
  const float* head_w;      // FWD: Dense(1) on the last layer's output (density head), fp32 copy of the bf16 row
  const float* head_b;
  float* head_out;
  int prefetch;             // pull the next unit's streamed tiles into L2 ahead of time (render form only)
  long long* trace;         // -DMNRF_TIMING_KNOBS + MNRF_CHAIN_TRACE=<device ptr>: clock64 event log of CTA 0
  int debug;                // MNRF_CHAIN_DEBUG (timing experiments, -DMNRF_TIMING_KNOBS builds only; results are wrong):
                            // 1 = no epilogue math/smem writes, 2 = no bulk stores, 4 = no mask / head global writes
};

// two fp32 -> packed bf16x2 with ReLU in the conversion (one instruction for both lanes)
__device__ __forceinline__ uint32_t pack_bf16_relu(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
#ifdef MNRF_TIMING_KNOBS
// event log of the leader CTA of pair 0: trace[0] = event count, then (tag, unit*100 + j*10 + X, clock64) triples
#define CH_TRACE(tag, unit, j, X)                                                              \
  do {                                                                                          \
    if (p.trace && blockIdx.x == 0 && (unit) < 3 * (gridDim.x >> 1)) {                          \
      const unsigned long long n_ = atomicAdd((unsigned long long*)p.trace, 1ull);              \
      if (n_ < 4000) {                                                                          \
        p.trace[1 + 3 * n_] = (tag); p.trace[2 + 3 * n_] = (long long)((unit) * 100 + (j) * 10 + (X)); \
        p.trace[3 + 3 * n_] = clock64();                                                        \
      }                                                                                         \
    }                                                                                           \
  } while (0)
#else
#define CH_TRACE(tag, unit, j, X) do {} while (0)
#endif
__device__ __forceinline__ void named_bar_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
// MODE 0: forward  -- epilogue = + bias, ReLU, 1-bit masks out, bf16 activation to smem (+ HBM), density head
// MODE 1: backward -- epilogue = x ReLU mask (bits in), bias-gradient column sums, bf16 gradient to smem + HBM
template <int MODE>
__global__ void __launch_bounds__(CH_THREADS, 1)
mlp_chain_kernel(const __grid_constant__ ChainMaps maps, const ChainParams p) {
  extern __shared__ uint8_t smem_dyn[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  uint8_t* act = smem;                                     // [2][CH_ACT]
  uint8_t* ring = smem + 2 * CH_ACT;                       // [CH_SLOTS][CH_SLOT]
  float* hpart = reinterpret_cast<float*>(ring + CH_SLOTS * CH_SLOT);      // [2][128] head partial of column half 1, per block
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(hpart) + 1024);
  uint64_t* full_bar = bars;                               // [CH_SLOTS]  (the leader's are used)
  uint64_t* empty_bar = bars + CH_SLOTS;                   // [CH_SLOTS]
  uint64_t* acc_full = bars + 2 * CH_SLOTS;                // [2] accumulator of block X complete
  uint64_t* act_ready = acc_full + 2;                      // [2] (leader's) epilogue of block X done in both CTAs
  uint64_t* buf_free = act_ready + 2;                      // [2] the bulk store has finished reading block X
  uint64_t* blk_written = buf_free + 2;                    // [2] all epilogue threads of this CTA have written block X
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(blk_written + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const int64_t pair = blockIdx.x >> 1;
  const int64_t num_pairs = gridDim.x >> 1;

  if (warp == 0 && elect_one()) {
    bool any_stream = false;
    for (int j = 0; j < p.num_layers; ++j) {
      prefetch_tmap(&maps.w[j]);
      if (p.layer[j].store) prefetch_tmap(&maps.out[j]);
      any_stream |= p.layer[j].n_stream > 0;
    }
    if (any_stream) prefetch_tmap(&maps.stream);
  }
  if (warp == 1 && elect_one()) {
    for (int i = 0; i < CH_SLOTS; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&act_ready[i], 2 * CH_EPI_THREADS);
      mbar_init(&buf_free[i], 1);
      mbar_init(&blk_written[i], CH_EPI_THREADS);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<2>(tmem_ptr, 512);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (elect_one()) {
      uint32_t slot = 0, phase = 0;
      auto load = [&](const CUtensorMap* map, int c0, int c1) {
        mbar_wait(&empty_bar[slot], phase ^ 1, 1);
        if (rank == 0) mbar_expect_tx(&full_bar[slot], 2 * CH_SLOT);
        tma_load_2d_pair(ring + slot * CH_SLOT, map, &full_bar[slot], c0, c1);
        if (++slot == CH_SLOTS) { slot = 0; phase ^= 1; }
      };
      for (int64_t unit = pair; unit < p.num_units; unit += num_pairs) {
        // The streamed operand comes from HBM: with three k-blocks in flight (1.5k cycles of MMA work) a cold
        // DRAM access (~3k cycles) stalls the first layer, so the NEXT unit's tiles are pulled into L2 now -- but
        // only in the render form.  With every layer's activations streaming out through L2 (training form,
        // backward) the prefetched lines are evicted before they are used and the operand is read from DRAM
        // twice (ncu: 1.98 GB read for 1.07 GB of features), on a launch that is HBM-bound to begin with.
        if (p.prefetch && unit + num_pairs < p.num_units) {
          for (int j = 0; j < p.num_layers; ++j) {
            const ChainLayer& L = p.layer[j];
            for (int X = 0; X < 2; ++X) {
              const int prow = (int)((unit + num_pairs) * CH_UNIT_ROWS + X * 256 + rank * 128);
              for (int s2 = 0; s2 < L.n_stream; ++s2) tma_prefetch_2d(&maps.stream, L.stream_col0 + s2 * 64, prow);
            }
          }
        }
        for (int j = 0; j < p.num_layers; ++j) {
          const ChainLayer& L = p.layer[j];
          for (int X = 0; X < 2; ++X) {
            const int row0 = (int)(unit * CH_UNIT_ROWS + X * 256 + rank * 128);
            auto stream_part = [&]() {
              for (int s = 0; s < L.n_stream; ++s) {
                load(&maps.w[j], (L.stream_kb0 + s) * 64, rank * 128);      // this CTA's half of the N rows
                load(&maps.stream, L.stream_col0 + s * 64, row0);           // this CTA's 128 sample rows
              }
            };
            if (X == 0) {
              stream_part();
              for (int r = 0; r < L.n_res; ++r) load(&maps.w[j], (L.res_kb0 + r) * 64, rank * 128);
            } else {
              stream_part();          // the resident-operand weights are already in the ring (held since X = 0)
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA, one lane) =====================
    if (rank == 0 && elect_one()) {
      const uint32_t idesc = make_idesc(256, CH_W, 0, 0);
      const uint32_t ring_addr = smem_u32(ring), act_addr = smem_u32(act);
      uint32_t slot = 0, phase = 0, res_slot = 0;
      uint32_t nready[2] = {0u, 0u};
      for (int64_t unit = pair; unit < p.num_units; unit += num_pairs) {
        for (int j = 0; j < p.num_layers; ++j) {
          const ChainLayer& L = p.layer[j];
          for (int X = 0; X < 2; ++X) {
            // accumulator X drained and (for resident operands) activation block X written, in both CTAs
            CH_TRACE(10, unit, j, X);
            mbar_wait(&act_ready[X], (nready[X] & 1u) ^ 1u, 2);
            ++nready[X];
            tc_fence_after();
            CH_TRACE(11, unit, j, X);
            const uint32_t tmem_d = tmem_base + (uint32_t)X * CH_W;
            uint32_t accumulate = 0u;
            auto mma_kblock = [&](uint32_t a_addr, uint32_t b_addr) {
#pragma unroll
              for (int k = 0; k < 64 / UMMA_K; ++k) {
                umma_bf16<2>(tmem_d, make_smem_desc(a_addr + k * (UMMA_K * 2), 0, 1024),
                             make_smem_desc(b_addr + k * (UMMA_K * 2), 0, 1024), idesc, accumulate);
                accumulate = 1u;
              }
            };
            auto stream_part = [&]() {
              for (int s = 0; s < L.n_stream; ++s) {
                const uint32_t ws = slot;
                mbar_wait(&full_bar[ws], phase, 3);
                if (++slot == CH_SLOTS) { slot = 0; phase ^= 1; }
                const uint32_t as = slot;
                mbar_wait(&full_bar[as], phase, 3);
                if (++slot == CH_SLOTS) { slot = 0; phase ^= 1; }
                tc_fence_after();
                mma_kblock(ring_addr + as * CH_SLOT, ring_addr + ws * CH_SLOT);
                umma_commit<2>(&empty_bar[ws]);
                umma_commit<2>(&empty_bar[as]);
              }
            };
            auto res_part = [&]() {
              for (int r = 0; r < L.n_res; ++r) {
                uint32_t ws;
                if (X == 0) {
                  ws = slot;
                  if (r == 0) res_slot = slot;
                  mbar_wait(&full_bar[ws], phase, 3);
                  if (++slot == CH_SLOTS) { slot = 0; phase ^= 1; }
                  tc_fence_after();
                } else {
                  ws = res_slot + r;
                  if (ws >= CH_SLOTS) ws -= CH_SLOTS;
                }
                mma_kblock(act_addr + X * CH_ACT + r * CH_SLOT, ring_addr + ws * CH_SLOT);
                if (X == 1) umma_commit<2>(&empty_bar[ws]);       // second and last user: free the slot
              }
            };
            if (X == 0) { stream_part(); res_part(); } else { res_part(); stream_part(); }
            umma_commit<2>(&acc_full[X]);
            CH_TRACE(12, unit, j, X);
          }
        }
      }
    }
  } else if (warp == 3) {
    // ===================== store warp (both CTAs) =====================
    // Waits until all epilogue threads of this CTA have written (and fenced) an activation block, issues its bulk
    // stores and tells the epilogue when the block may be overwritten.  (The MMA issuer is signalled by the
    // epilogue threads themselves, so the stores are off the critical path.)
    if (lane == 0) {
      uint32_t nwritten[2] = {0u, 0u};
      for (int64_t unit = pair; unit < p.num_units; unit += num_pairs) {
        for (int j = 0; j < p.num_layers; ++j) {
          const ChainLayer& L = p.layer[j];
          for (int X = 0; X < 2; ++X) {
            mbar_wait(&blk_written[X], nwritten[X] & 1u, 6);
            ++nwritten[X];
            CH_TRACE(30, unit, j, X);
            if (L.store
#ifdef MNRF_TIMING_KNOBS
                && !(p.debug & 2)
#endif
            ) {
              const int row0 = (int)(unit * CH_UNIT_ROWS + X * 256 + rank * 128);
              const uint8_t* ablk = act + X * CH_ACT;
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4) tma_store_2d(&maps.out[j], ablk + k4 * CH_SLOT, k4 * 64, row0);
              tma_store_commit();
              tma_store_wait_read<0>();                 // the block may be overwritten once the store has read it
            }
            mbar_arrive(&buf_free[X]);
            CH_TRACE(32, unit, j, X);
          }
        }
      }
      tma_store_wait_all();
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int q = warp & 3;                 // TMEM lane quadrant this warp may touch
    const int ew = warp - 4;
    const int half = ew >> 2;               // column half: [half*128, half*128 + 128)
    const int r_blk = q * 32 + lane;        // row within the CTA's 128-row block
    // shared-space addresses of this thread's row in the two activation blocks, and the eight swizzled 16-byte
    // chunk offsets of a 128-byte row (SWIZZLE_128B: chunk index XOR (row & 7))
    const uint32_t row_s = smem_u32(act) + (uint32_t)r_blk * 128u;
    uint32_t swz[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) swz[c] = (uint32_t)((c ^ (r_blk & 7)) << 4);
    const uint32_t taddr_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * 128);
    uint32_t nfull[2] = {0u, 0u};
    float csacc[CH_MAX_LAYERS][4];
#pragma unroll
    for (int jj = 0; jj < CH_MAX_LAYERS; ++jj)
#pragma unroll
      for (int c = 0; c < 4; ++c) csacc[jj][c] = 0.f;

    for (int64_t unit = pair; unit < p.num_units; unit += num_pairs) {
      for (int j = 0; j < p.num_layers; ++j) {
        const ChainLayer& L = p.layer[j];
        const bool last = (j == p.num_layers - 1);
        const bool do_head = (MODE == 0) && last && p.head_w != nullptr;
        for (int X = 0; X < 2; ++X) {
          const int64_t row0 = unit * CH_UNIT_ROWS + X * 256 + rank * 128;
          const int64_t row = row0 + r_blk;
          const bool row_ok = row < p.m;
          uint32_t mbits[4] = {0u, 0u, 0u, 0u};
          if (MODE == 1 && L.maskbits && row_ok) {
            const uint4 t = *reinterpret_cast<const uint4*>(L.maskbits + row * L.ldmaskbits + half * 4);
            mbits[0] = t.x; mbits[1] = t.y; mbits[2] = t.z; mbits[3] = t.w;
          }
          if (ew == 0 && lane == 0) CH_TRACE(20, unit, j, X);
          mbar_wait(&acc_full[X], nfull[X] & 1u, 4);
          ++nfull[X];
          tc_fence_after();
          if (ew == 0 && lane == 0) CH_TRACE(21, unit, j, X);
          // the bulk store that last read this activation block (two phases ago) must have finished reading it
          mbar_wait(&buf_free[X], (nfull[X] & 1u), 5);      // nfull already counts this phase: parity of the previous one
          const uint32_t blk_s = row_s + (uint32_t)(X * CH_ACT + half * 2 * CH_SLOT);
          float hdot = 0.f;
#ifdef MNRF_TIMING_KNOBS
          if (!(p.debug & 1))
#endif
#pragma unroll
          for (int ci = 0; ci < 4; ++ci) {
            const int c0 = half * 128 + ci * 32;      // first of this pass's 32 columns
            uint32_t r[32];
            tmem_ld32(taddr_row + (uint32_t)(X * CH_W + ci * 32), r);
            tmem_ld_wait();
            float v[32];
#pragma unroll
            for (int t = 0; t < 32; ++t) v[t] = __uint_as_float(r[t]);
            uint32_t o[16];
            if (MODE == 0) {
              const float4* cp = reinterpret_cast<const float4*>(L.bias + c0);
#pragma unroll
              for (int t = 0; t < 8; ++t) {
                const float4 bv = __ldg(cp + t);
                v[4 * t] += bv.x; v[4 * t + 1] += bv.y; v[4 * t + 2] += bv.z; v[4 * t + 3] += bv.w;
              }
              // ReLU is folded into the bf16 conversion (cvt.rn.relu); the mask is the sign of the fp32
              // pre-activation (v > 0  <=>  stored activation > 0: bf16 keeps fp32's exponent range)
              uint32_t bits = 0u;
#pragma unroll
              for (int t = 0; t < 32; ++t) bits |= (v[t] > 0.f ? 1u : 0u) << t;
              mbits[ci] = bits;
#pragma unroll
              for (int t = 0; t < 16; ++t) o[t] = pack_bf16_relu(v[2 * t], v[2 * t + 1]);
              if (do_head) {
                // Dense(1) on the bf16-rounded activation, fp32 accumulate (what the head kernel computes)
                const float4* hw = reinterpret_cast<const float4*>(p.head_w + c0);
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                  const float4 h = __ldg(hw + t);
                  hdot += bf16_lo(o[2 * t]) * h.x + bf16_hi(o[2 * t]) * h.y + bf16_lo(o[2 * t + 1]) * h.z +
                          bf16_hi(o[2 * t + 1]) * h.w;
                }
              }
            } else {
              if (L.maskbits) {
                const uint32_t bits = mbits[ci];
#pragma unroll
                for (int t = 0; t < 32; ++t) v[t] = (bits >> t) & 1u ? v[t] : 0.f;
              }
#pragma unroll
              for (int t = 0; t < 16; ++t) o[t] = pack_bf16(v[2 * t], v[2 * t + 1]);
              if (L.colsum) {
                // column sums over this warp's 32 rows, in place on v (already packed): shuffle transpose-reduce,
                // lane t ends with column t; rows past M hold zeros (zero-filled operand, zero mask)
#pragma unroll
                for (int sh = 16, n = 32; sh >= 1; sh >>= 1, n >>= 1) {
                  const bool up = (lane & sh) != 0;
#pragma unroll
                  for (int i = 0; i < n / 2; ++i) {
                    const float send = up ? v[i] : v[i + n / 2];
                    const float keep = up ? v[i + n / 2] : v[i];
                    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, sh);
                  }
                }
#pragma unroll
                for (int jj = 0; jj < CH_MAX_LAYERS; ++jj)
                  if (jj == j) csacc[jj][ci] += v[0];
              }
            }
            // K-major SWIZZLE_128B k-block (the layout TMA produces and UMMA / the bulk store consume)
            const uint32_t kb_s = blk_s + (uint32_t)((ci >> 1) * CH_SLOT);
#pragma unroll
            for (int g = 0; g < 4; ++g)
              st_shared_v4(kb_s + swz[(ci & 1) * 4 + g], o[4 * g], o[4 * g + 1], o[4 * g + 2], o[4 * g + 3]);
          }
          if (ew == 0 && lane == 0) CH_TRACE(23, unit, j, X);
          tc_fence_before();
          fence_proxy_async();                // generic-proxy writes -> visible to UMMA / TMA (async proxy)
          // accumulator X drained + this thread's part of block X written: signal the MMA issuer (leader CTA) and
          // the store warp.  Plain (CTA-scope) arrives: no DATA crosses SMs here -- each CTA's tensor core reads
          // its own rows of the A operand from its own shared memory -- so a cluster-scope release (MEMBAR.ALL.GPU
          // in SASS) is not needed.
          mbar_arrive_leader(&act_ready[X]);
          mbar_arrive(&blk_written[X]);
          if (ew == 0 && lane == 0) CH_TRACE(25, unit, j, X);
#ifdef MNRF_TIMING_KNOBS
          if (p.debug & 4) continue;
#endif
          if (MODE == 0) {
            if (L.maskbits && row_ok)
              *reinterpret_cast<uint4*>(L.maskbits + row * L.ldmaskbits + half * 4) =
                  make_uint4(mbits[0], mbits[1], mbits[2], mbits[3]);
            if (do_head) {
              // the two column halves of a row meet in shared memory (warps of one half only sync among the
              // 256 epilogue threads here, once per unit and block -- off the MMA's critical path)
              if (half == 1) hpart[X * 128 + r_blk] = hdot;
              named_bar_sync(1, CH_EPI_THREADS);
              if (half == 0 && row_ok)
                p.head_out[row] = (hdot + hpart[X * 128 + r_blk]) + (p.head_b ? __ldg(p.head_b) : 0.f);
            }
          }
        }
      }
    }
    if (MODE == 1) {
#pragma unroll
      for (int jj = 0; jj < CH_MAX_LAYERS; ++jj) {
        if (jj < p.num_layers && p.layer[jj].colsum) {
#pragma unroll
          for (int ci = 0; ci < 4; ++ci) atomicAdd(p.layer[jj].colsum + half * 128 + ci * 32 + lane, csacc[jj][ci]);
        }
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();           // no peer may still signal this CTA's barriers / read its shared memory
  if (warp == 2) tmem_dealloc<2>(tmem_base, 512);
}

}  // namespace mnrf

extern "C" int mnrf_mlp_chain_max_layers(void) { return mnrf::CH_MAX_LAYERS; }

extern "C" int mnrf_mlp_chain(const mnrf_chain_desc* d, mnrf_stream stream_) {
  using namespace mnrf;
  cudaStream_t stream = (cudaStream_t)stream_;
  MNRF_CHECK(d, "mnrf_mlp_chain: null descriptor");
  if (d->m == 0) return 0;
  MNRF_CHECK(d->mode == MNRF_CHAIN_FWD || d->mode == MNRF_CHAIN_BWD, "mnrf_mlp_chain: bad mode %d", d->mode);
  MNRF_CHECK(d->num_layers >= 1 && d->num_layers <= CH_MAX_LAYERS, "mnrf_mlp_chain: 1..%d layers, got %d",
             CH_MAX_LAYERS, d->num_layers);
  MNRF_CHECK(d->width == CH_W, "mnrf_mlp_chain: layer width must be %d, got %d", CH_W, d->width);
  const int sms = mnrf_num_sms();
  MNRF_CHECK(sms >= 2, "mnrf_mlp_chain: needs CTA pairs");
  ChainMaps maps;
  memset(&maps, 0, sizeof(maps));
  ChainParams p{};
  p.num_layers = d->num_layers;
  p.m = d->m;
  p.num_units = (d->m + CH_UNIT_ROWS - 1) / CH_UNIT_ROWS;
  bool any_stream = false;
  for (int j = 0; j < d->num_layers; ++j) {
    const mnrf_chain_layer& s = d->layer[j];
    ChainLayer& L = p.layer[j];
    MNRF_CHECK(s.n_res == 0 || s.n_res == CH_W / 64, "mnrf_mlp_chain: layer %d: n_res must be 0 or %d", j, CH_W / 64);
    MNRF_CHECK(s.n_stream >= 0 && (s.n_stream > 0 || s.n_res > 0), "mnrf_mlp_chain: layer %d has no operand", j);
    MNRF_CHECK(j > 0 || s.n_res == 0, "mnrf_mlp_chain: the first layer has no resident operand");
    MNRF_CHECK(s.w && ((uintptr_t)s.w % 16) == 0 && s.ldw % 8 == 0, "mnrf_mlp_chain: layer %d: weights must be 16-byte aligned", j);
    const int kblocks = std::max(s.n_stream > 0 ? s.stream_kb0 + s.n_stream : 0, s.n_res > 0 ? s.res_kb0 + s.n_res : 0);
    MNRF_CHECK(s.ldw >= (int64_t)kblocks * 64, "mnrf_mlp_chain: layer %d: weight pitch %lld < K %d", j, (long long)s.ldw, kblocks * 64);
    L.n_stream = s.n_stream; L.stream_col0 = s.stream_col0; L.stream_kb0 = s.stream_kb0;
    L.n_res = s.n_res; L.res_kb0 = s.res_kb0;
    L.store = s.out ? 1 : 0;
    L.bias = s.bias; L.maskbits = s.maskbits; L.ldmaskbits = s.ldmaskbits; L.colsum = s.colsum;
    if (s.bias) MNRF_CHECK(((uintptr_t)s.bias % 16) == 0, "mnrf_mlp_chain: layer %d: bias must be 16-byte aligned", j);
    if (s.maskbits)
      MNRF_CHECK(s.ldmaskbits % 4 == 0 && s.ldmaskbits >= CH_W / 32 && ((uintptr_t)s.maskbits % 16) == 0,
                 "mnrf_mlp_chain: layer %d: maskbits rows must be 16-byte aligned, >= %d words", j, CH_W / 32);
    if (d->mode == MNRF_CHAIN_BWD) MNRF_CHECK(!s.bias, "mnrf_mlp_chain: bias is a forward input");
    else MNRF_CHECK(!s.colsum, "mnrf_mlp_chain: colsum is a backward output");
    // K-major weights [256 rows, K]: box = [64 k][128 rows] (each CTA of the pair stages half of the N rows)
    if (make_tmap(&maps.w[j], s.w, CH_W, (int64_t)kblocks * 64, s.ldw, 64, 128)) return 1;
    if (s.out) {
      MNRF_CHECK(((uintptr_t)s.out % 16) == 0 && s.ldo % 8 == 0 && s.ldo >= CH_W, "mnrf_mlp_chain: layer %d: output alignment", j);
      if (make_tmap(&maps.out[j], s.out, d->m, CH_W, s.ldo, 64, 128)) return 1;
    }
    any_stream |= s.n_stream > 0;
    if (s.n_stream > 0)
      MNRF_CHECK(s.stream_col0 % 64 == 0 && s.stream_col0 + s.n_stream * 64 <= d->stream_cols,
                 "mnrf_mlp_chain: layer %d: streamed columns [%d, %d) outside the stream tensor (%d columns)", j,
                 s.stream_col0, s.stream_col0 + s.n_stream * 64, d->stream_cols);
  }
  if (any_stream) {
    MNRF_CHECK(d->stream && ((uintptr_t)d->stream % 16) == 0 && d->ldstream % 8 == 0 && d->stream_cols % 64 == 0,
               "mnrf_mlp_chain: streamed operand must be 16-byte aligned with a multiple of 64 columns");
    if (make_tmap(&maps.stream, d->stream, d->m, d->stream_cols, d->ldstream, 64, 128)) return 1;
  }
  p.head_w = d->head_w; p.head_b = d->head_b; p.head_out = d->head_out;
  {
    int stores = 0;
    for (int j = 0; j < d->num_layers; ++j) stores += d->layer[j].out ? 1 : 0;
    p.prefetch = (d->mode == MNRF_CHAIN_FWD && stores <= 1) ? 1 : 0;
  }
#ifdef MNRF_TIMING_KNOBS
  p.debug = getenv("MNRF_CHAIN_DEBUG") ? atoi(getenv("MNRF_CHAIN_DEBUG")) : 0;
  p.trace = getenv("MNRF_CHAIN_TRACE") ? reinterpret_cast<long long*>(strtoull(getenv("MNRF_CHAIN_TRACE"), nullptr, 0)) : nullptr;
#endif
  if (d->head_w) MNRF_CHECK(d->mode == MNRF_CHAIN_FWD && d->head_out && ((uintptr_t)d->head_w % 16) == 0,
                            "mnrf_mlp_chain: the head is a forward output (16-byte aligned weights)");
  const int pairs = (int)std::min<int64_t>(p.num_units, sms / 2);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs); cfg.blockDim = dim3(CH_THREADS);
  cfg.dynamicSmemBytes = CH_SMEM; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (d->mode == MNRF_CHAIN_FWD) {
    static bool set0 = false;
    auto kern = mlp_chain_kernel<0>;
    if (!set0) { MNRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM)); set0 = true; }
    MNRF_CUDA(cudaLaunchKernelEx(&cfg, kern, maps, p));
  } else {
    static bool set1 = false;
    auto kern = mlp_chain_kernel<1>;
    if (!set1) { MNRF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM)); set1 = true; }
    MNRF_CUDA(cudaLaunchKernelEx(&cfg, kern, maps, p));
  }
  MNRF_LAUNCH_CHECK();
  return 0;
}
