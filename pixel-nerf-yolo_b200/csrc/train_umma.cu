// tcgen05 GEMMs of the training step (BASELINE config 3; the reference's loss.backward(), train/trainlib/PixelNerfTrainer.py:133-157).
//
// The training path runs the ResnetFC (src/model/resnetfc.py:134-186) layer by layer over ALL rows of the ray batch, with bf16
// operands kept in HBM (the "tape": relu'd block inputs and fc_0 outputs, 1 KiB per row and layer) and fp32 accumulation in TMEM:
//
//   rowgemm_kernel  OUT[M, N] = epilogue( A0[M, K0] W0^T (+ A1[M, K1] W1^T) )        forward layers and input gradients (dgrad)
//        activation-major: one tcgen05.mma.cta_group::2 = 256 rows (128 per CTA) x 256 output features x K 16; A tiles by TMA
//        (SWIZZLE_128B, K-major) from the row-major bf16 activations, W tiles by TMA from a pre-swizzled packed stream (each CTA
//        streams its 128-feature half); accumulators double-buffered in TMEM (2 x 256 columns), so the epilogue of one
//        (row tile, feature half) unit runs under the MMAs of the next.  Epilogue: [* (mask_src > 0)] [+ bias] [+ res_in] ->
//        fp32 and/or bf16 (optionally relu'd) outputs, staged through shared memory so that every global access is coalesced.
//   wgrad_kernel    dW[N, K] += dY[M, N]^T X[M, K]                                     weight gradients
//        both operands MN-major (the contraction runs over ROWS): TMA boxes of 64 features x 64 rows land exactly in the
//        canonical SWIZZLE_128B MN-major layout; one unit = (256 output features, 256 input features, a slab of rows), fp32
//        partial sums reduced into dW with coalesced red.global.add.
// Both are persistent (one CTA pair per SM pair), 5 x 32 KiB stages, one TMA thread per CTA, one MMA thread in the leader.
#include "pnr_common.cuh"
#include "umma.cuh"
#include "train_umma.cuh"
#include "pnr_lab.h"

namespace pnr {
namespace tg {
using namespace umma;

constexpr int kStagesG = 5;
constexpr int kHalf = 16384;                     // one operand tile: 128 rows x 64 k (K-major) or 2 x (64 rows x 64 features) (MN-major)
constexpr int kStageG = 2 * kHalf;
constexpr int kThreadsG = 384;                   // warp 0 TMA, warp 1 MMA, warp 2 TMEM alloc, warps 4..11 epilogue
constexpr int kStagePitch = 36;                  // floats per row of an epilogue staging tile (32 + 4: conflict-free 16-byte rows)
constexpr int kStageTile = 32 * kStagePitch * 4; // 4 608 B per epilogue warp
constexpr int kEpiTile = kStageTile + 32 * 40 * 2;   // rowgemm: + a 32 x 40 bf16 mask tile per epilogue warp
constexpr int kThreadsR = 320;                   // rowgemm: warp 0 TMA, warp 1 TMEM alloc + MMA, warps 2..9 epilogue (quadrant = warp % 4)
struct SmemG {
  static constexpr uint32_t ring = 0;
  static constexpr uint32_t epi = ring + kStagesG * kStageG;
  static constexpr uint32_t colsum = epi + 8 * kEpiTile;           // fp32 partial column sums of this CTA (<= 512 output columns)
  static constexpr uint32_t bias = colsum + 512 * 4;               // bias + bias2 of the (<= 512) output columns, staged once
  static constexpr uint32_t bars = bias + 512 * 4;
  static constexpr uint32_t total = bars + 256;
};
enum { G_FULL = 0, G_EMPTY = G_FULL + kStagesG, G_ACC_FULL = G_EMPTY + kStagesG, G_ACC_FREE = G_ACC_FULL + 2, G_COUNT = G_ACC_FREE + 2 };
static_assert(SmemG::total <= 227 * 1024, "shared memory budget");

// ------------------------------------------------------------------------------------------------------------------------
template <bool kDummy>
__global__ void __launch_bounds__(kThreadsR, 1)
rowgemm_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapW0,
               const __grid_constant__ CUtensorMap mapA1, const __grid_constant__ CUtensorMap mapW1, const RowGemmArgs g) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const uint32_t crank = cluster_ctarank();
  const int pair_id = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  auto bar = [&](int i) -> uint32_t { return sbase + SmemG::bars + 8u * i; };
  auto lbar = [&](int i) -> uint32_t { return mapa_u32(sbase + SmemG::bars + 8u * i, 0); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + SmemG::bars + 8 * G_COUNT);
  if ((sbase & 1023u) != 0) { if (threadIdx.x == 0) printf("pnr: dynamic smem not 1024-aligned\n"); __trap(); }
  if (threadIdx.x == 0) {
    for (int i = 0; i < kStagesG; ++i) { mbar_init(bar(G_FULL + i), 1); mbar_init(bar(G_EMPTY + i), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(bar(G_ACC_FULL + i), 1); mbar_init(bar(G_ACC_FREE + i), 16); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2sm(sbase + SmemG::bars + 8 * G_COUNT, 512);
  float* const csum = reinterpret_cast<float*>(smem + SmemG::colsum);
  float* const sbias = reinterpret_cast<float*>(smem + SmemG::bias);
  if (g.colsum_out) for (int i = threadIdx.x; i < g.n_pad; i += kThreadsR) csum[i] = 0.f;
  // the bias vectors are read from shared memory in the epilogue: 8 broadcast global loads per 32-column chunk cost ~70 us per
  // GEMM (measured: "f32 out + bias" 137 us vs "f32 out" 70 us on 147 456 rows)
  if (g.bias) for (int i = threadIdx.x; i < g.n_pad; i += kThreadsR) sbias[i] = i < g.n_valid ? g.bias[i] + (g.bias2 ? g.bias2[i] : 0.f) : 0.f;
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const long long n_tiles = (g.M + 255) / 256;
  const long long n_units = n_tiles * g.nN;
  const int n_stage_unit = g.nK0 + g.nK1;

  if (warp == 0) {
    if (elect_one()) {
      uint32_t slot = 0, par = 1;
      for (long long u = pair_id; u < n_units; u += n_pairs) {
        const long long t = u / g.nN;
        const int nh = (int)(u - t * g.nN);
        const int row = (int)(t * 256 + crank * 128);
        for (int s = 0; s < n_stage_unit; ++s) {
          const bool second = s >= g.nK0;
          const int kb = second ? s - g.nK0 : s;
          const int nK = second ? g.nK1 : g.nK0;
          mbar_wait_cluster(bar(G_EMPTY + slot), par);
          if (crank == 0) mbar_arrive_expect_tx(bar(G_FULL + slot), 2 * kStageG);
          const uint32_t dst = sbase + SmemG::ring + slot * kStageG;
          tma_load_2d_2sm(dst, second ? (const void*)&mapA1 : (const void*)&mapA0, kb * 64, row, bar(G_FULL + slot));
          tma_load_2d_2sm(dst + kHalf, second ? (const void*)&mapW1 : (const void*)&mapW0, 0, ((nh * nK + kb) * 2 + (int)crank) * 128,
                          bar(G_FULL + slot));
          if (++slot == kStagesG) { slot = 0; par ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (crank == 0 && elect_one()) {
      const uint32_t idesc = instr_desc_bf16_2sm(256);
      uint32_t slot = 0, fpar = 0;
      long long i = 0;
      for (long long u = pair_id; u < n_units; u += n_pairs, ++i) {
        const uint32_t buf = (uint32_t)(i & 1);
        mbar_wait_cluster(bar(G_ACC_FREE + buf), (uint32_t)(((i >> 1) & 1) ^ 1));     // the epilogue has drained this accumulator
        tc_fence_after();
        for (int s = 0; s < n_stage_unit; ++s) {
          mbar_wait(bar(G_FULL + slot), fpar);
          const uint32_t a = sbase + SmemG::ring + slot * kStageG;
          mma_kblock_desc_2sm(tmem_base + buf * 256, smem_desc(a), smem_desc(a + kHalf), idesc, s > 0);
          mma_commit_2sm(bar(G_EMPTY + slot), 3);
          if (++slot == kStagesG) { slot = 0; fpar ^= 1; }
        }
        mma_commit_2sm(bar(G_ACC_FULL + buf), 3);
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue: 8 warps = 4 TMEM lane quadrants x 2 column halves; a unit is walked in 4 chunks of 32 columns.
    // The global reads of a chunk (residual tile, relu-mask tile) are issued ONE CHUNK AHEAD into registers -- across unit
    // boundaries too, before the accumulator is even complete -- so that their latency hides under the previous chunk's work.
    const int q = warp & 3, h = warp >= 6 ? 1 : 0;
    float* S = reinterpret_cast<float*>(smem + SmemG::epi + (warp - 2) * kEpiTile);
    __nv_bfloat16* Sb = reinterpret_cast<__nv_bfloat16*>(S);                       // bf16 view of the fp32 tile (output staging)
    __nv_bfloat16* Sm = reinterpret_cast<__nv_bfloat16*>(smem + SmemG::epi + (warp - 2) * kEpiTile + kStageTile);   // mask tile
    const bool res_vec = g.res_in && (g.ld_res & 3) == 0, mask_vec = g.mask_src && (g.ld_mask & 7) == 0;
    float4 pr[8];
    uint4 pm[4];
    auto chunk_pos = [&](long long u, int c, long long& row0, int& col0) {
      const long long t = u / g.nN;
      const int nh = (int)(u - t * g.nN);
      row0 = t * 256 + crank * 128 + q * 32;
      col0 = nh * 256 + h * 128 + c * 32;
    };
    auto prefetch = [&](long long u, int c) {
      if (u >= n_units) return;
      long long row0; int col0;
      chunk_pos(u, c, row0, col0);
      if (col0 + 32 > g.n_valid) return;                 // partial / empty chunk: the scalar path reads on demand
      if (res_vec) {
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {                 // 4 rows x 128 B per instruction
          const int rr = jj * 4 + (lane >> 3), cc = (lane & 7) * 4;
          pr[jj] = (row0 + rr < g.M) ? __ldcg(reinterpret_cast<const float4*>(g.res_in + (row0 + rr) * g.ld_res + col0 + cc))
                                     : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      if (mask_vec) {
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {                 // 8 rows x 64 B per instruction
          const int rr = jj * 8 + (lane >> 2), cc = (lane & 3) * 8;
          pm[jj] = (row0 + rr < g.M) ? __ldg(reinterpret_cast<const uint4*>(g.mask_src + (row0 + rr) * g.ld_mask + col0 + cc))
                                     : make_uint4(0u, 0u, 0u, 0u);
        }
      }
    };
    long long i = 0;
    prefetch(pair_id, 0);
    for (long long u = pair_id; u < n_units; u += n_pairs, ++i) {
      const uint32_t buf = (uint32_t)(i & 1);
      bool acc_ready = false;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        long long row0; int col0;
        chunk_pos(u, c, row0, col0);
        const bool fast = col0 + 32 <= g.n_valid;        // full chunk: staged, coalesced accesses; else the scalar tail path
        // the prefetched tiles of THIS chunk go to shared memory, then the next chunk's loads are issued
        if (fast && res_vec) {
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) *reinterpret_cast<float4*>(S + (jj * 4 + (lane >> 3)) * kStagePitch + (lane & 7) * 4) = pr[jj];
        }
        if (fast && mask_vec) {
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) *reinterpret_cast<uint4*>(Sm + (jj * 8 + (lane >> 2)) * 40 + (lane & 3) * 8) = pm[jj];
        }
        if (c < 3) prefetch(u, c + 1); else prefetch(u + n_pairs, 0);
        if (!acc_ready) {
          mbar_wait_cluster(bar(G_ACC_FULL + buf), (uint32_t)((i >> 1) & 1));
          tc_fence_after();
          acc_ready = true;
        }
        uint32_t vr[32];
        tmem_ld<32>(tmem_base + ((uint32_t)(q * 32) << 16) + buf * 256 + h * 128 + c * 32, vr);
        if (c == 3) {                                   // last TMEM read of this unit: hand the accumulator back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { if (crank == 0) mbar_arrive(bar(G_ACC_FREE + buf)); else mbar_arrive_cluster_relaxed(lbar(G_ACC_FREE + buf)); }
        }
        __syncwarp();                                    // the staged tiles are complete
        if (col0 >= g.n_valid) continue;
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(vr[j]);
        if (g.mask_src) {
          if (fast && mask_vec) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 m = *reinterpret_cast<const uint4*>(Sm + lane * 40 + j * 8);
              const uint32_t w[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {               // bf16 > 0  <=>  sign bit clear and not zero
                const uint32_t lo = w[e] & 0xFFFFu, hi = w[e] >> 16;
                if (!(lo != 0u && lo < 0x8000u)) v[j * 8 + 2 * e] = 0.f;
                if (!(hi != 0u && hi < 0x8000u)) v[j * 8 + 2 * e + 1] = 0.f;
              }
            }
          } else if (row0 + lane < g.M) {
#pragma unroll
            for (int j = 0; j < 32; ++j)                  // static indices: a dynamically indexed v[] would live in local memory
              if (col0 + j < g.n_valid && !(__bfloat162float(g.mask_src[(row0 + lane) * g.ld_mask + col0 + j]) > 0.f)) v[j] = 0.f;
          }
        }
        if (g.bias) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 b = *reinterpret_cast<const float4*>(sbias + col0 + j);      // same address in every lane: broadcast
            v[j] += b.x; v[j + 1] += b.y; v[j + 2] += b.z; v[j + 3] += b.w;
          }
        }
        if (g.res_in) {
          if (fast && res_vec) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 r = *reinterpret_cast<const float4*>(S + lane * kStagePitch + j * 4);
              v[j * 4] += r.x; v[j * 4 + 1] += r.y; v[j * 4 + 2] += r.z; v[j * 4 + 3] += r.w;
            }
          } else if (row0 + lane < g.M) {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (col0 + j < g.n_valid) v[j] += g.res_in[(row0 + lane) * g.ld_res + col0 + j];
          }
        }
        __syncwarp();                                    // every lane has read its rows: S is free for the outputs
        if (g.colsum_out) {                              // bias gradient: sum of v over this chunk's 32 rows, per column
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const bool ok = row0 + lane < g.M;
            *reinterpret_cast<float4*>(S + lane * kStagePitch + j * 4) =
                ok ? make_float4(v[j * 4], v[j * 4 + 1], v[j * 4 + 2], v[j * 4 + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
          __syncwarp();
          float cs = 0.f;
#pragma unroll 8
          for (int rr = 0; rr < 32; ++rr) cs += S[rr * kStagePitch + lane];
          if (col0 + lane < g.n_valid) atomicAdd(csum + col0 + lane, cs);
          __syncwarp();
        }
        if (g.out_f32) {
          if (fast && (g.ld_f32 & 3) == 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              *reinterpret_cast<float4*>(S + lane * kStagePitch + j * 4) = make_float4(v[j * 4], v[j * 4 + 1], v[j * 4 + 2], v[j * 4 + 3]);
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int rr = j * 4 + (lane >> 3), cc = (lane & 7) * 4;
              if (row0 + rr < g.M)
                *reinterpret_cast<float4*>(g.out_f32 + (row0 + rr) * g.ld_f32 + col0 + cc) = *reinterpret_cast<const float4*>(S + rr * kStagePitch + cc);
            }
            __syncwarp();
          } else if (row0 + lane < g.M) {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (col0 + j < g.n_valid) g.out_f32[(row0 + lane) * g.ld_f32 + col0 + j] = v[j];
          }
        }
        if (g.out_bf16) {
          if (fast && (g.ld_bf16 & 7) == 0) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint32_t p[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                float a = v[j * 8 + 2 * e], b = v[j * 8 + 2 * e + 1];
                if (g.relu_out) { a = fmaxf(a, 0.f); b = fmaxf(b, 0.f); }
                const __nv_bfloat162 pk = __floats2bfloat162_rn(a, b);
                p[e] = *reinterpret_cast<const uint32_t*>(&pk);
              }
              *reinterpret_cast<uint4*>(Sb + lane * 40 + j * 8) = make_uint4(p[0], p[1], p[2], p[3]);
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int rr = j * 8 + (lane >> 2), cc = (lane & 3) * 8;
              if (row0 + rr < g.M)
                *reinterpret_cast<uint4*>(g.out_bf16 + (row0 + rr) * g.ld_bf16 + col0 + cc) = *reinterpret_cast<const uint4*>(Sb + rr * 40 + cc);
            }
            __syncwarp();
          } else if (row0 + lane < g.M) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j < g.n_valid) g.out_bf16[(row0 + lane) * g.ld_bf16 + col0 + j] = __float2bfloat16_rn(g.relu_out ? fmaxf(v[j], 0.f) : v[j]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (g.colsum_out)
    for (int i = threadIdx.x; i < g.n_valid; i += kThreadsR) {
      const float c = csum[i];
      if (c != 0.f) { atomicAdd(g.colsum_out + i, c); if (g.colsum_out2) atomicAdd(g.colsum_out2 + i, c); }
    }
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_2sm(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------------------------------
// dW[n, k] += sum_m dY[m, n] X[m, k].  Unit = (n block of 256, k block of 256, row slab).  Per 64-row step each CTA loads
// dY[64 rows x its 128 n features] and X[64 rows x its 128 k features] as two 64-feature boxes each (MN-major tiles).
__global__ void __launch_bounds__(kThreadsG, 1)
wgrad_kernel(const __grid_constant__ CUtensorMap mapY, const __grid_constant__ CUtensorMap mapX, const WgradArgs g) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const uint32_t crank = cluster_ctarank();
  const int pair_id = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  auto bar = [&](int i) -> uint32_t { return sbase + SmemG::bars + 8u * i; };
  auto lbar = [&](int i) -> uint32_t { return mapa_u32(sbase + SmemG::bars + 8u * i, 0); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + SmemG::bars + 8 * G_COUNT);
  if (threadIdx.x == 0) {
    for (int i = 0; i < kStagesG; ++i) { mbar_init(bar(G_FULL + i), 1); mbar_init(bar(G_EMPTY + i), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(bar(G_ACC_FULL + i), 1); mbar_init(bar(G_ACC_FREE + i), 16); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2sm(sbase + SmemG::bars + 8 * G_COUNT, 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_blocks = g.nNb * g.nKb;                         // output blocks of 256 x 256
  const long long n_units = (long long)n_blocks * g.n_slabs;
  const long long steps_total = (g.M + 63) / 64;
  const long long steps_per_slab = (steps_total + g.n_slabs - 1) / g.n_slabs;

  auto unit = [&](long long u, int& nb, int& kb, long long& s0, long long& s1) {
    const int blk = (int)(u % n_blocks);
    const long long slab = u / n_blocks;
    nb = blk / g.nKb; kb = blk - nb * g.nKb;
    s0 = slab * steps_per_slab;
    s1 = s0 + steps_per_slab < steps_total ? s0 + steps_per_slab : steps_total;
  };

  if (warp == 0) {
    if (elect_one()) {
      uint32_t slot = 0, par = 1;
      for (long long u = pair_id; u < n_units; u += n_pairs) {
        int nb, kb; long long s0, s1;
        unit(u, nb, kb, s0, s1);
        for (long long s = s0; s < s1; ++s) {
          mbar_wait_cluster(bar(G_EMPTY + slot), par);
          if (crank == 0) mbar_arrive_expect_tx(bar(G_FULL + slot), 2 * kStageG);
          const uint32_t dst = sbase + SmemG::ring + slot * kStageG;
          const int row = (int)(s * 64);
          const int yc = nb * 256 + (int)crank * 128, xc = kb * 256 + (int)crank * 128;
          tma_load_2d_2sm(dst, &mapY, yc, row, bar(G_FULL + slot));
          tma_load_2d_2sm(dst + 8192, &mapY, yc + 64, row, bar(G_FULL + slot));
          tma_load_2d_2sm(dst + kHalf, &mapX, xc, row, bar(G_FULL + slot));
          tma_load_2d_2sm(dst + kHalf + 8192, &mapX, xc + 64, row, bar(G_FULL + slot));
          if (++slot == kStagesG) { slot = 0; par ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (crank == 0 && elect_one()) {
      const uint32_t idesc = instr_desc_bf16_2sm(256, 1, 1);
      uint32_t slot = 0, fpar = 0;
      long long i = 0;
      for (long long u = pair_id; u < n_units; u += n_pairs, ++i) {
        int nb, kb; long long s0, s1;
        unit(u, nb, kb, s0, s1);
        const uint32_t buf = (uint32_t)(i & 1);
        mbar_wait_cluster(bar(G_ACC_FREE + buf), (uint32_t)(((i >> 1) & 1) ^ 1));
        tc_fence_after();
        for (long long s = s0; s < s1; ++s) {
          mbar_wait(bar(G_FULL + slot), fpar);
          const uint32_t a = sbase + SmemG::ring + slot * kStageG;
          const uint64_t ad = smem_desc_mn(a), bd = smem_desc_mn(a + kHalf);
          constexpr uint32_t kKStep = 2048 >> 4;             // 16 rows (contraction) = 2 048 B further into both tiles
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            mma_bf16_2sm(tmem_base + buf * 256, ad + (uint64_t)(ks * kKStep), bd + (uint64_t)(ks * kKStep), idesc, (s > s0 || ks > 0) ? 1u : 0u);
          mma_commit_2sm(bar(G_EMPTY + slot), 3);
          if (++slot == kStagesG) { slot = 0; fpar ^= 1; }
        }
        mma_commit_2sm(bar(G_ACC_FULL + buf), 3);
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    const int q = warp & 3, h = (warp - 4) >> 2;
    float* S = reinterpret_cast<float*>(smem + SmemG::epi + (warp - 4) * kStageTile);
    long long i = 0;
    for (long long u = pair_id; u < n_units; u += n_pairs, ++i) {
      int nb, kb; long long s0, s1;
      unit(u, nb, kb, s0, s1);
      const uint32_t buf = (uint32_t)(i & 1);
      mbar_wait_cluster(bar(G_ACC_FULL + buf), (uint32_t)((i >> 1) & 1));
      tc_fence_after();
      const int n0 = nb * 256 + (int)crank * 128 + q * 32;    // output row (feature of dY) of lane 0
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int k0 = kb * 256 + h * 128 + c * 32;           // output columns (features of X)
        uint32_t vr[32];
        tmem_ld<32>(tmem_base + ((uint32_t)(q * 32) << 16) + buf * 256 + h * 128 + c * 32, vr);
        if (c == 3) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { if (crank == 0) mbar_arrive(bar(G_ACC_FREE + buf)); else mbar_arrive_cluster_relaxed(lbar(G_ACC_FREE + buf)); }
        }
        if (s1 <= s0) continue;                                // empty slab: nothing was accumulated (TMEM holds stale data)
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<float4*>(S + lane * kStagePitch + j * 4) =
              make_float4(__uint_as_float(vr[j * 4]), __uint_as_float(vr[j * 4 + 1]), __uint_as_float(vr[j * 4 + 2]), __uint_as_float(vr[j * 4 + 3]));
        __syncwarp();
#pragma unroll 4
        for (int rr = 0; rr < 32; ++rr) {                      // one output row per instruction: 32 consecutive columns
          const int n = n0 + rr, k = k0 + lane;
          if (n < g.N && k < g.K) atomicAdd(g.dW + (size_t)n * g.ldw + k, S[rr * kStagePitch + lane]);
        }
        __syncwarp();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_2sm(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------------------------------
// Packed weight stream of rowgemm: stage (nh, kb) = [CTA0 half: 128 output features x 64 k][CTA1 half], pre-swizzled K-major.
//   transposed = 0: out(o, i) = W[o * ldw + i]   (forward: y = x W^T)      transposed = 1: out(o, i) = W[i * ldw + o]   (dgrad: dx = dy W)
__global__ void pack_rowgemm_kernel(const float* __restrict__ W, int rows, int cols, int ldw, int transposed, int nN, int nK,
                                    uint8_t* __restrict__ dst) {
  const int stage = blockIdx.x >> 1, half = blockIdx.x & 1;
  const int nh = stage / nK, kb = stage - nh * nK;
  uint8_t* out = dst + ((size_t)stage * 2 + half) * kHalf;
  const int n_out = transposed ? cols : rows, n_in = transposed ? rows : cols;
  for (int idx = threadIdx.x; idx < 128 * 64; idx += blockDim.x) {
    const int r = idx >> 6, k = idx & 63;
    const int o = nh * 256 + half * 128 + r, in = kb * 64 + k;
    float v = 0.f;
    if (o < n_out && in < n_in) v = transposed ? W[(size_t)in * ldw + o] : W[(size_t)o * ldw + in];
    *reinterpret_cast<__nv_bfloat16*>(out + swz_offset(r, k)) = __float2bfloat16_rn(v);
  }
}

struct PackJobs { PackJob j[kMaxPackJobs]; int first_block[kMaxPackJobs + 1]; int nK[kMaxPackJobs]; int n; int transposed; };
__global__ void pack_rowgemm_many_kernel(const PackJobs jobs) {
  int ji = 0;
  while (ji + 1 < jobs.n && (int)blockIdx.x >= jobs.first_block[ji + 1]) ++ji;
  const PackJob& J = jobs.j[ji];
  const int local = blockIdx.x - jobs.first_block[ji];
  const int stage = local >> 1, half = local & 1, nK = jobs.nK[ji];
  const int nh = stage / nK, kb = stage - nh * nK;
  uint8_t* out = (uint8_t*)J.dst + ((size_t)stage * 2 + half) * kHalf;
  const int n_out = jobs.transposed ? J.cols : J.rows, n_in = jobs.transposed ? J.rows : J.cols;
  for (int idx = threadIdx.x; idx < 128 * 64; idx += blockDim.x) {
    const int r = idx >> 6, k = idx & 63;
    const int o = nh * 256 + half * 128 + r, in = kb * 64 + k;
    float v = 0.f;
    if (o < n_out && in < n_in) v = jobs.transposed ? J.W[(size_t)in * J.ldw + o] : J.W[(size_t)o * J.ldw + in];
    *reinterpret_cast<__nv_bfloat16*>(out + swz_offset(r, k)) = __float2bfloat16_rn(v);
  }
}

size_t packed_rowgemm_bytes(int n_out, int n_in) {
  const int nN = (n_out + 255) / 256, nK = (n_in + 63) / 64;
  return (size_t)nN * nK * 2 * kHalf;
}

int pack_rowgemm(const float* W, int rows, int cols, int ldw, int transposed, void* dst, cudaStream_t st) {
  const int n_out = transposed ? cols : rows, n_in = transposed ? rows : cols;
  const int nN = (n_out + 255) / 256, nK = (n_in + 63) / 64;
  PNR_REQUIRE(((uintptr_t)dst & 1023) == 0, PNR_ERR_ARG, "pack_rowgemm: destination must be 1024-byte aligned");
  pack_rowgemm_kernel<<<nN * nK * 2, 256, 0, st>>>(W, rows, cols, ldw, transposed, nN, nK, (uint8_t*)dst);
  PNR_CHECK_LAUNCH("tg::pack_rowgemm_kernel");
  return PNR_OK;
}

int pack_rowgemm_many(const PackJob* jobs, int n_jobs, int transposed, cudaStream_t st) {
  PNR_REQUIRE(jobs && n_jobs >= 1 && n_jobs <= kMaxPackJobs, PNR_ERR_ARG, "pack_rowgemm_many: 1..%d jobs", kMaxPackJobs);
  PackJobs pj = {};
  pj.n = n_jobs; pj.transposed = transposed;
  int blocks = 0;
  for (int i = 0; i < n_jobs; ++i) {
    const int n_out = transposed ? jobs[i].cols : jobs[i].rows, n_in = transposed ? jobs[i].rows : jobs[i].cols;
    PNR_REQUIRE(((uintptr_t)jobs[i].dst & 1023) == 0, PNR_ERR_ARG, "pack_rowgemm_many: destination must be 1024-byte aligned");
    pj.j[i] = jobs[i];
    pj.nK[i] = (n_in + 63) / 64;
    pj.first_block[i] = blocks;
    blocks += ((n_out + 255) / 256) * pj.nK[i] * 2;
  }
  pj.first_block[n_jobs] = blocks;
  pack_rowgemm_many_kernel<<<blocks, 256, 0, st>>>(pj);
  PNR_CHECK_LAUNCH("tg::pack_rowgemm_many_kernel");
  return PNR_OK;
}

int rowgemm(const RowGemmSrc& s0, const RowGemmSrc* s1, RowGemmArgs g, cudaStream_t st) {
  if (g.M <= 0) return PNR_OK;
  PNR_REQUIRE(s0.A && s0.Wp && s0.K > 0 && s0.K % 64 == 0, PNR_ERR_ARG, "rowgemm: bad first source (K=%d)", s0.K);
  PNR_REQUIRE(g.n_valid > 0 && g.M < (1LL << 31) - 256, PNR_ERR_ARG, "rowgemm: bad shape");
  g.nN = (g.n_valid + 255) / 256;
  g.n_pad = g.nN * 256;
  PNR_REQUIRE((!g.colsum_out && !g.bias) || g.n_pad <= 512, PNR_ERR_UNSUPPORTED, "rowgemm: bias / fused column sums support up to 512 output columns");
  PNR_REQUIRE(g.bias || !g.bias2, PNR_ERR_ARG, "rowgemm: bias2 without bias");
  g.nK0 = s0.K / 64;
  g.nK1 = s1 ? s1->K / 64 : 0;
  CUtensorMap mA0, mW0, mA1, mW1;
  int rc;
  if ((rc = make_map(&mA0, s0.A, g.M, s0.K, s0.lda, 64, 128, true))) return rc;
  if ((rc = make_map(&mW0, s0.Wp, (long long)g.nN * g.nK0 * 256, 64, 64, 64, 128, false))) return rc;
  if (s1) {
    PNR_REQUIRE(s1->A && s1->Wp && s1->K > 0 && s1->K % 64 == 0, PNR_ERR_ARG, "rowgemm: bad second source");
    if ((rc = make_map(&mA1, s1->A, g.M, s1->K, s1->lda, 64, 128, true))) return rc;
    if ((rc = make_map(&mW1, s1->Wp, (long long)g.nN * g.nK1 * 256, 64, 64, 64, 128, false))) return rc;
  } else { mA1 = mA0; mW1 = mW0; }
  auto kern = rowgemm_kernel<false>;
  int max_pairs;
  if ((rc = pair_capacity(kern, kThreadsR, SmemG::total, &max_pairs))) return rc;
  const long long n_units = ((g.M + 255) / 256) * g.nN;
  const int n_pairs = (int)(n_units < max_pairs ? n_units : max_pairs);
  return launch_pairs(kern, n_pairs, kThreadsR, SmemG::total, st, "tg::rowgemm_kernel", mA0, mW0, mA1, mW1, g);
}

int wgrad(const __nv_bfloat16* dY, long long ldy, const __nv_bfloat16* X, long long ldx, float* dW, int ldw, long long M, int N, int K,
          cudaStream_t st) {
  if (M <= 0) return PNR_OK;
  PNR_REQUIRE(dY && X && dW && N > 0 && K > 0 && M < (1LL << 31) - 64, PNR_ERR_ARG, "wgrad: bad arguments");
  WgradArgs g = {};
  g.dW = dW; g.ldw = ldw; g.M = M; g.N = N; g.K = K;
  g.nNb = (N + 255) / 256; g.nKb = (K + 255) / 256;
  int max_pairs, rc;
  if ((rc = pair_capacity(wgrad_kernel, kThreadsG, SmemG::total, &max_pairs))) return rc;
  const long long steps = (M + 63) / 64;
  long long slabs = (2LL * max_pairs + g.nNb * g.nKb - 1) / (g.nNb * g.nKb);      // ~2 units per CTA pair
  if (slabs > steps) slabs = steps;
  if (slabs < 1) slabs = 1;
  g.n_slabs = (int)slabs;
  // boxes of 64 features x 64 rows; the feature extent is padded to the boxes by the caller's leading dimension (zero-filled OOB)
  CUtensorMap mY, mX;
  // declared widths are rounded up to whole 64-feature boxes where the leading dimension has room (the caller's padding
  // columns are zero); anything beyond the declared width is zero-filled by the TMA unit
  auto width = [](int n, long long ld) -> long long { const long long r = (n + 63) / 64 * 64; return r <= ld ? r : n; };
  if ((rc = make_map(&mY, dY, M, width(N, ldy), ldy, 64, 64, true))) return rc;
  if ((rc = make_map(&mX, X, M, width(K, ldx), ldx, 64, 64, true))) return rc;
  const long long n_units = (long long)g.nNb * g.nKb * g.n_slabs;
  const int n_pairs = (int)(n_units < max_pairs ? n_units : max_pairs);
  return launch_pairs(wgrad_kernel, n_pairs, kThreadsG, SmemG::total, st, "tg::wgrad_kernel", mY, mX, g);
}

}  // namespace tg
}  // namespace pnr

// ---- stand-alone entry points of the two GEMMs (csrc/pnr_lab.h), for tests/test_gpu_train.py and scripts/ ------------------------
namespace pnr {
__global__ void lab_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long rows, int cols, int ld) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * ld) return;
  const long long r = i / ld;
  const int c = (int)(i - r * ld);
  dst[i] = __float2bfloat16_rn(c < cols ? src[r * cols + c] : 0.f);
}
}  // namespace pnr

extern "C" size_t pnr_lab_gemm_workspace_bytes(long long M, int N, int K) {
  const size_t ldk = (size_t)((K + 63) / 64 * 64), ldn = (size_t)((N + 63) / 64 * 64);
  return (size_t)M * ldk * 2 + (size_t)M * ldn * 2 + pnr::tg::packed_rowgemm_bytes(N, K) + 4096;
}

// out[M, N] = epilogue(A[M, K] W[N, K]^T): A, W fp32 device inputs rounded to bf16; optional bias [N], mask_src [M, N] (fp32,
// rounded to bf16), res_in [M, N]; out_f32 and / or out_bf16_as_f32 ([M, N] fp32 copy of the bf16 output) may be null.
extern "C" int pnr_lab_rowgemm(const float* A, const float* W, const float* bias, const float* mask_src, const float* res_in,
                               float* out_f32, void* out_bf16, long long M, int N, int K, int relu_out, void* workspace,
                               size_t workspace_bytes, void* stream) {
  using namespace pnr;
  reset_launch_count();
  PNR_REQUIRE(A && W && workspace && workspace_bytes >= pnr_lab_gemm_workspace_bytes(M, N, K), PNR_ERR_ARG, "pnr_lab_rowgemm: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int ldk = (K + 63) / 64 * 64, ldn = (N + 63) / 64 * 64;
  uint8_t* p = (uint8_t*)(((uintptr_t)workspace + 1023) & ~(uintptr_t)1023);
  __nv_bfloat16* A16 = (__nv_bfloat16*)p; p += ((size_t)M * ldk * 2 + 1023) & ~(size_t)1023;
  __nv_bfloat16* M16 = (__nv_bfloat16*)p; p += ((size_t)M * ldn * 2 + 1023) & ~(size_t)1023;
  uint8_t* Wp = p;
  lab_to_bf16_kernel<<<(unsigned)((M * ldk + 255) / 256), 256, 0, st>>>(A, A16, M, K, ldk);
  if (mask_src) lab_to_bf16_kernel<<<(unsigned)((M * ldn + 255) / 256), 256, 0, st>>>(mask_src, M16, M, N, ldn);
  int rc = tg::pack_rowgemm(W, N, K, K, 0, Wp, st);
  if (rc) return rc;
  tg::RowGemmArgs g = {};
  g.M = M; g.n_valid = N; g.bias = bias; g.mask_src = mask_src ? M16 : nullptr; g.ld_mask = ldn; g.res_in = res_in; g.ld_res = N;
  g.out_f32 = out_f32; g.ld_f32 = N; g.out_bf16 = (__nv_bfloat16*)out_bf16; g.ld_bf16 = N; g.relu_out = relu_out;
  tg::RowGemmSrc s0 = {A16, ldk, ldk, Wp};
  return tg::rowgemm(s0, nullptr, g, st);
}

// dW[N, K] += dY[M, N]^T X[M, K] (fp32 device inputs rounded to bf16)
extern "C" int pnr_lab_wgrad(const float* dY, const float* X, float* dW, long long M, int N, int K, void* workspace,
                             size_t workspace_bytes, void* stream) {
  using namespace pnr;
  reset_launch_count();
  PNR_REQUIRE(dY && X && dW && workspace && workspace_bytes >= pnr_lab_gemm_workspace_bytes(M, N, K), PNR_ERR_ARG, "pnr_lab_wgrad: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int ldk = (K + 63) / 64 * 64, ldn = (N + 63) / 64 * 64;
  uint8_t* p = (uint8_t*)(((uintptr_t)workspace + 1023) & ~(uintptr_t)1023);
  __nv_bfloat16* X16 = (__nv_bfloat16*)p; p += ((size_t)M * ldk * 2 + 1023) & ~(size_t)1023;
  __nv_bfloat16* Y16 = (__nv_bfloat16*)p;
  lab_to_bf16_kernel<<<(unsigned)((M * ldk + 255) / 256), 256, 0, st>>>(X, X16, M, K, ldk);
  lab_to_bf16_kernel<<<(unsigned)((M * ldn + 255) / 256), 256, 0, st>>>(dY, Y16, M, N, ldn);
  return tg::wgrad(Y16, ldn, X16, ldk, dW, K, M, N, K, st);
}
