// F2+F3 fused, CTA-pair version: PixelNeRFNet.forward (src/model/models.py:153-318) on tcgen05.mma.cta_group::2.
//
// Same feature-major formulation as mlp_umma.cu (D^T[feat, col] (+)= W[feat, K] * act^T[K, col]) but one MMA now spans
// the two SMs of a cluster of 2:  M = 256 features (128 per CTA), N = 128 columns (64 per CTA: each CTA gathers and
// owns its own tile of 64 columns = PP points x NS views), K = 16.
//   * per MMA each CTA reads 4 KiB of weights + 2 KiB of activations from its own shared memory for 4x the MACs of
//     the single-CTA N=64 MMA, and N=128 runs the tensor pipe at its full rate (scripts/umma_bench.py);
//   * each CTA streams only ITS half (128 rows) of every 256-row weight slab (tensor-map TMA, cta_group::2, completion
//     on the leader's mbarrier);
//   * TMEM per CTA: x^T = MT feature tiles x 128 columns (cols [0,256)), h^T likewise (cols [256,512)).
// Hidden widths: the network is zero-padded to Hp = 256 * MT features (pnr_mlp_pack): MT = 2 (Hp = 512) for d_hidden in
// (256, 512], MT = 1 (Hp = 256) for d_hidden <= 256.  Padded weight rows / columns and bias entries are zero, so the padded
// features stay exactly 0 through every layer and both pooling modes.
// The price: D rows are FEATURES (CTA c holds features 256*mt + 128*c + lane of all 128 columns) while the B operand
// needs COLUMNS (CTA c holds the rows of its own 64 columns for all K).  So every epilogue unit sends half of its
// bf16 output to the peer CTA's shared memory: values are transposed 8x8 across lanes (shuffles) into 16-byte chunks
// = 8 consecutive K elements of one operand row; the peer's rows leave as st.async (counted on a barrier of the
// destination CTA), the own rows as st.shared.  Epilogue warp (quadrant qd, half hs) handles 32 columns of both tiles.
//
// Warp roles (16 warps per CTA): 0, 12, 13 weight producers (one elected thread each); 1 = MMA issuer in the leader CTA
// (ONE elected thread, lean per-stage loop) / relay in the other CTA; 2, 3, 14, 15 gather; 4..11 epilogue.
//
// Hand-offs (L = leader CTA 0; "mc" = tcgen05.commit.cta_group::2 multicast to both CTAs):
//   W_FULL[s]  @L    : leader producer's expect_tx(32 KiB) + TMA bytes of both CTAs      W_EMPTY[s] @both : mc
//   IN_READY   @L    : gather warps of both CTAs (remote arrive)                         IN_FREE    @both : mc
//   RDY[kc]    @L    : chunk kc (produced by CTA kc % 2) is in place in both CTAs: the producing warps' arrivals, plus
//                      the st.async bytes landing in L (odd kc) or the relay's arrival for bytes that landed in CTA 1 (even kc)
//   LAND[mt]   @CTA1 : st.async bytes of chunk 2*mt from L have landed (+ L's warps' remote arrive.expect_tx)
//   X_FULL[mt], H_FULL[mt] @both : mc, one per feature tile        X_FREE[mt] @L : view-mean epilogue has read x tile mt
//   OUT_FREE   @L    : the output epilogue has read lin_out's result
#include "pnr_common.cuh"
#include "umma.cuh"
#include <cuda.h>

namespace pnr {
using namespace umma;

namespace pair {

constexpr int kNCol = 64;                    // columns per CTA tile
constexpr int kMaxMT = kHidden / 256;        // 256-feature tiles of the widest (512) hidden layer
constexpr int kKBlocksLat = 512 / kBlockK;   // 8 k-blocks: one pass over 512 latent channels
constexpr int kStages = 5;                   // weight ring depth (16 KiB each): the most that fits the shared-memory budget
constexpr int kThreads = 512;
constexpr int kProducers = 3;                // warps 0,12,13
constexpr int kGatherWarps = 4;              // warps 2,3,14,15
constexpr int kEpiWarps = 8;                 // warps 4..11
constexpr int kOperandKB = kNCol * kRowBytes;   // 8 KiB
constexpr int kChunkBytes = 2 * kOperandKB;     // 16 KiB: a 128-feature K-chunk of one CTA's 64 operand rows
constexpr int kTmemCols = 512;
constexpr int kHCol = 256;
constexpr int kMaxStages = 1024;

struct Sched { int n_blocks, CL, n_linz, KBz, proj; };
// proj: the feature maps hold the lin_z pre-projections (d_hidden channels per lin_z layer, PNR_SCENE_PROJECTED): every
// lin_z[b] is an IDENTITY-weight accumulate of its own freshly gathered d_hidden-channel slice (KBz = d_hidden / 64)
// MT = 256-feature tiles of the padded hidden width Hp = 256 * MT.  Stages of one layer: lin_in MT, lin_z MT * KBz,
// fc_0 / fc_1 (2 MT K-chunks x MT tiles x 2 k-blocks) 4 MT^2, lin_out 4 MT.
enum { MAT_LIN_IN = 0, MAT_LINZ = 1, MAT_FC0 = 2, MAT_FC1 = 3, MAT_LIN_OUT = 4 };
struct Seg { int kind, blk, t, len; };
struct StageSrc { int mat, blk, row0, k0; };   // row0 = first row of the 256-row slab

template <int MT> constexpr int kSquareStages = 4 * MT * MT;   // stages of one fc_0 / fc_1 layer
__host__ __device__ inline int z_passes(const Sched& s) { return (s.KBz + 7) / 8; }
template <int MT>
__host__ __device__ inline int sched_total(const Sched& s) {
  return MT + s.n_linz * MT * s.KBz + s.n_blocks * 2 * kSquareStages<MT> + 4 * MT;
}
// stages [0, sched_pre) are the pre-combine part (run once per tile), the rest the post-combine part
template <int MT>
__host__ __device__ inline int sched_pre(const Sched& s) { return MT + s.n_linz * MT * s.KBz + s.CL * 2 * kSquareStages<MT>; }
// per-tile stage order = MMA issue order:
//   lin_in (MT) | lin_z[0] | per block: fc_0 (2 MT^2 (chunk, tile) pairs x kk(2), see fc_pair) | lin_z[b+1] | fc_1 (same) |
//   lin_out (4 MT)
// Order of the (K-chunk kc, feature tile mt) pairs inside a 512x512 layer: (c1,t0)(c0,t0)(c1,t1)(c0,t1)(c3,t0)(c2,t0)(c3,t1)(c2,t1);
// inside a 256x256 layer (MT = 1): (c1,t0)(c0,t0).
// Chunks 0,1 come from the previous layer's tile 0 and arrive first, so both output tiles consume them first; then tile 0 is
// finished (its completion is signalled on its own barrier, so its epilogue overlaps the last two pairs), then tile 1.
// Each pair of chunks starts with its ODD chunk: odd chunks are produced by the non-leader CTA and their remote rows land in
// the leader, on the very barrier the MMA warp waits on, while even chunks need the relay hop from the non-leader -- that hop
// then overlaps the MMAs of the odd chunk.
// first / last: this is the first / last (k-block of the) pair that touches output tile mt.
template <int MT>
__host__ __device__ inline void fc_pair(int t, int& kc, int& mt, int& kk, bool& first, bool& last) {
  const int pr = t >> 1;                       // 0..2 MT^2 - 1
  kk = t & 1;
  if constexpr (MT == 1) {
    kc = pr ^ 1;
    mt = 0;
    first = pr == 0 && kk == 0;
    last = pr == 1 && kk == 1;
  } else {
    kc = ((pr < 4) ? (pr & 1) : (2 + (pr & 1))) ^ 1;
    mt = (pr >> 1) & 1;
    first = (pr == 0 || pr == 2) && kk == 0;
    last = (pr == 5 || pr == 7) && kk == 1;
  }
}
// chunk order of lin_out (one output tile): 1,0,3,2 (MT = 2) or 1,0 (MT = 1), odd chunk first as in fc_pair
__host__ __device__ inline int out_chunk(int t) { return (t >> 1) ^ 1; }
template <int MT>
__host__ __device__ inline Seg walk_stage(const Sched& sc, int s) {
  constexpr int sq = kSquareStages<MT>;
  Seg g;
  const int s1 = MT * sc.KBz;
  if (s < MT) { g.kind = MAT_LIN_IN; g.blk = 0; g.t = s; g.len = MT; return g; }
  s -= MT;
  if (s < s1) { g.kind = MAT_LINZ; g.blk = 0; g.t = s; g.len = s1; return g; }
  s -= s1;
  for (int b = 0; b < sc.n_blocks; ++b) {
    const bool has_z = b + 1 < sc.n_linz;
    if (s < sq) { g.kind = MAT_FC0; g.blk = b; g.t = s; g.len = sq; return g; }
    s -= sq;
    if (has_z) {
      if (s < s1) { g.kind = MAT_LINZ; g.blk = b + 1; g.t = s; g.len = s1; return g; }
      s -= s1;
    }
    if (s < sq) { g.kind = MAT_FC1; g.blk = b; g.t = s; g.len = sq; return g; }
    s -= sq;
  }
  g.kind = MAT_LIN_OUT; g.blk = 0; g.t = s; g.len = 4 * MT;
  return g;
}
struct ZPos { int pass, mt, kbi, kp; };
template <int MT>
__host__ __device__ inline ZPos z_position(int KBz, int t) {
  ZPos z;
  z.pass = t / (MT * 8);
  const int tt = t - z.pass * MT * 8;
  z.kp = KBz - z.pass * 8 < 8 ? KBz - z.pass * 8 : 8;
  z.mt = tt / z.kp;
  z.kbi = tt - z.mt * z.kp;
  return z;
}
template <int MT>
__host__ __device__ inline StageSrc decode_stage(const Sched& sc, int s) {
  const Seg g = walk_stage<MT>(sc, s);
  StageSrc r;
  r.mat = g.kind; r.blk = g.blk;
  switch (g.kind) {
    case MAT_LIN_IN: r.row0 = g.t * 256; r.k0 = 0; break;
    case MAT_LINZ: { const ZPos z = z_position<MT>(sc.KBz, g.t); r.row0 = z.mt * 256; r.k0 = (z.pass * 8 + z.kbi) * 64; } break;
    case MAT_FC0:
    case MAT_FC1: { int kc, mt, kk; bool f, l; fc_pair<MT>(g.t, kc, mt, kk, f, l); r.row0 = mt * 256; r.k0 = kc * 128 + kk * 64; } break;
    default: r.row0 = 0; r.k0 = out_chunk(g.t) * 128 + (g.t & 1) * 64; break;
  }
  return r;
}

// Packed pair stream: stage s = [CTA0 half: 128 rows x 64 k][CTA1 half], both pre-swizzled 16 KiB k-blocks.  Rows and k
// past the layer's true size (the padding to Hp, d_in < 64, d_out < 128) are zero.
template <int MT>
__global__ void pack_stages_kernel(pnr_mlp_params mp, Sched sc, uint8_t* __restrict__ stages) {
  const int s = blockIdx.x >> 1, half = blockIdx.x & 1;
  const StageSrc src = decode_stage<MT>(sc, s);
  const float* W; int rows, cols;
  switch (src.mat) {
    case MAT_LIN_IN: W = mp.lin_in_w; rows = mp.d_hidden; cols = mp.d_in; break;
    case MAT_LINZ: W = mp.linz_w[src.blk]; rows = mp.d_hidden; cols = mp.d_latent; break;
    case MAT_FC0: W = mp.fc0_w[src.blk]; rows = mp.d_hidden; cols = mp.d_hidden; break;
    case MAT_FC1: W = mp.fc1_w[src.blk]; rows = mp.d_hidden; cols = mp.d_hidden; break;
    default: W = mp.lin_out_w; rows = mp.d_out; cols = mp.d_hidden; break;
  }
  const bool identity = sc.proj && src.mat == MAT_LINZ;
  uint8_t* dst = stages + ((size_t)s * 2 + half) * kStageBytes;
  for (int i = threadIdx.x; i < kStageRows * kBlockK; i += blockDim.x) {
    const int r = i / kBlockK, k = i % kBlockK;
    const int gr = src.row0 + half * 128 + r, gk = src.k0 + k;
    const float v = identity ? (gr == gk ? 1.f : 0.f) : ((gr < rows && gk < cols) ? W[(size_t)gr * cols + gk] : 0.f);
    *reinterpret_cast<__nv_bfloat16*>(dst + swz_offset(r, k)) = __float2bfloat16_rn(v);
  }
}

struct Smem {
  static constexpr uint32_t w = 0;
  static constexpr uint32_t ring = w + kStages * kStageBytes;             // 4 K-chunk buffers (16 KiB each): chunk kc -> buffer kc
  static constexpr uint32_t lat = ring + 4 * kChunkBytes;
  static constexpr uint32_t zf = lat + kKBlocksLat * kOperandKB;
  static constexpr uint32_t bars = zf + kOperandKB;
  static constexpr uint32_t prog = bars + 512;
  static constexpr uint32_t total = prog + 8 * kMaxStages;
};
enum {
  B_W_FULL = 0, B_W_EMPTY = B_W_FULL + kStages, B_IN_READY = B_W_EMPTY + kStages, B_IN_FREE,
  // laid out for MT = 2; MT = 1 uses the first of each group (feature tile 0, K-chunks 0 and 1)
  B_X_FULL, B_H_FULL = B_X_FULL + kMaxMT,          // one per feature tile
  B_RDY = B_H_FULL + kMaxMT, B_X_FREE = B_RDY + 2 * kMaxMT,  // one per feature tile: the view-mean epilogue has read x tile mt out of TMEM
  B_LAND = B_X_FREE + kMaxMT,                                    // non-leader CTA only: remote rows of chunk 2*i have landed (st.async bytes)
  B_OUT_FREE = B_LAND + kMaxMT,                 // leader: the output epilogue has read lin_out's result out of the h region
  B_COUNT
};
static_assert(B_COUNT <= 30, "barrier parity bits live in one 32-bit word");
static_assert(Smem::total <= 227 * 1024, "shared memory budget");

struct ProgEntry { uint32_t w0, w1; };
template <int MT>
__device__ inline ProgEntry make_prog(const Sched& sc, int s, uint32_t sbase) {
  const Seg g = walk_stage<MT>(sc, s);
  uint32_t b_addr = 0, dcol = 0, acc = 1, wait_id = 0, c1 = 0, c2 = 0, c3 = 0;
  const bool last = g.t == g.len - 1;
  switch (g.kind) {
    case MAT_LIN_IN:
      b_addr = sbase + Smem::zf; dcol = g.t * 128; acc = 0;
      if (g.t == 0) wait_id = B_IN_READY + 1;
      break;
    case MAT_LINZ: {
      const ZPos z = z_position<MT>(sc.KBz, g.t);
      const bool streaming = z_passes(sc) > 1 || sc.proj;      // the latent tile is refilled for every pass / lin_z layer
      const bool pass_first = z.mt == 0 && z.kbi == 0, pass_last = z.mt == MT - 1 && z.kbi == z.kp - 1;
      b_addr = sbase + Smem::lat + z.kbi * kOperandKB; dcol = z.mt * 128;
      if (streaming && pass_first && !(g.blk == 0 && z.pass == 0)) wait_id = B_IN_READY + 1;
      if (pass_last && (streaming || g.blk == sc.n_linz - 1)) c1 = B_IN_FREE + 1;
      if (last && g.blk == 0) { c2 = B_X_FULL + 1; if (MT > 1) c3 = B_X_FULL + 2; }
    } break;
    case MAT_FC0:
    case MAT_FC1: {
      int kc, mt, kk;
      bool first_of_tile, last_of_tile;
      fc_pair<MT>(g.t, kc, mt, kk, first_of_tile, last_of_tile);
      const bool fc0 = g.kind == MAT_FC0;
      b_addr = sbase + Smem::ring + (kc * 2 + kk) * kOperandKB; dcol = (fc0 ? kHCol : 0) + mt * 128;
      if (fc0) acc = first_of_tile ? 0 : 1;                      // fc_1 always accumulates into x
      if (mt == 0 && kk == 0) wait_id = B_RDY + kc + 1;          // first use of chunk kc (tile 0 precedes tile 1 for every chunk)
      if (last_of_tile) c2 = (fc0 ? B_H_FULL : B_X_FULL) + mt + 1;   // tile mt complete
    } break;
    default: {
      const int kc = out_chunk(g.t), kk = g.t % 2;
      b_addr = sbase + Smem::ring + (kc * 2 + kk) * kOperandKB; dcol = kHCol; acc = g.t > 0;
      if (kk == 0) wait_id = B_RDY + kc + 1;
      if (last) c2 = B_H_FULL + 1;
    } break;
  }
  ProgEntry e;
  e.w0 = ((b_addr >> 4) & 0x3FFFu) | (dcol << 14) | (acc << 23) | (wait_id << 25);
  e.w1 = c1 | (c2 << 5) | (c3 << 14) | ((c1 | c2 | c3) ? (1u << 19) : 0u);   // bit 19: the stage has commits besides W_EMPTY
  return e;
}

// Column i (< 16) of gather warp gw: at any time the four warps work on four adjacent columns = adjacent points of one
// source view, whose 2x2 tap blocks overlap (their requests merge in L1).
__device__ __forceinline__ int gather_col(int gw, int i) { return gw + kGatherWarps * i; }

// Store an epilogue warp's [32 features x NC columns] block as operand rows (row = column, 16-byte chunk = 8 consecutive
// features).  vals[c] = fp32 bits of this lane's feature at column c; bias/ReLU/bf16 rounding happen here.  Per 16
// columns: pack column pairs to bf16x2, one 8x8 transpose of 32-bit registers across the 8 lanes of a lane group, then
// split low/high halves -> every lane owns two complete 16-byte chunks (columns c0+2i and c0+2i+1).
// `base` = address of the K-chunk (two k-blocks) in the destination CTA; kq = qd*32 = this warp's feature offset in it.
// relu + round-to-nearest bf16 of two floats in one instruction: low half = lo, high half = hi
__device__ __forceinline__ uint32_t pack_relu_bf16x2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}

template <int NC, bool REMOTE, bool ADD_BIAS>
__device__ __forceinline__ void store_transposed(uint32_t base, const uint32_t* vals, float bias, int lane, int kq, int row0,
                                                 uint32_t async_bar = 0) {   // REMOTE: the rows go out as st.async counted on that barrier
  const int g = lane >> 3, i = lane & 7;
  const int k = kq + 8 * g;                                     // first of the 8 features this lane stores, within the chunk
  const uint32_t kb_off = (uint32_t)(k >> 6) * kOperandKB;
#pragma unroll
  for (int c0 = 0; c0 < NC; c0 += 16) {
    // pair column j with column j+8: after the transpose lane i owns rows c0+i and c0+8+i, whose (row & 7) differ
    // across the 8 lanes of a group -> the swizzled 16-byte stores of a quarter warp hit 8 different bank groups
    uint32_t p[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float x = __uint_as_float(vals[c0 + j]), y = __uint_as_float(vals[c0 + 8 + j]);
      if (ADD_BIAS) { x += bias; y += bias; }
      p[j] = pack_relu_bf16x2(x, y);
    }
    transpose8x8(p, lane);                                      // p[f] = (feature 8g+f at column c0+i, at column c0+8+i)
    const uint32_t e0 = __byte_perm(p[0], p[1], 0x5410), e1 = __byte_perm(p[2], p[3], 0x5410);
    const uint32_t e2 = __byte_perm(p[4], p[5], 0x5410), e3 = __byte_perm(p[6], p[7], 0x5410);
    const uint32_t o0 = __byte_perm(p[0], p[1], 0x7632), o1 = __byte_perm(p[2], p[3], 0x7632);
    const uint32_t o2 = __byte_perm(p[4], p[5], 0x7632), o3 = __byte_perm(p[6], p[7], 0x7632);
    const uint32_t addr_e = base + kb_off + swz_offset(row0 + c0 + i, k & 63);
    const uint32_t addr_o = base + kb_off + swz_offset(row0 + c0 + 8 + i, k & 63);
    if (REMOTE) { st_async_v4(addr_e, e0, e1, e2, e3, async_bar); st_async_v4(addr_o, o0, o1, o2, o3, async_bar); }
    else { st_shared_v4(addr_e, e0, e1, e2, e3); st_shared_v4(addr_o, o0, o1, o2, o3); }
  }
}

// Work unit of a CTA pair = a "super group": G = 64 / PP consecutive tile pairs.
//   pre-combine  (G times): tile of PP points x NS views per CTA: gather, lin_in, lin_z, blocks [0, CL), view pooling
//                (mean, or elementwise max when VMAX) -> x-bar (fp32, bias folded in) into this pair's private scratch
//                (L2-resident, 256 KiB per pair);
//   post-combine (once)   : the G x PP (<= 64) points each CTA gathered form ONE 64-column tile: x-bar -> TMEM,
//                blocks [CL, n_blocks), lin_out, sigmoid/relu.
// Without pooling (CL == n_blocks, NS == 1 only: G = 1) the pre-combine part runs every block and the post-combine part is
// lin_out alone on relu(x-bar).
// So every MMA of the kernel runs at N = 128, and the post-combine layers need 1/G of the weight passes and
// epilogue hand-offs per point that a per-tile post phase would.
//
// Epilogue exchange: the half of every epilogue unit that belongs to the peer CTA goes out as st.async (16 bytes per store,
// counted on an mbarrier of the DESTINATION CTA), so the epilogue warps do not sit in fence.proxy.async.shared::cluster
// waiting for their remote rows to be performed (14.5 % of all warp-stall samples of a synchronous exchange).  Rows landing
// in the leader are counted directly on the chunk barrier the MMA warp waits on; rows landing in the non-leader are counted
// on its B_LAND barrier, and its otherwise idle warp 1 relays that to the leader.
// VMAX: combine_type "max".  MT: 256-feature tiles of the padded hidden width (1 or 2, see Sched).
template <int NS, bool VMAX, int MT>
__global__ void __launch_bounds__(kThreads, 1)
field_pair_kernel(const pnr_scene sc, const pnr_points q, const __grid_constant__ CUtensorMap wmap,
                  const float* __restrict__ bias_x, const float* __restrict__ bias_h,
                  const float* __restrict__ bias_out, float* __restrict__ out, float* __restrict__ xbar_all,
                  const Sched sch, const int num_freqs, const float freq_factor, const int tiles_per_obj,
                  const int n_tiles, const int d_out, const int raw_out) {
  const uint32_t crank = cluster_ctarank();            // 0 = leader (issues every MMA of the pair)
  const int pair_id = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  constexpr int PP = kNCol / NS;                       // points per pre-combine tile
  constexpr int G = kNCol / PP;                        // pre-combine tile pairs per super group
  constexpr int NLIVE = G * PP;                        // live columns of a post-combine tile (<= 64)
  const bool pooled = NS > 1 || sch.CL < sch.n_blocks;   // false: no block after the combine step, lin_out follows it
  const int n_sg = ((n_tiles + 1) / 2 + G - 1) / G;
  // [tile slot 2][column 64][feature 512]: laid out for the widest hidden layer whatever MT is (features >= Hp unused)
  float* const xbar = xbar_all + (size_t)pair_id * (2 * kNCol * kHidden);
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  volatile uint32_t* tmem_base_slot = reinterpret_cast<volatile uint32_t*>(smem + Smem::bars + 8 * B_COUNT);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  auto bar = [&](int i) -> uint32_t { return sbase + Smem::bars + 8u * i; };
  auto lbar = [&](int i) -> uint32_t { return mapa_u32(sbase + Smem::bars + 8u * i, 0); };   // the leader's copy
  if ((sbase & 1023u) != 0) { if (threadIdx.x == 0) printf("pnr: dynamic smem not 1024-aligned\n"); __trap(); }

  if (threadIdx.x == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(bar(B_W_FULL + i), 1); mbar_init(bar(B_W_EMPTY + i), 1); }
    mbar_init(bar(B_IN_READY), 2 * kGatherWarps);
    mbar_init(bar(B_IN_FREE), 1);
    for (int i = 0; i < MT; ++i) { mbar_init(bar(B_X_FULL + i), 1); mbar_init(bar(B_H_FULL + i), 1); }
    // chunk kc is produced by CTA kc % 2; even chunks need one more arrival: the relay of the non-leader CTA
    for (int i = 0; i < 2 * MT; ++i) mbar_init(bar(B_RDY + i), kEpiWarps + ((i & 1) == 0 ? 1 : 0));
    for (int i = 0; i < MT; ++i) mbar_init(bar(B_LAND + i), kEpiWarps);
    mbar_init(bar(B_OUT_FREE), 2);
    for (int i = 0; i < MT; ++i) mbar_init(bar(B_X_FREE + i), 2 * kEpiWarps);
    fence_barrier_init();
  }
  const int n_stages = sched_total<MT>(sch);
  const int s_pre = sched_pre<MT>(sch);                 // stages [0, s_pre) run per pre-combine tile, [s_pre, n_stages) per super group
  const int n_flat = G * s_pre + (n_stages - s_pre);   // weight stages one super group consumes
  for (int i = threadIdx.x; i < n_stages; i += kThreads) {
    const ProgEntry pe = make_prog<MT>(sch, i, sbase);
    reinterpret_cast<ProgEntry*>(smem + Smem::prog)[i] = pe;
    if (i == n_stages - 1) reinterpret_cast<ProgEntry*>(smem + Smem::prog)[n_stages] = pe;   // pad: the issuer prefetches entry st + 1
  }
  if (warp == 1) tmem_alloc_2sm(sbase + Smem::bars + 8 * B_COUNT, kTmemCols);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                    // both CTAs' barriers initialised and TMEM allocated before any remote signal
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_base_slot, 0);
  const uint32_t idesc = instr_desc_bf16_2sm(2 * kNCol);

  if (warp == 0 || warp == 12 || warp == 13) {
    // ===================== weight producers: warp p streams global stages g = p (mod kProducers); each CTA loads its
    // 128-row half of every 256-row slab, both halves complete on the LEADER's W_FULL barrier
    const int pid = warp == 0 ? 0 : warp - 11;
    if (elect_one()) {                                  // one thread per producer warp, tight loop (no per-stage elect/syncwarp)
      uint32_t slot = pid, par = 1;
      int carry = pid;                                  // first stage of this producer inside the current super group
      for (int sg = pair_id; sg < n_sg; sg += n_pairs) {
        int fi = carry;
        int st = fi < G * s_pre ? fi % s_pre : fi - (G - 1) * s_pre;   // G passes over the pre stages, one over the post stages
        for (; fi < n_flat; fi += kProducers) {
          mbar_wait_cluster(bar(B_W_EMPTY + slot), par);
          if (crank == 0) mbar_arrive_expect_tx(bar(B_W_FULL + slot), 2 * kStageBytes);
          tma_load_2d_2sm(sbase + Smem::w + slot * kStageBytes, &wmap, 0, (st * 2 + (int)crank) * kStageRows, bar(B_W_FULL + slot));
          slot += kProducers;
          if (slot >= kStages) { slot -= kStages; par ^= 1; }
          // next stage id without a division: inside the pre passes the id wraps at s_pre, after them it just continues
          const int nf = fi + kProducers;
          if (nf < G * s_pre) { st += kProducers; if (st >= s_pre) st -= s_pre; }
          else st = nf - (G - 1) * s_pre;
        }
        carry = fi - n_flat;                            // the ring position continues across super groups
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (crank == 0) {
      // ===================== MMA issuer (leader CTA only): ONE thread walks the per-tile stage program ==========
      // Measured (MMA N = 128 / 64 / 32 give the same step time): the tensor pipe is not what this kernel waits for, the
      // issuing warp's own instruction stream is.  So the whole role is a single elected thread in a tight per-stage loop --
      // no ballot probe of the ring, no per-batch elect / __syncwarp: it polls the barriers itself (try_wait), issues the four
      // MMAs of the stage (~45 cycles) and its commits (~70 cycles), and prefetches the next program entry meanwhile.
      if (elect_one()) {
        uint32_t slot = 0, wpar = 0, ph = 0;
        uint32_t full_bar = bar(B_W_FULL), empty_bar = bar(B_W_EMPTY);      // running addresses of the current ring slot's barriers
        const uint64_t wdesc0 = smem_desc(sbase + Smem::w);
        uint64_t a_desc = wdesc0;                                           // ... and of its A descriptor
        const uint64_t bdesc_hi = smem_desc(0);
        constexpr uint64_t kStageStep = kStageBytes >> 4;
        const uint2* prog = reinterpret_cast<const uint2*>(smem + Smem::prog);
        for (int sg = pair_id; sg < n_sg; sg += n_pairs) {
          for (int seg = 0; seg <= G; ++seg) {              // G pre-combine passes, then the post-combine pass
            const bool after_mean = seg > 0 && seg < G;
            if (after_mean) {
              // the view-mean epilogue of the previous tile must have read x tile 0 out of TMEM before lin_in (stage 0) overwrites
              // it; tile 1 (MT = 2) is first written by stage 1 (see below)
              mbar_wait_cluster(bar(B_X_FREE), (ph >> B_X_FREE) & 1u);
              ph ^= (1u << B_X_FREE);
              tc_fence_after();
            }
            const int st_beg = seg < G ? 0 : s_pre, st_end = seg < G ? s_pre : n_stages;
            if (seg == 0 && sg != pair_id) {
              // The previous super group's output epilogue (two warps of this CTA) reads lin_out's result from h tile 0; the first
              // fc_0 of this super group only waits for a chunk signalled by the OTHER CTA's warps (odd-chunk-first order).  In
              // practice that is thousands of cycles later; this wait (a few hundred cycles after lin_out at most) makes it explicit.
              mbar_wait(bar(B_OUT_FREE), (ph >> B_OUT_FREE) & 1u);
              ph ^= (1u << B_OUT_FREE);
            }
            uint2 cur = prog[st_beg];
            // one stage: wait for what the entry names and for the weight slot, issue the four MMAs and the commits
            auto issue_stage = [&](int st) {
              const uint2 nxt = prog[st + 1];               // in flight while this stage is issued (the program is padded by one entry)
              const uint32_t wait_id = cur.x >> 25;
              if (wait_id) {
                const uint32_t id = wait_id - 1;
                mbar_wait_cluster(bar(id), (ph >> id) & 1u);
                ph ^= (1u << id);
                fence_proxy_async();                        // rows that landed in this CTA by st.async
                tc_fence_after();                           // the other warps' tcgen05.ld / st of this TMEM precede the MMAs below
              }
              mbar_wait(full_bar, wpar);                    // completed by the TMA engine: no tcgen05 fence needed
              const uint64_t b_desc = bdesc_hi | (uint64_t)(cur.x & 0x3FFFu);
              const uint32_t d_col = (cur.x >> 14) & 0x1FFu;
              mma_kblock_desc_2sm(tmem_base + d_col, a_desc, b_desc, idesc, (cur.x >> 23) & 1u);
              mma_commit_2sm(empty_bar, 3);
              if (cur.y & (1u << 19)) {
                const uint32_t c1 = cur.y & 31u, c2 = (cur.y >> 5) & 31u, c3 = (cur.y >> 14) & 31u;
                if (c1) mma_commit_2sm(bar(c1 - 1), 3);
                if (c2) mma_commit_2sm(bar(c2 - 1), 3);
                if (c3) mma_commit_2sm(bar(c3 - 1), 3);
              }
              if (++slot == kStages) { slot = 0; wpar ^= 1; full_bar = bar(B_W_FULL); empty_bar = bar(B_W_EMPTY); a_desc = wdesc0; }
              else { full_bar += 8; empty_bar += 8; a_desc += kStageStep; }
              cur = nxt;
            };
            int st = st_beg;
            if (MT > 1 && after_mean) {                     // lin_in's second stage is the first write into x tile 1
              issue_stage(st++);
              mbar_wait_cluster(bar(B_X_FREE + 1), (ph >> (B_X_FREE + 1)) & 1u);
              ph ^= (1u << (B_X_FREE + 1));
              tc_fence_after();
            }
            for (; st < st_end; ++st) issue_stage(st);
          }
        }
      }
      __syncwarp();
    } else {
      // ===================== relay (non-leader CTA): remote rows of the even chunks have landed here -> tell the leader
      const int n_pub = G * 2 * sch.CL + 2 * (sch.n_blocks - sch.CL) + 1;     // publishes of each chunk per super group
      uint32_t par = 0;
      for (int sg = pair_id; sg < n_sg; sg += n_pairs) {
        for (int i = 0; i < n_pub; ++i) {
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            mbar_wait_cluster(bar(B_LAND + mt), par);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster_relaxed(lbar(B_RDY + 2 * mt));
          }
          par ^= 1;
        }
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ===================== epilogue warps ===================================================================
    // 8 warps = 4 TMEM lane quadrants (qd) x 2.  Unit = this CTA's 128 features of feature tile mt x all 128 columns of
    // the pair = K-chunk kc = 2*mt + crank, written to chunk buffer kc of BOTH CTAs (rows = that CTA's own columns).
    //  * regular epilogues: warp (qd, part) converts columns [part*NC/2, (part+1)*NC/2) of BOTH tiles, the peer's first
    //    (remote st.async stores are in flight while the local half is computed), one publish per unit;
    //  * view-mean epilogue: warp (qd, hs) needs all 64 columns of tile hs (the three views of a point) in one thread.
    const int qd = warp & 3;                       // TMEM lane quadrant (warp % 4)
    const int hs = (warp - 4) >> 2;                // second index: column part, or tile in the mean / output epilogues
    const int fl = qd * 32 + lane;                 // feature row inside this CTA's 128-row half
    const uint32_t tlane = tmem_base + ((uint32_t)(qd * 32) << 16);
    uint32_t ph = 0;
    auto wait = [&](int id) { mbar_wait_cluster(bar(id), (ph >> id) & 1u); ph ^= (1u << id); tc_fence_after(); };
    const uint32_t peer = crank ^ 1u;
    constexpr uint32_t kRemoteBytes = (kNCol / 2) * 32 * 2;        // remote half of one warp's unit: 32 columns x 32 features bf16
    // barrier (in the peer CTA) that counts this CTA's st.async rows of chunk kc = 2*mt + crank
    auto land_bar = [&](int kc) -> uint32_t { return crank == 0 ? mapa_u32(bar(B_LAND + (kc >> 1)), 1) : lbar(B_RDY + kc); };
    auto publish = [&](int kc) {                   // operand rows of chunk kc written -> tell the leader's MMA warp
      fence_proxy_async();                         // local rows only; the remote rows are counted where they land
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (crank == 0) { mbar_arrive(bar(B_RDY + kc)); mbar_arrive_expect_tx_cluster(land_bar(kc), kRemoteBytes); }
        else mbar_arrive_expect_tx_cluster(land_bar(kc), kRemoteBytes);        // = the leader's chunk barrier
      }
    };
    // both halves of a unit: columns [hs*32, hs*32+32) of tile `peer` (remote rows) then of tile `crank` (local rows)
    auto convert_unit = [&](uint32_t tcol, int kc, float bias) {
      const uint32_t loc = sbase + Smem::ring + kc * kChunkBytes;
      const uint32_t rem = mapa_u32(loc, peer);
      uint32_t v[kNCol / 2], u[kNCol / 2];
      tmem_ld_nowait<kNCol / 2>(tlane + tcol + peer * kNCol + hs * (kNCol / 2), v);     // both halves in flight at once
      tmem_ld_nowait<kNCol / 2>(tlane + tcol + crank * kNCol + hs * (kNCol / 2), u);
      tmem_ld_wait();
      store_transposed<kNCol / 2, true, true>(rem, v, bias, lane, qd * 32, hs * (kNCol / 2), land_bar(kc));
      store_transposed<kNCol / 2, false, true>(loc, u, bias, lane, qd * 32, hs * (kNCol / 2));
    };
    auto x_epilogue = [&](int e) {                 // relu(x + cumulative bias) -> bf16 K-chunks
      for (int mt = 0; mt < MT; ++mt) {
        // the bias is fetched BEFORE the wait: a global load issued after it sits on the hand-off's critical path
        const float bias = __ldg(bias_x + e * kHidden + mt * 256 + crank * 128 + fl);
        wait(B_X_FULL + mt);
        const int kc = 2 * mt + (int)crank;
        convert_unit(mt * 128, kc, bias);
        publish(kc);
      }
    };
    auto h_epilogue = [&](int b) {                 // relu(fc_0 out + b) -> bf16 K-chunks for fc_1
      for (int mt = 0; mt < MT; ++mt) {
        const float bias = __ldg(bias_h + b * kHidden + mt * 256 + crank * 128 + fl);
        wait(B_H_FULL + mt);
        const int kc = 2 * mt + (int)crank;
        convert_unit(kHCol + mt * 128, kc, bias);
        publish(kc);
      }
    };
    for (int sg = pair_id; sg < n_sg; sg += n_pairs) {
      // ================= pre-combine: G tile pairs; warp (qd, hs) takes the view mean of tile hs of each pair
      for (int g = 0; g < G; ++g) {
        const int tile = (sg * G + g) * 2 + hs;
        const bool live = tile < n_tiles;
        const int obj = tile / tiles_per_obj;
        const int p0 = (tile - obj * tiles_per_obj) * PP;
        for (int e = 0; e < sch.CL; ++e) { x_epilogue(e); h_epilogue(e); }
        float bias_mean[MT];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) bias_mean[mt] = __ldg(bias_x + sch.CL * kHidden + mt * 256 + (int)crank * 128 + fl);
        for (int mt = 0; mt < MT; ++mt) wait(B_X_FULL + mt);
        // view pooling (combine_interleaved) + cumulative bias -> x-bar, column g*PP + p of slot hs.  max(x_v + b) = max(x_v) + b
        // exactly: rounding is monotonic
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          const int f = mt * 256 + (int)crank * 128 + fl;
          const float bias = bias_mean[mt];
          uint32_t v[kNCol];
          tmem_ld<kNCol>(tlane + mt * 128 + hs * kNCol, v);
          if (g + 1 < G) {                          // x tile mt is in registers -> the next tile's lin_in / lin_z may overwrite it
            tc_fence_before();
            __syncwarp();
            if (lane == 0) { if (crank == 0) mbar_arrive(bar(B_X_FREE + mt)); else mbar_arrive_cluster_relaxed(lbar(B_X_FREE + mt)); }
          }
          float* dst = xbar + ((size_t)hs * kNCol + g * PP) * kHidden + f;
#pragma unroll
          for (int p = 0; p < PP; ++p) {
            float pooled_x;
            if constexpr (VMAX) {
              pooled_x = __uint_as_float(v[p]);
#pragma unroll
              for (int vw = 1; vw < NS; ++vw) pooled_x = fmaxf(pooled_x, __uint_as_float(v[vw * PP + p]));
            } else {
              float acc = 0.f;
#pragma unroll
              for (int vw = 0; vw < NS; ++vw) acc += __uint_as_float(v[vw * PP + p]);
              pooled_x = __fdiv_rn(acc, (float)NS);
            }
            const bool ok = live && p0 + p < q.P;
            __stcg(dst + (size_t)p * kHidden, ok ? pooled_x + bias : 0.f);
          }
        }
      }
      // ================= post-combine: one tile of 64 columns per CTA (column j = g*PP + p of the tiles above)
      // warp (qd, 1-hs) wrote the x-bar values this warp loads and read the TMEM columns it overwrites
      tc_fence_before();
      asm volatile("bar.sync %0, 64;" ::"r"(1 + qd) : "memory");
      tc_fence_after();
      for (int mt = 0; mt < MT; ++mt) {
        const int kc = 2 * mt + (int)crank;
        const int f = mt * 256 + (int)crank * 128 + fl;
        const uint32_t loc = sbase + Smem::ring + kc * kChunkBytes;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const uint32_t t = half == 0 ? peer : crank;            // peer's columns first (remote rows)
          const float* src = xbar + ((size_t)t * kNCol + hs * (kNCol / 2)) * kHidden + f;
          uint32_t v[kNCol / 2];
#pragma unroll
          for (int c = 0; c < kNCol / 2; ++c)
            v[c] = (hs * (kNCol / 2) + c < NLIVE) ? __float_as_uint(__ldcg(src + (size_t)c * kHidden)) : 0u;
          tmem_st<kNCol / 2>(tlane + mt * 128 + t * kNCol + hs * (kNCol / 2), v);
          if (half == 0) store_transposed<kNCol / 2, true, false>(mapa_u32(loc, peer), v, 0.f, lane, qd * 32, hs * (kNCol / 2), land_bar(kc));
          else store_transposed<kNCol / 2, false, false>(loc, v, 0.f, lane, qd * 32, hs * (kNCol / 2));
        }
        publish(kc);
      }
      if (pooled) h_epilogue(sch.CL);
      for (int e = sch.CL + 1; e <= sch.n_blocks; ++e) {
        x_epilogue(e);
        if (e < sch.n_blocks) h_epilogue(e);
      }
      // ---- output: lin_out rows are features 0..d_out-1 -> leader CTA, TMEM lanes 0..d_out-1 of h tile 0
      wait(B_H_FULL);                              // lin_out signals tile 0 only
      if (crank == 0 && qd == 0) {
        uint32_t r[kNCol];
        tmem_ld<kNCol>(tlane + kHCol + hs * kNCol, r);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(B_OUT_FREE));
        if (lane < d_out) {
          const float bias = bias_out[lane];
#pragma unroll
          for (int g = 0; g < G; ++g) {
            const int tile = (sg * G + g) * 2 + hs;
            const int obj = tile / tiles_per_obj;
            const int p0 = (tile - obj * tiles_per_obj) * PP;
            if (tile < n_tiles) {
#pragma unroll
              for (int p = 0; p < PP; ++p) {
                if (p0 + p < q.P) {
                  float val = __uint_as_float(r[g * PP + p]) + bias;
                  if (!raw_out) val = lane < 3 ? 1.0f / (1.0f + expf(-val)) : fmaxf(val, 0.f);   // models.py:312-317
                  out[((size_t)obj * q.P + p0 + p) * d_out + lane] = val;
                }
              }
            }
          }
        }
      }
      tc_fence_before();
    }
  } else if (warp == 2 || warp == 3 || warp == 14 || warp == 15) {
    // ===================== gather warps: this CTA's 64 columns -> its own z-feature / latent operand rows =======
    const int gw = warp < 4 ? warp - 2 : warp - 12;
    uint32_t par_free = 1;
    const int n_pass = z_passes(sch);
    const int fills = (n_pass > 1 || sch.proj) ? sch.n_linz * n_pass : 1;
    for (int it = 0;; ++it) {                        // tile pairs sg*G + g of super groups sg = pair_id, pair_id + n_pairs, ...
      const int sg = pair_id + (it / G) * n_pairs;
      if (sg >= n_sg) break;
      const int tile = (sg * G + it % G) * 2 + (int)crank;
      const int obj = tile / tiles_per_obj;
      const int p0 = (tile - obj * tiles_per_obj) * PP;
      // ---- pre-pass, before the operand buffers are free (touches no shared memory): this warp owns columns
      // c_i = gw + 4 i (i < 16); lane i (and i + 16) projects column c_i, then every lane computes its two
      // z-feature elements of all 16 columns
      Taps tp;
      long long vbase = -1;                          // element offset of this lane's column's source view, -1 = dead column
      Projection pr;
      {
        const int c = gather_col(gw, lane & 15);
        const int v = c / PP, p = c - v * PP;
        const bool valid = (tile < n_tiles) && (v < NS) && (p0 + p < q.P);
        pr.xr = pr.yr = pr.zr = pr.dx = pr.dy = pr.dz = pr.ix = pr.iy = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) { tp.off[k] = -1; tp.w[k] = 0.f; }
        if (valid) {
          float px, py, pz, vx, vy, vz;
          const int view = obj * NS + v;
          fetch_point(q, (long long)obj * q.P + p0 + p, px, py, pz, vx, vy, vz);
          pr = project_point(sc, view, px, py, pz, vx, vy, vz);
          tp = make_taps(pr.ix, pr.iy, sc.Hl, sc.Wl, sc.C);
          vbase = (long long)view * sc.Hl * sc.Wl * sc.C;
        }
      }
      auto zfeat_col = [&](int i) {                  // z-feature row of column c_i: every lane computes two elements
        Projection pi;
        pi.xr = __shfl_sync(0xffffffffu, pr.xr, i); pi.yr = __shfl_sync(0xffffffffu, pr.yr, i);
        pi.zr = __shfl_sync(0xffffffffu, pr.zr, i); pi.dx = __shfl_sync(0xffffffffu, pr.dx, i);
        pi.dy = __shfl_sync(0xffffffffu, pr.dy, i); pi.dz = __shfl_sync(0xffffffffu, pr.dz, i);
        pi.ix = pi.iy = 0.f;
        const bool vi = __shfl_sync(0xffffffffu, vbase, i) >= 0;
        const int j0 = lane * 2, d_in = 6 * num_freqs + 6;
        float a = 0.f, b = 0.f;
        if (vi) {
          if (j0 < d_in) a = zfeat_value_fast(pi, j0, num_freqs, freq_factor);
          if (j0 + 1 < d_in) b = zfeat_value_fast(pi, j0 + 1, num_freqs, freq_factor);
        }
        *reinterpret_cast<__nv_bfloat162*>(smem + Smem::zf + swz_offset(gather_col(gw, i), j0)) = __floats2bfloat162_rn(a, b);
      };
      for (int fill = 0; fill < fills; ++fill) {
        const int pass = fill % n_pass;
        const int kp = sch.KBz - pass * 8 < 8 ? sch.KBz - pass * 8 : 8;
        // projected maps: lin_z[b]'s own d_hidden-channel slice (one pass, KBz = d_hidden / 64)
        const int ch0 = sch.proj ? (fill / n_pass) * (sch.KBz * kBlockK) : pass * 512;
        // ---- 4 taps x 1 KiB per column, two columns in flight per warp (the loads are L2 hits with ~1-2 k cycles of
        // latency under the weight stream's load; one column at a time left the tensor cores waiting for the gather)
        const bool act = (lane >> 2) < kp;
        const __nv_bfloat16* fl0 = (const __nv_bfloat16*)sc.feat + ch0 + lane * 16;
        auto load_col = [&](int i, uint4 (&r)[8], float (&w)[4]) {
          const long long vb = __shfl_sync(0xffffffffu, vbase, i);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int off = __shfl_sync(0xffffffffu, tp.off[k], i);
            w[k] = __shfl_sync(0xffffffffu, tp.w[k], i);
            if (off >= 0 && act) {
              const uint4* src = reinterpret_cast<const uint4*>(fl0 + vb + off);
              r[2 * k] = __ldg(src); r[2 * k + 1] = __ldg(src + 1);
            } else {
              r[2 * k] = make_uint4(0u, 0u, 0u, 0u); r[2 * k + 1] = make_uint4(0u, 0u, 0u, 0u);
            }
          }
        };
        auto blend_col = [&](int i, const uint4 (&r)[8], const float (&w)[4]) {
          if (!act) return;
          float acc[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[j] = 0.f;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const __nv_bfloat162* h0 = reinterpret_cast<const __nv_bfloat162*>(&r[2 * k]);
            const __nv_bfloat162* h1 = reinterpret_cast<const __nv_bfloat162*>(&r[2 * k + 1]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float2 f0 = __bfloat1622float2(h0[j]), f1 = __bfloat1622float2(h1[j]);
              acc[2 * j] += w[k] * f0.x; acc[2 * j + 1] += w[k] * f0.y;
              acc[8 + 2 * j] += w[k] * f1.x; acc[8 + 2 * j + 1] += w[k] * f1.y;
            }
          }
          uint4 o0, o1;
          __nv_bfloat162* q0 = reinterpret_cast<__nv_bfloat162*>(&o0);
          __nv_bfloat162* q1 = reinterpret_cast<__nv_bfloat162*>(&o1);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            q0[j] = __floats2bfloat162_rn(acc[2 * j], acc[2 * j + 1]);
            q1[j] = __floats2bfloat162_rn(acc[8 + 2 * j], acc[8 + 2 * j + 1]);
          }
          const int c = gather_col(gw, i);
          uint8_t* kb_base = smem + Smem::lat + (lane >> 2) * kOperandKB;
          const int k_in = (lane & 3) * 16;
          *reinterpret_cast<uint4*>(kb_base + swz_offset(c, k_in)) = o0;
          *reinterpret_cast<uint4*>(kb_base + swz_offset(c, k_in + 8)) = o1;
        };
        {
          uint4 ra[8], rb[8];
          float wa[4], wb[4];
          load_col(0, ra, wa);                       // the first two columns' loads go out BEFORE the operand buffers are free:
          load_col(1, rb, wb);                       // they only fill registers
          mbar_wait_cluster(bar(B_IN_FREE), par_free);
          par_free ^= 1;
          if (fill == 0) {                           // the sin/cos work runs under the first loads' latency
#pragma unroll 1
            for (int i = 0; i < 16; ++i) zfeat_col(i);
          }
#pragma unroll 1
          for (int i = 0; i < 16; i += 2) {
            blend_col(i, ra, wa);
            if (i + 2 < 16) load_col(i + 2, ra, wa);
            blend_col(i + 1, rb, wb);
            if (i + 3 < 16) load_col(i + 3, rb, wb);
          }
        }
        fence_proxy_async();                 // the gather writes this CTA's own shared memory only
        __syncwarp();
        if (lane == 0) { if (crank == 0) mbar_arrive(bar(B_IN_READY)); else mbar_arrive_cluster_relaxed(lbar(B_IN_READY)); }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                    // no CTA exits (or frees TMEM) while the pair may still touch it
  if (warp == 1) tmem_dealloc_2sm(tmem_base, kTmemCols);
}

}  // namespace pair

// ---- host side ---------------------------------------------------------------------------------------------
static pair::Sched pair_sched(const pnr_mlp_params* p, int proj) {
  return pair::Sched{p->n_blocks, p->combine_layer, p->combine_layer, proj ? p->d_hidden / 64 : p->d_latent / 64, proj};
}
// padded hidden width Hp of the packed network: 256 * hidden_tiles
int hidden_tiles(const pnr_mlp_params* p) { return p->d_hidden <= 256 ? 1 : 2; }
int pair_stages(const pnr_mlp_params* p, int proj) {
  pair::Sched s = pair_sched(p, proj);
  return hidden_tiles(p) == 1 ? pair::sched_total<1>(s) : pair::sched_total<2>(s);
}
size_t pair_stream_bytes(const pnr_mlp_params* p, int proj) { return (size_t)pair_stages(p, proj) * 2 * kStageBytes; }
int pair_pack(const pnr_mlp_params* p, uint8_t* stream, int proj, cudaStream_t st) {
  pair::Sched s = pair_sched(p, proj);
  const int n = pair_stages(p, proj);
  PNR_REQUIRE(n < pair::kMaxStages, PNR_ERR_UNSUPPORTED, "pair_pack: %d stages exceed the stage program (one padding entry is needed)", n);
  if (hidden_tiles(p) == 1) pair::pack_stages_kernel<1><<<n * 2, 256, 0, st>>>(*p, s, stream);
  else pair::pack_stages_kernel<2><<<n * 2, 256, 0, st>>>(*p, s, stream);
  PNR_CHECK_LAUNCH("pair::pack_stages_kernel");
  return PNR_OK;
}

// scratch for the view means: 2 tiles x 64 columns x 512 features fp32 per resident CTA pair.  Sized for the widest hidden
// layer: an upper bound for narrower networks (pnr_field_workspace_bytes has no parameters to size it from).
size_t pair_workspace_bytes() {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return (size_t)(sms / 2) * 2 * pair::kNCol * kHidden * sizeof(float);
}

int field_forward_pair(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp, const uint8_t* stream,
                       const float* bx, const float* bh, const float* bo, float* out, void* ws, size_t ws_bytes,
                       int num_freqs, float freq_factor, int raw, int proj, cudaStream_t st) {
  PNR_REQUIRE(ws && ws_bytes >= pair_workspace_bytes() && ((uintptr_t)ws & 15) == 0, PNR_ERR_ARG,
              "field_forward_pair: workspace of pnr_field_workspace_bytes() = %zu bytes required (got %zu)",
              pair_workspace_bytes(), ws_bytes);
  float* xbar = (float*)ws;
  pair::Sched sch = pair_sched(mp, proj);
  const int PP = pair::kNCol / sc->NS;
  const int tiles_per_obj = (q->P + PP - 1) / PP;
  const long long n_tiles_ll = (long long)tiles_per_obj * sc->SB;
  PNR_REQUIRE(n_tiles_ll < (1LL << 31), PNR_ERR_ARG, "field_forward_pair: too many tiles");
  const int n_tiles = (int)n_tiles_ll;
  // tensor map over the packed pair stream: rows = stages x 256, 64 bf16 per row (128 B), box = 64 x 128, no swizzle
  // (the stream is already stored in the swizzled operand layout)
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    PNR_REQUIRE(e == cudaSuccess && fn, PNR_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
    encode = (EncodeFn)fn;
  }
  CUtensorMap tmap;
  cuuint64_t gdim[2] = {64, (cuuint64_t)pair_stages(mp, proj) * 256};
  cuuint64_t gstride[1] = {128};
  cuuint32_t box[2] = {64, 128};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)stream, gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PNR_REQUIRE(r == CUDA_SUCCESS, PNR_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int G = pair::kNCol / PP;                        // tile pairs per super group (see field_pair_kernel)
  // max over one view is the view itself: NS == 1 runs the average instantiation whatever combine_type says
  const bool vmax = mp->combine_type == PNR_COMBINE_MAX && sc->NS > 1;
  const int n_groups = ((n_tiles + 1) / 2 + G - 1) / G;  // super groups
  const bool mt1 = hidden_tiles(mp) == 1;
#define PNR_LAUNCH_PAIR(NSV)                                                                                     \
  case NSV: {                                                                                                    \
    auto kern = mt1 ? (vmax ? pair::field_pair_kernel<NSV, (NSV > 1), 1> : pair::field_pair_kernel<NSV, false, 1>)  \
                    : (vmax ? pair::field_pair_kernel<NSV, (NSV > 1), 2> : pair::field_pair_kernel<NSV, false, 2>); \
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pair::Smem::total); \
    PNR_REQUIRE(e == cudaSuccess, PNR_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));             \
    cudaLaunchConfig_t cfg = {};                                                                                 \
    cudaLaunchAttribute attr[1];                                                                                 \
    attr[0].id = cudaLaunchAttributeClusterDimension;                                                            \
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;                    \
    cfg.blockDim = dim3(pair::kThreads); cfg.dynamicSmemBytes = pair::Smem::total; cfg.stream = st;              \
    cfg.attrs = attr; cfg.numAttrs = 1;                                                                          \
    cfg.gridDim = dim3(sms / 2 * 2);                                                                             \
    int max_pairs = sms / 2, mc = 0;                                                                             \
    if (cudaOccupancyMaxActiveClusters(&mc, kern, &cfg) == cudaSuccess && mc > 0 && mc < max_pairs) max_pairs = mc; \
    const int n_pairs = n_groups < max_pairs ? n_groups : max_pairs;                                             \
    cfg.gridDim = dim3(n_pairs * 2);                                                                             \
    e = cudaLaunchKernelEx(&cfg, kern, *sc, *q, tmap, bx, bh, bo, out, xbar, sch, num_freqs, freq_factor, tiles_per_obj, \
                           n_tiles, (int)mp->d_out, raw);                                                        \
    PNR_REQUIRE(e == cudaSuccess, PNR_ERR_CUDA, "field_pair_kernel launch: %s", cudaGetErrorString(e));          \
  } break;
  switch (sc->NS) {
    PNR_LAUNCH_PAIR(1) PNR_LAUNCH_PAIR(2) PNR_LAUNCH_PAIR(3) PNR_LAUNCH_PAIR(4) PNR_LAUNCH_PAIR(5) PNR_LAUNCH_PAIR(6) PNR_LAUNCH_PAIR(8)
    default: PNR_REQUIRE(false, PNR_ERR_UNSUPPORTED, "field_forward_pair: NS=%d", sc->NS);
  }
#undef PNR_LAUNCH_PAIR
  PNR_CHECK_LAUNCH("field_pair_kernel");
  return PNR_OK;
}

}  // namespace pnr
