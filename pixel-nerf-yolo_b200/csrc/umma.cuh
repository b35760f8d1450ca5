// sm_100a building blocks of the CTA-pair kernels: mbarrier, tensor-map (TMA) loads, TMEM allocation, tcgen05.mma / ld / st,
// the shared-memory operand layout used by every tensor-core tile in this library, and the host side of a pair launch
// (tensor maps, co-resident pair count, cluster launch).
//
// Operand layout (K-major, the default for both A and B of D = A * B^T): a k-block is [rows x 64] bf16, one row =
// 128 bytes, rows packed densely, 16-byte chunks XOR-swizzled with (row % 8) -- the canonical
// SWIZZLE_128B layout that tcgen05 smem descriptors (layout_type = 2, SBO = 1024 B) and TMA share.
// Every k-block base is 1024-byte aligned.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "pnr_common.cuh"

namespace pnr {
namespace umma {

constexpr int kBlockK = 64;                 // bf16 elements per k-block row (128 B)
constexpr int kRowBytes = 128;
constexpr int kUmmaK = 16;                  // K of one tcgen05.mma kind::f16
constexpr int kStageRows = 128;             // weight tile rows (UMMA M)
constexpr int kStageBytes = kStageRows * kRowBytes;   // 16 KiB

// byte offset of element (row, k) inside a k-block
__host__ __device__ __forceinline__ uint32_t swz_offset(int row, int k) {
  return (uint32_t)(row * kRowBytes + ((((k >> 3) ^ (row & 7)) & 7) << 4) + ((k & 7) << 1));
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

// One lane of a converged warp (PTX elect.sync); the others get 0.  Code under `if (elect_one())` that only uses
// values computed OUTSIDE it in warp-uniform control flow lets ptxas keep tcgen05 operands in uniform registers.
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred;
}

// ---- mbarrier -----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (launch error) instead of hanging the GPU.  The spin lives out of line so
// that the (latency-critical, single-thread) MMA issue loop stays small.
static __device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity) {
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      printf("pnr: mbarrier wait timed out (block %d thread %d bar 0x%x parity %u)\n", (int)blockIdx.x,
             (int)threadIdx.x, bar, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (!mbar_try_wait(bar, parity)) mbar_wait_slow(bar, parity);
}

// ---- proxies / fences -------------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async() {   // generic-proxy smem writes -> visible to UMMA/TMA
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- thread-block cluster -------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---- descriptors ------------------------------------------------------------------------------------
// K-major, SWIZZLE_128B: start>>4 | LBO(1)<<16 | SBO(1024>>4)<<32 | version(1)<<46 | layout(2)<<61
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// MN-major SWIZZLE_128B tile made of 64-feature x 64-row boxes (8 KiB each) laid one after the other along MN:
// LBO = byte distance between 64-element MN atoms = 8 192, SBO = byte distance between 8-row K groups = 1 024
__device__ __forceinline__ uint64_t smem_desc_mn(uint32_t saddr) {
  constexpr uint32_t lbo = 8192, sbo = 1024;
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

// ---- TMEM <-> registers (32 lanes x 32-bit, N consecutive columns per thread) ---------------------------
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
// NCOLS in {16,32,64}: issue all loads, then one wait.
template <int NCOLS>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t* r) {
#pragma unroll
  for (int c = 0; c < NCOLS; c += 16) tmem_ld16(taddr + c, r + c);
  tmem_ld_wait();
}
template <int NCOLS>
__device__ __forceinline__ void tmem_ld_nowait(uint32_t taddr, uint32_t* r) {   // caller issues tmem_ld_wait() before using r
#pragma unroll
  for (int c = 0; c < NCOLS; c += 16) tmem_ld16(taddr + c, r + c);
}
template <int NCOLS>
__device__ __forceinline__ void tmem_st(uint32_t taddr, const uint32_t* r) {
#pragma unroll
  for (int c = 0; c < NCOLS; c += 16) tmem_st16(taddr + c, r + c);
  tmem_st_wait();
}

}  // namespace umma
}  // namespace pnr

// =====================================================================================================
// CTA-pair (cta_group::2) building blocks: one tcgen05.mma spans the two SMs of a cluster of 2.  A (M=256) is split
// by rows and B (N) by rows between the two CTAs, each reading its half from ITS OWN shared memory at the same
// offset; each CTA's TMEM receives its 128 rows x N columns of D.  Issued by one thread of the leader CTA (rank 0).
// =====================================================================================================
namespace pnr {
namespace umma {

__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t cta_rank) {   // address of the same offset in a peer CTA
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(cta_rank));
  return r;
}
// arrive (count 1) on an mbarrier anywhere in the cluster, without the (costly, ~1k cycles) cluster-scope release: only valid
// after an explicit fence that already made the data visible where it will be consumed (fence.proxy.async on the writer side)
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint32_t bar, uint32_t parity) {       // acquire at cluster scope
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
static __device__ __noinline__ void mbar_wait_cluster_slow(uint32_t bar, uint32_t parity) {
  const long long t0 = clock64();
  while (!mbar_try_wait_cluster(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      printf("pnr: cluster mbarrier wait timed out (block %d thread %d bar 0x%x parity %u)\n", (int)blockIdx.x,
             (int)threadIdx.x, bar, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  if (!mbar_try_wait_cluster(bar, parity)) mbar_wait_cluster_slow(bar, parity);
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// Asynchronous 16-byte store into a peer CTA's shared memory: the bytes are counted on an mbarrier of the DESTINATION CTA
// (complete_tx), so the sender never waits for the write to be performed (no fence on its side).
__device__ __forceinline__ void st_async_v4(uint32_t cluster_addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d,
                                            uint32_t cluster_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(cluster_addr),
               "r"(a), "r"(b), "r"(c), "r"(d), "r"(cluster_bar)
               : "memory");
}
// One arrival on a (possibly remote) mbarrier that also announces `bytes` of st.async / bulk traffic for the current phase.
__device__ __forceinline__ void mbar_arrive_expect_tx_cluster(uint32_t cluster_bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.relaxed.cluster.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_bar), "r"(bytes) : "memory");
}

__device__ __forceinline__ void tmem_alloc_2sm(uint32_t dst_smem, uint32_t ncols) {   // one full warp in EACH CTA, same dst offset
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// kind::f16, A=B=bf16, D=f32, M=256 (pair), N=n; a_mn / b_mn: that operand is MN-major instead of K-major
__host__ __device__ __forceinline__ uint32_t instr_desc_bf16_2sm(int n, int a_mn = 0, int b_mn = 0) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(256 >> 4) << 24);
}
__device__ __forceinline__ void mma_bf16_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_kblock_desc_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                    bool accumulate_first) {
#pragma unroll
  for (int ks = 0; ks < kBlockK / kUmmaK; ++ks)
    mma_bf16_2sm(d_tmem, a_desc + 2 * ks, b_desc + 2 * ks, idesc, (accumulate_first || ks > 0) ? 1u : 0u);
}
// completion of all prior tcgen05 ops of this thread -> arrive on the barrier at this offset in every CTA of cta_mask
__device__ __forceinline__ void mma_commit_2sm(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(cta_mask)
               : "memory");
}
// 2-D tensor-map TMA load into THIS CTA's shared memory whose completion is signalled on the LEADER CTA's mbarrier
// (same offset; bit 24 of a shared::cluster address selects the CTA of the pair)
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const void* tmap, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(tmap), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}

// 8x8 transpose across the 8 lanes of a lane group (lanes 8g..8g+7): in: a[k] = value of THIS lane for item k;
// out: a[k] = value of lane (8g + k) for item (lane % 8).  Three butterfly rounds of 4 shuffles, static register indices.
__device__ __forceinline__ void transpose8x8(uint32_t (&a)[8], int lane) {
#pragma unroll
  for (int d = 4; d >= 1; d >>= 1) {
    const bool up = (lane & d) != 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      if (k & d) continue;
      const uint32_t send = up ? a[k] : a[k | d];
      const uint32_t recv = __shfl_xor_sync(0xffffffffu, send, d);
      if (up) a[k] = recv; else a[k | d] = recv;
    }
  }
}

// ---- host side of a pair launch ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// 2-D bf16 tensor map over a row-major [rows x cols] matrix with leading dimension ld (elements); box = box_c x box_r
inline int make_map(CUtensorMap* m, const void* base, long long rows, long long cols, long long ld, int box_c, int box_r, bool swizzle) {
  static EncodeFn enc = nullptr;
  if (!enc) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess) enc = (EncodeFn)fn;
  }
  PNR_REQUIRE(enc, PNR_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  PNR_REQUIRE(((uintptr_t)base & 15) == 0 && (ld * 2) % 16 == 0, PNR_ERR_ARG, "tensor map: base / row pitch must be 16-byte aligned");
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_c, (cuuint32_t)box_r};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PNR_REQUIRE(r == CUDA_SUCCESS, PNR_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return PNR_OK;
}

// launch configuration of n_pairs clusters of 2 CTAs; attr must outlive the returned configuration
inline cudaLaunchConfig_t pair_config(cudaLaunchAttribute* attr, int n_pairs, int threads, int smem_bytes, cudaStream_t st) {
  attr->id = cudaLaunchAttributeClusterDimension;
  attr->val.clusterDim.x = 2; attr->val.clusterDim.y = 1; attr->val.clusterDim.z = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * n_pairs); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem_bytes; cfg.stream = st;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cfg;
}

// Sets kern's dynamic shared-memory limit to smem_bytes and returns in *n_pairs the CTA pairs of kern that can be resident at
// once: cudaOccupancyMaxActiveClusters, at most SMs / 2.  The pair kernels are persistent with a static round-robin over
// their units, so they must not be launched with more pairs than that.
template <typename Kern>
int pair_capacity(Kern kern, int threads, int smem_bytes, int* n_pairs) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
  PNR_REQUIRE(e == cudaSuccess, PNR_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int pairs = sms / 2, mc = 0;
  cudaLaunchAttribute attr;
  const cudaLaunchConfig_t cfg = pair_config(&attr, pairs, threads, smem_bytes, 0);
  if (cudaOccupancyMaxActiveClusters(&mc, kern, &cfg) == cudaSuccess && mc > 0 && mc < pairs) pairs = mc;
  *n_pairs = pairs;
  return PNR_OK;
}

// Launches 2 x n_pairs CTAs of kern (after pair_capacity) as clusters of 2; `name` names the kernel in error messages.
template <typename Kern, typename... Args>
int launch_pairs(Kern kern, int n_pairs, int threads, int smem_bytes, cudaStream_t st, const char* name, const Args&... args) {
  cudaLaunchAttribute attr;
  const cudaLaunchConfig_t cfg = pair_config(&attr, n_pairs, threads, smem_bytes, st);
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, args...);
  PNR_REQUIRE(e == cudaSuccess, PNR_ERR_CUDA, "%s launch: %s", name, cudaGetErrorString(e));
  PNR_CHECK_LAUNCH(name);
  return PNR_OK;
}

}  // namespace umma
}  // namespace pnr
