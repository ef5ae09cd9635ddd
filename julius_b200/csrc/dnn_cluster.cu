// dnn_cluster.cu -- EXPERIMENTAL 2-CTA cluster variant of the DNN GEMM (JB200_DNN_KERNEL=2).  Opt-in (not faster than the
// persistent kernel); held bit-identical to dnn_gemm_persistent by tests/test_gpu_scoring_shapes.py.  Kept in its own translation unit so that the shipped kernels in dnn.cu stay bit-for-bit what was
// validated (adding a kernel to dnn.cu perturbed ptxas' register allocation of the others).  The small PTX wrappers and
// the argument block are repeated from dnn.cu on purpose.
#include "common.cuh"
#include <cuda.h>
#include <cuda_bf16.h>
#include <algorithm>

namespace jb200 {
namespace cluster2 {

static constexpr int BM = 128, BN = 128, BK = 64, STAGES = 3;
static constexpr int TILE_BYTES = BM * BK * 2;                 // 16 KB (A and B tiles are the same size)
static constexpr int STAGE_BYTES = 4 * TILE_BYTES;             // A_hi A_lo B_hi B_lo
static constexpr int GEMM_THREADS = 192;
static constexpr int GEMM_SMEM = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
static constexpr int LOGISTIC_N = 320001;

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               :: "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// K-major, 128-byte swizzle operand descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor):
// start>>4 [0,14) | LBO=1 [16,30) | SBO=1024>>4 [32,46) | version=1 [46,48) | layout SWIZZLE_128B=2 [61,64)
__device__ __forceinline__ uint64_t make_desc(const void *smem) {
  uint64_t d = (uint64_t)((smem_u32(smem) & 0x3ffff) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, N=BN, M=BM
__device__ __forceinline__ uint32_t make_idesc() {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t *r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// logistic_func, calc_dnn.c:362-369
__device__ __forceinline__ float logistic_ref(float x, const float *__restrict__ tbl) {
  if (x <= -8.0f) return 0.000334f;
  if (x >= 8.0f) return 0.999666f;
  const float t = __fadd_rn(x, 8.0f);
  const int idx = (int)__dadd_rn((double)__fmul_rn(t, 20000.0f), 0.5);
  return __ldg(tbl + idx);
}

struct GemmArgs {
  int M, N, K;                 // rows (frames), outputs, inputs
  const float *bias;           // [N]
  const float *logistic;       // table
  __nv_bfloat16 *out_hi, *out_lo; int ld_out;   // hidden layers: next operands [M][ld_out]
  float *logits; int ld_logits;                 // last layer: fp32 [M][ld_logits]
  int last;
};

template <int BN_>
struct PersistentCfg {
  static constexpr int STAGES_ = (BN_ == 128) ? 3 : 2;
  static constexpr int B_TILE = BN_ * BK * 2;
  static constexpr int STAGE = 2 * TILE_BYTES + 2 * B_TILE;     // A_hi A_lo B_hi B_lo
  static constexpr int SMEM = STAGES_ * STAGE + 1024 + 256;
};

// ---- 2-CTA cluster variant (EXPERIMENTAL: JB200_DNN_KERNEL=2) ------------------------------------------------------------
// dnn_gemm_persistent<256> is bound by the TMA feed (DESIGN.md K2): ~6100 cycles for the six 128-row boxes of a stage.
// Here two CTAs of a cluster work on vertically adjacent 128x256 tiles (same weight columns): each CTA issues its own
// activation boxes plus HALF of the weight boxes, multicast into both CTAs' shared memory, so a stage costs four boxes
// instead of six per CTA while both still receive all 96 KB.  Protocol differences to the single-CTA kernel:
//   * full[s] of a CTA collects the transaction bytes of its own loads and of the peer's multicast half;
//   * a stage may only be refilled when BOTH CTAs' MMAs are done with it (the peer writes into it): empty[s] counts two
//     arrivals, every MMA warp commits to the empty barrier of both CTAs (tcgen05.commit ... multicast::cluster);
//   * cluster-wide barrier after the mbarrier initialisation and before exit.
__device__ __forceinline__ void tma_load_2d_mc(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, uint16_t mask) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
               :: "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask) : "memory");
}
__device__ __forceinline__ void tc_commit_mc(uint64_t *bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               :: "r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r;
}

__global__ void __launch_bounds__(GEMM_THREADS, 1)
dnn_gemm_cluster2(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                  const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                  const GemmArgs g) {
  constexpr int BN_ = 256;
  using Cfg = PersistentCfg<BN_>;
  constexpr int S = Cfg::STAGES_;
  extern __shared__ unsigned char dsm_raw[];
  unsigned char *dsm = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(dsm_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t *full = reinterpret_cast<uint64_t *>(dsm + S * Cfg::STAGE);
  uint64_t *empty = full + S;
  uint64_t *tmem_full = empty + S;
  uint64_t *tmem_empty = tmem_full + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();                    // 0 or 1: which of the two row blocks / weight halves is mine
  const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
  const int nkb = (g.K + BK - 1) / BK;
  const int n_nblk = (g.N + BN_ - 1) / BN_, n_mblk = (g.M + BM - 1) / BM;
  const int n_pairs = ((n_mblk + 1) >> 1) * n_nblk;            // both CTAs walk the same pair list (an odd last row block is padding)

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 2); }
    for (int b = 0; b < 2; b++) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], 4); }
    mbar_fence_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tmem_slot)), "r"((uint32_t)(2 * BN_)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                           // the peer's barriers exist before anything is multicast at them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int it = 0;
      for (int pair = cluster_id; pair < n_pairs; pair += n_clusters) {
        const int m0 = (2 * (pair / n_nblk) + (int)rank) * BM, n0 = (pair % n_nblk) * BN_;
        for (int kb = 0; kb < nkb; kb++, it++) {
          const int s = it % S;
          const uint32_t ph = (it / S) & 1;
          mbar_wait(&empty[s], ph ^ 1);                         // both CTAs have released the stage
          unsigned char *st = dsm + s * Cfg::STAGE;
          mbar_expect_tx(&full[s], Cfg::STAGE);                 // own A (32 KB) + both halves of B (64 KB)
          tma_load_2d(st, &map_a_hi, &full[s], kb * BK, m0);
          tma_load_2d(st + TILE_BYTES, &map_a_lo, &full[s], kb * BK, m0);
          unsigned char *bh = st + 2 * TILE_BYTES, *bl = bh + Cfg::B_TILE;
          tma_load_2d_mc(bh + rank * TILE_BYTES, &map_b_hi, &full[s], kb * BK, n0 + (int)rank * 128, (uint16_t)3);
          tma_load_2d_mc(bl + rank * TILE_BYTES, &map_b_lo, &full[s], kb * BK, n0 + (int)rank * 128, (uint16_t)3);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN_ >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      int it = 0, i = 0;
      for (int pair = cluster_id; pair < n_pairs; pair += n_clusters, i++) {
        const int b = i & 1;
        mbar_wait(&tmem_empty[b], (uint32_t)((i >> 1) & 1) ^ 1u);
        tc_fence_after();
        const uint32_t acc = tmem_base + (uint32_t)(b * BN_);
        for (int kb = 0; kb < nkb; kb++, it++) {
          const int s = it % S;
          const uint32_t ph = (it / S) & 1;
          mbar_wait(&full[s], ph);
          tc_fence_after();
          unsigned char *st = dsm + s * Cfg::STAGE;
          const uint64_t a_hi = make_desc(st), a_lo = make_desc(st + TILE_BYTES);
          const uint64_t b_hi = make_desc(st + 2 * TILE_BYTES), b_lo = make_desc(st + 2 * TILE_BYTES + Cfg::B_TILE);
#pragma unroll
          for (int k = 0; k < BK / 16; k++) {
            const uint64_t adv = (uint64_t)(k * 32 >> 4);
            tc_mma_bf16(acc, a_hi + adv, b_hi + adv, idesc, (kb | k) ? 1u : 0u);
            tc_mma_bf16(acc, a_hi + adv, b_lo + adv, idesc, 1u);
            tc_mma_bf16(acc, a_lo + adv, b_hi + adv, idesc, 1u);
          }
          tc_commit_mc(&empty[s], (uint16_t)3);                 // release the stage in BOTH CTAs
        }
        tc_commit(&tmem_full[b]);
      }
    }
  } else {
    const int q = warp & 3;
    int i = 0;
    for (int pair = cluster_id; pair < n_pairs; pair += n_clusters, i++) {
      const int b = i & 1;
      const int m0 = (2 * (pair / n_nblk) + (int)rank) * BM, n0 = (pair % n_nblk) * BN_;
      mbar_wait(&tmem_full[b], (uint32_t)((i >> 1) & 1));
      tc_fence_after();
      const int row = m0 + q * 32 + lane;
#pragma unroll 1
      for (int c = 0; c < BN_ / 32; c++) {
        uint32_t r[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(b * BN_ + c * 32), r);
        const int col0 = n0 + c * 32;
        if (row < g.M) {
          if (g.last) {
            float *dst = g.logits + (size_t)row * g.ld_logits + col0;
#pragma unroll
            for (int e = 0; e < 32; e++)
              if (col0 + e < g.N) dst[e] = __uint_as_float(r[e]) + __ldg(g.bias + col0 + e);
          } else {
            __align__(16) __nv_bfloat16 hi[32], lo[32];
#pragma unroll
            for (int e = 0; e < 32; e++) {
              float v = 0.0f;
              if (col0 + e < g.N) v = logistic_ref(__uint_as_float(r[e]) + __ldg(g.bias + col0 + e), g.logistic);
              const __nv_bfloat16 h = __float2bfloat16_rn(v);
              hi[e] = h;
              lo[e] = __float2bfloat16_rn(v - __bfloat162float(h));
            }
            uint4 *dh = reinterpret_cast<uint4 *>(g.out_hi + (size_t)row * g.ld_out + col0);
            uint4 *dl = reinterpret_cast<uint4 *>(g.out_lo + (size_t)row * g.ld_out + col0);
#pragma unroll
            for (int v4 = 0; v4 < 4; v4++)
              if (col0 + v4 * 8 < g.ld_out) { dh[v4] = reinterpret_cast<const uint4 *>(hi)[v4]; dl[v4] = reinterpret_cast<const uint4 *>(lo)[v4]; }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[b]);
    }
  }
  __syncthreads();
  cluster_sync_all();                                           // nobody leaves while the peer may still write into it
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"((uint32_t)(2 * BN_)) : "memory");
  }
}


}  // namespace cluster2

// one layer: C[M x N] = A . W^T through the cluster kernel; returns a JB200 error code
int dnn_launch_cluster2(const CUtensorMap &ma_hi, const CUtensorMap &ma_lo, const CUtensorMap &mw_hi, const CUtensorMap &mw_lo,
                        int M, int N, int K, const float *bias, const float *logistic, __nv_bfloat16 *out_hi, __nv_bfloat16 *out_lo,
                        int ld_out, float *logits, int ld_logits, int last, int n_sm, cudaStream_t st) {
  using namespace cluster2;
  static bool attr_set = false;
  if (!attr_set) {
    JB_CUDA(cudaFuncSetAttribute(dnn_gemm_cluster2, cudaFuncAttributeMaxDynamicSharedMemorySize, PersistentCfg<256>::SMEM));
    JB_CUDA(cudaFuncSetAttribute(dnn_gemm_cluster2, cudaFuncAttributeNonPortableClusterSizeAllowed, 0));
    attr_set = true;
  }
  GemmArgs g;
  g.M = M; g.N = N; g.K = K; g.bias = bias; g.logistic = logistic; g.out_hi = out_hi; g.out_lo = out_lo; g.ld_out = ld_out;
  g.logits = logits; g.ld_logits = ld_logits; g.last = last;
  const int pairs = ((N + 255) / 256) * ((((M + BM - 1) / BM) + 1) / 2);
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.gridDim = dim3(2 * (unsigned)std::max(1, std::min(pairs, n_sm / 2)));
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = PersistentCfg<256>::SMEM;
  cfg.stream = st; cfg.attrs = attr; cfg.numAttrs = 1;
  JB_CUDA(cudaLaunchKernelEx(&cfg, dnn_gemm_cluster2, ma_hi, ma_lo, mw_hi, mw_lo, g));
  g_launches.fetch_add(1);
  return JB200_OK;
}

}  // namespace jb200
