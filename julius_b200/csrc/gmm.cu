// gmm.cu -- K1: batched diagonal-Gaussian state scoring for all tied states of all frames.
//
// Stands in for the reference's per-(frame,state) lazy evaluation
//   outprob_state -> calc_mix -> gprune_{none,safe,beam,heu} -> compute_g_base -> addlog_array
//   (libsent/src/phmm/outprob.c:183-249, calc_mix.c:40-81, gprune_none.c:58-82,
//    gprune_safe.c:75-202, gprune_common.c:41-126, addlog.c:102-123)
// and for outprob_cd (outprob.c:286-400) in the cd-set kernel.
//
// Layout in HBM.  One 16-byte aligned record per Gaussian, in quads so that a 64-bit register pair
// holds two dimensions for the packed fp32x2 FMA (FFMA2):
//      [ (m0 m1 iv0 iv1) (m2 m3 iv2 iv3) ... (m38 gconst iv38 lnw) ]   (2D+2 floats -> 320 B for D=39)
// Records of a state are contiguous and states follow each other, so a tile of states is ONE
// contiguous byte range that a single 1-D bulk (TMA) copy stages into shared memory
// (cp.async.bulk + mbarrier, double buffered).  Every thread owns FPT frames whose feature
// vectors live in registers; all lanes of a warp read the same parameter word (shared-memory
// broadcast), so a record is fetched from L2/HBM once per 128*FPT frames.
//
// Two arithmetic modes:
//   EXACT  the reference's fp32 statement order (x=v-m; tmp += x*x*iv sequentially over d, no FMA
//          contraction; *-0.5; +ln w; table-driven addlog from the last mixture down to the first;
//          *INV_LOG_TEN in double) -> bit-identical to the compiled reference.
//   FAST   FMA accumulate + streaming exact log-sum-exp -> within 1e-4 relative.
#include "common.cuh"
#include <cmath>
#include <vector>

namespace jb200 {

static constexpr int GMM_THREADS = 128;
static constexpr int GMM_FPT = 2;              // frames per thread
static constexpr int GMM_TILE_STATES = 4;      // max states per staged tile
static constexpr int GMM_TILE_GAUSS = 64;      // max Gaussians per staged tile
static constexpr int GMM_NMAX = 16;            // max -tmix for the pruned variants

__host__ __device__ constexpr int gmm_stride(int D) { return ((2 * D + 2) + 3) & ~3; }

struct GmmTile { int s0, ns, g0, ng; };

// record layout: quads (m_2q, m_2q+1, iv_2q, iv_2q+1); gconst / lnw ride in the unused halves of the
// last quad when D is odd, or in an extra quad when D is even.  Same size as interleaving pairs.
__host__ __device__ constexpr int rec_mean(int d) { return 4 * (d >> 1) + (d & 1); }
__host__ __device__ constexpr int rec_ivar(int d) { return 4 * (d >> 1) + 2 + (d & 1); }
__host__ __device__ constexpr int rec_gconst(int D) { return (D & 1) ? 4 * (D >> 1) + 1 : 2 * D; }
__host__ __device__ constexpr int rec_lnw(int D) { return (D & 1) ? 4 * (D >> 1) + 3 : 2 * D + 1; }

// packed fp32x2 FMA (SASS FFMA2): one issue slot for two lanes' worth of work.  Every use below is an
// exactly-rounded single operation (a*b+0, a*(-1)+c), so the exact mode stays bit-identical.
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  return ((unsigned long long)__float_as_uint(hi) << 32) | __float_as_uint(lo);
}
__device__ __forceinline__ float lo2(unsigned long long v) { return __uint_as_float((unsigned)(v & 0xffffffffu)); }
__device__ __forceinline__ float hi2(unsigned long long v) { return __uint_as_float((unsigned)(v >> 32)); }

__device__ __forceinline__ float addlog_step_exact(float y, float x, const float *__restrict__ tbl) {
  // addlog.c:112-120
  if (x > y) { float t = x; x = y; y = t; }
  float tmp = __fsub_rn(x, y);
  if ((double)tmp < JB200_LOG_ADDMIN) return y;
  unsigned int idx = (unsigned int)__dadd_rn(__dmul_rn((double)(-tmp), 33333.3333), 0.5);
  return __fadd_rn(y, __ldg(tbl + idx));
}

__device__ __forceinline__ float finish_exact(float lp) {
  // calc_mix.c:72-80 for a single stream with weight 1
  if (lp <= JB200_LOG_ZERO || lp == 0.0f) return JB200_LOG_ZERO;
  return (float)((double)lp * JB200_INV_LOG_TEN);
}

// cache_push, gprune_common.c:87-126 (score list sorted descending)
__device__ __forceinline__ int cache_push_dev(float *cs, int *ci, int gprune_num, int id, float score, int len) {
  if (len == 0) { cs[0] = score; ci[0] = id; return 1; }
  if (cs[len - 1] >= score) {
    if (len < gprune_num) { cs[len] = score; ci[len] = id; len++; }
    return len;
  }
  int insertp;
  if (cs[0] < score) insertp = 0;
  else {
    int left = 0, right = len - 1;
    while (left < right) { int mid = (left + right) / 2; if (cs[mid] > score) left = mid + 1; else right = mid; }
    insertp = left;
  }
  int last = (len < gprune_num) ? len : len - 1;
  for (int k = last; k > insertp; k--) { cs[k] = cs[k - 1]; ci[k] = ci[k - 1]; }
  cs[insertp] = score; ci[insertp] = id;
  if (len < gprune_num) len++;
  return len;
}

template <int D, bool EXACT, bool PRUNE>
__global__ void __launch_bounds__(GMM_THREADS)
gmm_score_kernel(const float *__restrict__ pk, const GmmTile *__restrict__ tiles, int tiles_per_chunk, int n_tiles,
                 const float *__restrict__ feats, float *__restrict__ rows, int T, int row_stride,
                 const float *__restrict__ tbl, int gprune_num,
                 const int *__restrict__ seg_off, const int *__restrict__ seg_start, int n_seg) {
  constexpr int STRIDE = gmm_stride(D);
  constexpr int NQ = STRIDE / 4;                 // float4 per record
  __shared__ __align__(128) float buf[2][GMM_TILE_GAUSS * STRIDE];
  __shared__ __align__(8) uint64_t full[2];

  const int tid = threadIdx.x;
  const int f0 = blockIdx.x * (GMM_THREADS * GMM_FPT) + tid;
  const int tile_begin = blockIdx.y * tiles_per_chunk;
  const int tile_end = min(n_tiles, tile_begin + tiles_per_chunk);
  if (tile_begin >= tile_end) return;

  if (tid == 0) { mbar_init(&full[0], 1); mbar_init(&full[1], 1); mbar_fence_init(); }
  __syncthreads();
  if (tid == 0) {
    GmmTile t0 = tiles[tile_begin];
    uint32_t bytes = (uint32_t)t0.ng * STRIDE * 4u;
    mbar_expect_tx(&full[0], bytes);
    bulk_g2s(buf[0], pk + (size_t)t0.g0 * STRIDE, bytes, &full[0]);
  }

  // this thread's frames, in registers
  float v[GMM_FPT][D];                       // scalar copy (pruned variant)
  unsigned long long v2[GMM_FPT][NQ];        // the same, packed (x_2q, x_2q+1) for the FFMA2 path
  // T counts LOGICAL frames.  With a segment list (the batch pipeline scores one time slice of every utterance per
  // launch) logical frame f is frame seg_start[s] + f - seg_off[s] of the feature / score matrices, s = its segment
  int fr[GMM_FPT];
#pragma unroll
  for (int k = 0; k < GMM_FPT; k++) {
    const int fl = f0 + k * GMM_THREADS;
    int fp = min(fl, T - 1);
    if (seg_off != nullptr) {
      int lo = 0, hi = n_seg;
      while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (__ldg(seg_off + mid) <= fp) lo = mid; else hi = mid; }
      fp = __ldg(seg_start + lo) + (fp - __ldg(seg_off + lo));
    }
    fr[k] = (fl < T) ? fp : -1;                      // physical frame, -1 = padding lane
    const float *src = feats + (size_t)fp * D;
#pragma unroll
    for (int d = 0; d < D; d++) v[k][d] = __ldg(src + d);
#pragma unroll
    for (int q = 0; q < NQ; q++) v2[k][q] = pack2((2 * q < D) ? v[k][2 * q < D ? 2 * q : 0] : 0.0f, (2 * q + 1 < D) ? v[k][2 * q + 1 < D ? 2 * q + 1 : 0] : 0.0f);
  }
  const unsigned long long NEG1 = pack2(-1.0f, -1.0f), ZERO2 = pack2(0.0f, 0.0f);

  for (int ti = tile_begin; ti < tile_end; ti++) {
    const int b = (ti - tile_begin) & 1;
    const uint32_t parity = ((ti - tile_begin) >> 1) & 1;
    if (tid == 0 && ti + 1 < tile_end) {
      GmmTile tn = tiles[ti + 1];
      uint32_t bytes = (uint32_t)tn.ng * STRIDE * 4u;
      mbar_expect_tx(&full[b ^ 1], bytes);
      bulk_g2s(buf[b ^ 1], pk + (size_t)tn.g0 * STRIDE, bytes, &full[b ^ 1]);
    }
    const GmmTile tl = tiles[ti];
    mbar_wait(&full[b], parity);
    const float *pb = buf[b];

    int grel = 0;   // Gaussian index relative to tile start, advanced per state
    for (int si = 0; si < tl.ns; si++) {
      // number of mixtures of this state: encoded as consecutive tiles' state_off differences;
      // tile header carries only totals, per-state counts are in the record stream: the host
      // stores the mixture count of state (s0+si) in the pad word of its FIRST record when
      // STRIDE > 2D+2, else in a side table.  We use the side table appended after the tiles.
      const int *mixcnt = reinterpret_cast<const int *>(tiles + n_tiles);
      const int nm = mixcnt[tl.s0 + si];
      float res[GMM_FPT];
      if (!PRUNE) {
        // streaming log-add from the LAST mixture down to the first (addlog.c:108-121)
        float y[GMM_FPT], ssum[GMM_FPT];
#pragma unroll
        for (int k = 0; k < GMM_FPT; k++) { y[k] = JB200_LOG_ZERO; ssum[k] = 0.0f; }
        for (int m = nm - 1; m >= 0; m--) {
          const float4 *p = reinterpret_cast<const float4 *>(pb + (size_t)(grel + m) * STRIDE);
          const float gconst = pb[(size_t)(grel + m) * STRIDE + rec_gconst(D)];
          const float lnw = pb[(size_t)(grel + m) * STRIDE + rec_lnw(D)];
          float acc[GMM_FPT];
          unsigned long long acc2[GMM_FPT];
#pragma unroll
          for (int k = 0; k < GMM_FPT; k++) { acc[k] = gconst; acc2[k] = pack2(gconst, 0.0f); }
#pragma unroll
          for (int q = 0; q < NQ; q++) {
            const int d0 = 2 * q, d1 = 2 * q + 1;
            if (d0 < D) {
              const ulonglong2 w = reinterpret_cast<const ulonglong2 *>(p)[q];     // .x = (m_d0, m_d1)  .y = (iv_d0, iv_d1)
#pragma unroll
              for (int k = 0; k < GMM_FPT; k++) {
                const unsigned long long x2 = fma2(w.x, NEG1, v2[k][q]);           // x = v - m      (exact)
                if (EXACT) {
                  const unsigned long long t2 = fma2(fma2(x2, x2, ZERO2), w.y, ZERO2);   // (x*x)*iv, two roundings as the reference
                  acc[k] = __fadd_rn(acc[k], lo2(t2));                             // tmp += ... in dimension order
                  if (d1 < D) acc[k] = __fadd_rn(acc[k], hi2(t2));
                } else {
                  const unsigned long long xi = fma2(x2, w.y, ZERO2);
                  if (d1 < D) acc2[k] = fma2(xi, x2, acc2[k]);
                  else acc[k] = fmaf(lo2(xi), lo2(x2), 0.0f);                      // odd tail dimension
                }
              }
            }
          }
          if (!EXACT) {
#pragma unroll
            for (int k = 0; k < GMM_FPT; k++) acc[k] = ((D & 1) ? acc[k] : 0.0f) + lo2(acc2[k]) + hi2(acc2[k]);
          }
          const bool invalid = (gconst != gconst);   // NaN marks a NULL density (gprune_none.c:66)
#pragma unroll
          for (int k = 0; k < GMM_FPT; k++) {
            float sc = invalid ? JB200_LOG_ZERO : acc[k] * -0.5f;
            if (EXACT) {
              sc = __fadd_rn(sc, lnw);
              y[k] = addlog_step_exact(y[k], sc, tbl);
            } else {
              sc += lnw;
              if (sc > y[k]) { ssum[k] = ssum[k] * __expf(y[k] - sc) + 1.0f; y[k] = sc; }
              else ssum[k] += __expf(sc - y[k]);
            }
          }
        }
#pragma unroll
        for (int k = 0; k < GMM_FPT; k++) {
          if (EXACT) res[k] = finish_exact(y[k]);
          else {
            float lp = y[k] + __logf(ssum[k]);
            res[k] = (nm == 0 || lp <= JB200_LOG_ZERO) ? JB200_LOG_ZERO : lp * (float)JB200_INV_LOG_TEN;
          }
        }
      } else {
        // safe pruning replay (gprune_safe.c:187-199): mixtures in index order, top-N list,
        // a candidate is dropped iff its full score <= current N-th best (early exit in
        // compute_g_safe is equivalent because the partial sums are non-decreasing).
#pragma unroll
        for (int k = 0; k < GMM_FPT; k++) {
          float cs[GMM_NMAX]; int ci[GMM_NMAX];
          int num = 0; float thres = JB200_LOG_ZERO;
          for (int m = 0; m < nm; m++) {
            const float *rec = pb + (size_t)(grel + m) * STRIDE;
            const float gconst = rec[rec_gconst(D)];
            float acc = gconst;
#pragma unroll
            for (int d = 0; d < D; d++) {
              float x = __fsub_rn(v[k][d], rec[rec_mean(d)]);
              acc = __fadd_rn(acc, __fmul_rn(__fmul_rn(x, x), rec[rec_ivar(d)]));
            }
            float sc = (gconst != gconst) ? JB200_LOG_ZERO : acc * -0.5f;
            if (num >= gprune_num && sc <= thres) continue;
            num = cache_push_dev(cs, ci, gprune_num, m, sc, num);
            thres = cs[num - 1];
          }
          float y = JB200_LOG_ZERO, ssum = 0.0f;
          for (int i = num - 1; i >= 0; i--) {
            float sc = __fadd_rn(cs[i], pb[(size_t)(grel + ci[i]) * STRIDE + rec_lnw(D)]);
            if (EXACT) y = addlog_step_exact(y, sc, tbl);
            else { if (sc > y) { ssum = ssum * __expf(y - sc) + 1.0f; y = sc; } else ssum += __expf(sc - y); }
          }
          if (EXACT) res[k] = finish_exact(y);
          else { float lp = y + __logf(ssum); res[k] = (num == 0 || lp <= JB200_LOG_ZERO) ? JB200_LOG_ZERO : lp * (float)JB200_INV_LOG_TEN; }
        }
      }
#pragma unroll
      for (int k = 0; k < GMM_FPT; k++)
        if (fr[k] >= 0) rows[(size_t)fr[k] * row_stride + tl.s0 + si] = res[k];
      grel += nm;
    }
    __syncthreads();   // everyone is done with buf[b] before it is refilled two tiles later
  }
}

// ---- pseudo-phone set scores (outprob.c:286-400) -------------------------------------------
__global__ void __launch_bounds__(256)
cdset_kernel(float *__restrict__ rows, int T, int row_stride, int S, int C,
             const int *__restrict__ cd_off, const int *__restrict__ cd_states, int method, int maxn) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int t = blockIdx.y;
  if (c >= C || t >= T) return;
  const float *st = rows + (size_t)t * row_stride;
  const int b0 = cd_off[c], n_in = cd_off[c + 1] - b0;
  float out;
  if (method == JB200_IWCD_AVG) {
    float sum = 0.0f; int j = 0;
    for (int i = 0; i < n_in; i++) { float p = st[cd_states[b0 + i]]; if (p > JB200_LOG_ZERO) { sum = __fadd_rn(sum, p); j++; } }
    out = __fdiv_rn(sum, (float)j);
  } else if (method == JB200_IWCD_MAX) {
    float mx = JB200_LOG_ZERO;
    for (int i = 0; i < n_in; i++) { float p = st[cd_states[b0 + i]]; if (mx < p) mx = p; }
    out = mx;
  } else {
    float mp[GMM_NMAX + 1]; int n = 0;
    for (int i = 0; i < n_in; i++) {
      float prob = st[cd_states[b0 + i]];
      if (prob <= JB200_LOG_ZERO) continue;
      if (n == 0 || prob <= mp[n - 1]) {
        if (n == maxn) continue;
        mp[n] = prob; n++;
      } else {
        for (int k = 0; k < n; k++) {
          if (prob > mp[k]) {
            int cnt = n - k - ((n == maxn) ? 1 : 0);
            for (int q = k + cnt; q > k; q--) mp[q] = mp[q - 1];
            mp[k] = prob;
            break;
          }
        }
        if (n < maxn) n++;
      }
    }
    float prob = 0.0f;
    for (int i = 0; i < n; i++) prob = __fadd_rn(prob, mp[i]);
    out = __fdiv_rn(prob, (float)n);
  }
  rows[(size_t)t * row_stride + S + c] = out;
}

// ---- per-Gaussian scores of one frame (calcmix hook contract) ----------------------------------
__global__ void gauss_frame_kernel(const float *__restrict__ pk, int stride, int D, int G,
                                   const float *__restrict__ feat, float *__restrict__ out) {
  int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const float *rec = pk + (size_t)g * stride;
  float gconst = rec[rec_gconst(D)];
  float acc = gconst;
  for (int d = 0; d < D; d++) {
    float x = __fsub_rn(feat[d], rec[rec_mean(d)]);
    acc = __fadd_rn(acc, __fmul_rn(__fmul_rn(x, x), rec[rec_ivar(d)]));
  }
  out[g] = (gconst != gconst) ? JB200_LOG_ZERO : acc * -0.5f;
}

}  // namespace jb200

// =============================================================================================
using namespace jb200;

struct jb200_gmm {
  int device = 0, mode = 0;
  int S = 0, D = 0, G = 0, C = 0, max_mix = 0, stride = 0, row_stride = 0;
  int gprune_method = 0, gprune_num = 0, iwcd_method = 0, iwcd_nbest = 0;
  int n_tiles = 0;
  float *d_pk = nullptr;
  GmmTile *d_tiles = nullptr;      // [n_tiles] followed by int mixcnt[S]
  int *d_cd_off = nullptr, *d_cd_states = nullptr;
  float *d_tbl = nullptr;          // addlog table (exact mode)
  cudaStream_t stream = nullptr;
  // scratch for the host variants
  float *d_feats = nullptr, *d_rows = nullptr; size_t cap_frames = 0;
  int sm_count = 148;
};

namespace jb200 {
int gmm_device(const jb200_gmm *h) { return h->device; }
cudaStream_t gmm_stream(const jb200_gmm *h) { return h->stream; }
int gmm_dim(const jb200_gmm *h) { return h->D; }
int gmm_cd_device(const jb200_gmm *h, const int **cd_off, const int **cd_states, int *method, int *nbest) {
  *cd_off = h->d_cd_off; *cd_states = h->d_cd_states; *method = h->iwcd_method; *nbest = h->iwcd_nbest;
  return 0;
}
}

static void build_addlog_table(std::vector<float> &tbl) {
  // addlog.c:39-57 -- same libm calls on the host, uploaded once
  tbl.resize(500000);
  for (int i = 0; i < 500000; i++) {
    float f = -((float)15 * (float)i / (float)500000);
    tbl[i] = (float)log(1 + exp((double)f));
  }
}

extern "C" int jb200_gmm_create(const jb200_gmm_desc *d, int device, int mode, jb200_gmm **out) {
  if (!d || !out) { set_error("jb200_gmm_create: null argument"); return JB200_ERR_ARG; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { set_error("no CUDA device (libjb200 has no CPU fallback)"); return JB200_ERR_NODEVICE; }
  if (device < 0 || device >= ndev) { set_error("device %d out of range (%d devices)", device, ndev); return JB200_ERR_ARG; }
  if (d->gprune_method != JB200_GPRUNE_NONE && (d->gprune_num < 1 || d->gprune_num > GMM_NMAX)) {
    set_error("-tmix %d outside supported range 1..%d", d->gprune_num, GMM_NMAX); return JB200_ERR_UNSUPPORTED;
  }
  if (d->iwcd_method == JB200_IWCD_NBEST && d->iwcd_nbest > GMM_NMAX) { set_error("-iwcd1 best %d too large", d->iwcd_nbest); return JB200_ERR_UNSUPPORTED; }
  // the descriptor may come from a file: every offset the packer and the kernels follow is checked here
  if (d->n_states < 0 || d->n_gauss < 0 || d->n_cdsets < 0 || d->n_cdset_states < 0) { set_error("jb200_gmm_create: negative size"); return JB200_ERR_ARG; }
  if (d->n_gauss > 0) {
    if (d->dim != 39 && d->dim != 38 && d->dim != 26 && d->dim != 25) { set_error("feature dimension %d not instantiated (39, 38, 26, 25)", d->dim); return JB200_ERR_UNSUPPORTED; }
    if (!d->state_off || !d->mean || !d->ivar || !d->gconst || !d->lnweight || !d->valid) { set_error("jb200_gmm_create: missing Gaussian arrays"); return JB200_ERR_ARG; }
    if (d->state_off[0] != 0 || d->state_off[d->n_states] != d->n_gauss) {
      set_error("state_off runs from %d to %d, not from 0 to n_gauss = %d", d->state_off[0], d->state_off[d->n_states], d->n_gauss); return JB200_ERR_ARG;
    }
    for (int s = 0; s < d->n_states; s++)
      if (d->state_off[s + 1] < d->state_off[s]) { set_error("state_off decreases at state %d (%d -> %d)", s, d->state_off[s], d->state_off[s + 1]); return JB200_ERR_ARG; }
  }
  if (d->n_cdsets > 0) {
    if (!d->cd_off || !d->cd_states) { set_error("jb200_gmm_create: missing cd-set arrays"); return JB200_ERR_ARG; }
    if (d->cd_off[0] != 0 || d->cd_off[d->n_cdsets] != d->n_cdset_states) { set_error("cd_off does not run from 0 to n_cdset_states"); return JB200_ERR_ARG; }
    for (int c = 0; c < d->n_cdsets; c++)
      if (d->cd_off[c + 1] < d->cd_off[c]) { set_error("cd_off decreases at set %d", c); return JB200_ERR_ARG; }
    for (int i = 0; i < d->n_cdset_states; i++)
      if (d->cd_states[i] < 0 || d->cd_states[i] >= d->n_states) { set_error("cd_states[%d] = %d is not a state id", i, d->cd_states[i]); return JB200_ERR_ARG; }
  }
  JB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  JB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) { set_error("device %d is sm_%d%d; libjb200 is built for sm_100a only", device, prop.major, prop.minor); return JB200_ERR_NODEVICE; }

  jb200_gmm *h = new jb200_gmm();
  h->device = device; h->mode = mode; h->sm_count = prop.multiProcessorCount;
  h->S = d->n_states; h->D = d->dim; h->G = d->n_gauss; h->C = d->n_cdsets; h->max_mix = d->max_mix;
  h->gprune_method = d->gprune_method; h->gprune_num = d->gprune_num;
  h->iwcd_method = d->iwcd_method; h->iwcd_nbest = d->iwcd_nbest;
  h->stride = gmm_stride(h->D);
  h->row_stride = (h->S + h->C + 3) & ~3;
  JB_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));

  // pack records
  std::vector<float> pk((size_t)h->G * h->stride, 0.0f);
  for (int g = 0; g < h->G; g++) {
    float *rec = &pk[(size_t)g * h->stride];
    for (int k = 0; k < h->D; k++) { rec[rec_mean(k)] = d->mean[(size_t)g * h->D + k]; rec[rec_ivar(k)] = d->ivar[(size_t)g * h->D + k]; }
    rec[rec_gconst(h->D)] = d->valid[g] ? d->gconst[g] : NAN;
    rec[rec_lnw(h->D)] = d->lnweight[g];
  }
  // tiles: consecutive states, <= GMM_TILE_STATES states with mixtures and <= GMM_TILE_GAUSS Gaussians.  States without
  // mixture slots ride along in the tile of their neighbours (the kernel writes LOG_ZERO for them), so every tile
  // stages at least one Gaussian and every state column is written
  std::vector<GmmTile> tiles;
  std::vector<int> mixcnt(h->S);
  for (int s = 0; s < h->S; s++) {
    mixcnt[s] = (h->G > 0) ? d->state_off[s + 1] - d->state_off[s] : 0;
    if (mixcnt[s] > GMM_TILE_GAUSS) { set_error("state %d has %d mixtures (max %d)", s, mixcnt[s], GMM_TILE_GAUSS); jb200_gmm_destroy(h); return JB200_ERR_UNSUPPORTED; }
  }
  if (h->G > 0) {
    for (int s = 0; s < h->S;) {
      GmmTile t{s, 0, d->state_off[s], 0};
      int filled = 0;
      while (s < h->S && (mixcnt[s] == 0 || filled < GMM_TILE_STATES) && t.ng + mixcnt[s] <= GMM_TILE_GAUSS) {
        filled += mixcnt[s] > 0; t.ng += mixcnt[s]; t.ns++; s++;
      }
      tiles.push_back(t);
    }
  }
  h->n_tiles = (int)tiles.size();
  size_t tile_bytes = tiles.size() * sizeof(GmmTile) + mixcnt.size() * sizeof(int);
  std::vector<char> tb(tile_bytes);
  memcpy(tb.data(), tiles.data(), tiles.size() * sizeof(GmmTile));
  memcpy(tb.data() + tiles.size() * sizeof(GmmTile), mixcnt.data(), mixcnt.size() * sizeof(int));

  JB_CUDA(cudaMalloc(&h->d_pk, pk.size() * sizeof(float) + 16));
  if (!pk.empty()) JB_CUDA(cudaMemcpy(h->d_pk, pk.data(), pk.size() * sizeof(float), cudaMemcpyHostToDevice));
  JB_CUDA(cudaMalloc(&h->d_tiles, tile_bytes + 16));
  JB_CUDA(cudaMemcpy(h->d_tiles, tb.data(), tile_bytes, cudaMemcpyHostToDevice));
  if (h->C > 0) {
    JB_CUDA(cudaMalloc(&h->d_cd_off, sizeof(int) * (h->C + 1)));
    JB_CUDA(cudaMemcpy(h->d_cd_off, d->cd_off, sizeof(int) * (h->C + 1), cudaMemcpyHostToDevice));
    JB_CUDA(cudaMalloc(&h->d_cd_states, sizeof(int) * (d->n_cdset_states + 1)));
    JB_CUDA(cudaMemcpy(h->d_cd_states, d->cd_states, sizeof(int) * d->n_cdset_states, cudaMemcpyHostToDevice));
  }
  std::vector<float> tbl;
  build_addlog_table(tbl);
  JB_CUDA(cudaMalloc(&h->d_tbl, tbl.size() * sizeof(float)));
  JB_CUDA(cudaMemcpy(h->d_tbl, tbl.data(), tbl.size() * sizeof(float), cudaMemcpyHostToDevice));
  *out = h;
  return JB200_OK;
}

extern "C" void jb200_gmm_destroy(jb200_gmm *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaFree(h->d_pk); cudaFree(h->d_tiles); cudaFree(h->d_cd_off); cudaFree(h->d_cd_states); cudaFree(h->d_tbl);
  cudaFree(h->d_feats); cudaFree(h->d_rows);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

extern "C" int jb200_gmm_score_stride(const jb200_gmm *h) { return h ? h->row_stride : 0; }
extern "C" int jb200_gmm_n_states(const jb200_gmm *h) { return h ? h->S : 0; }
extern "C" int jb200_gmm_n_cdsets(const jb200_gmm *h) { return h ? h->C : 0; }

template <int D>
static int launch_gmm(jb200_gmm *h, const float *d_feats, int T, float *d_rows, int row_stride, cudaStream_t st,
                      const int *seg_off = nullptr, const int *seg_start = nullptr, int n_seg = 0) {
  const int fblocks = (T + GMM_THREADS * GMM_FPT - 1) / (GMM_THREADS * GMM_FPT);
  // enough CTAs for >= 2 waves of 4 CTAs/SM when the frame count alone does not provide them
  int want = h->sm_count * 8;
  int chunks = (want + fblocks - 1) / fblocks;
  if (chunks < 1) chunks = 1;
  if (chunks > h->n_tiles) chunks = h->n_tiles;
  int tiles_per_chunk = (h->n_tiles + chunks - 1) / chunks;
  chunks = (h->n_tiles + tiles_per_chunk - 1) / tiles_per_chunk;
  dim3 grid(fblocks, chunks);
  const bool prune = h->gprune_method != JB200_GPRUNE_NONE;
  const bool exact = h->mode == JB200_GMM_EXACT;
#define JB_GO(E, P) gmm_score_kernel<D, E, P><<<grid, GMM_THREADS, 0, st>>>(h->d_pk, h->d_tiles, tiles_per_chunk, h->n_tiles, d_feats, d_rows, T, row_stride, h->d_tbl, h->gprune_num, seg_off, seg_start, n_seg)
  if (exact && !prune) JB_GO(true, false);
  else if (exact && prune) JB_GO(true, true);
  else if (!exact && !prune) JB_GO(false, false);
  else JB_GO(false, true);
#undef JB_GO
  JB_LAUNCH_CHECK();
  return JB200_OK;
}

extern "C" int jb200_gmm_cdsets_device(jb200_gmm *h, float *d_rows, int T, void *stream) {
  if (!h) { set_error("null handle"); return JB200_ERR_ARG; }
  if (h->C == 0 || T == 0) return JB200_OK;
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  JB_CUDA(cudaSetDevice(h->device));
  // grid.y is limited to 65535 frames per launch
  for (int t0 = 0; t0 < T; t0 += 65535) {
    int tt = T - t0 < 65535 ? T - t0 : 65535;
    dim3 grid((h->C + 255) / 256, tt);
    cdset_kernel<<<grid, 256, 0, st>>>(d_rows + (size_t)t0 * h->row_stride, tt, h->row_stride, h->S, h->C, h->d_cd_off, h->d_cd_states,
                                       h->iwcd_method, h->iwcd_nbest);
    JB_LAUNCH_CHECK();
  }
  return JB200_OK;
}

namespace jb200 {
// state columns only, caller-chosen row stride (used by the decoder, which evaluates cd sets on demand)
// seg_off/seg_start (device, n_seg entries, may be null): T logical frames gathered from segments of the matrices
int gmm_launch_states(jb200_gmm *h, const float *d_feats, int T, float *d_rows, int row_stride, cudaStream_t st,
                      const int *seg_off, const int *seg_start, int n_seg) {
  if (T <= 0) return JB200_OK;
  if (h->G == 0) { set_error("this scorer carries no Gaussians (DNN-HMM layout only)"); return JB200_ERR_ARG; }
  JB_CUDA(cudaSetDevice(h->device));
  switch (h->D) {
    case 39: return launch_gmm<39>(h, d_feats, T, d_rows, row_stride, st, seg_off, seg_start, n_seg);
    case 38: return launch_gmm<38>(h, d_feats, T, d_rows, row_stride, st, seg_off, seg_start, n_seg);
    case 26: return launch_gmm<26>(h, d_feats, T, d_rows, row_stride, st, seg_off, seg_start, n_seg);
    case 25: return launch_gmm<25>(h, d_feats, T, d_rows, row_stride, st, seg_off, seg_start, n_seg);
    default: set_error("feature dimension %d not instantiated (39, 38, 26, 25)", h->D); return JB200_ERR_UNSUPPORTED;
  }
}
}  // namespace jb200

extern "C" int jb200_gmm_score_device(jb200_gmm *h, const float *d_feats, int T, float *d_rows, void *stream) {
  if (!h || !d_feats || !d_rows) { set_error("jb200_gmm_score_device: null argument"); return JB200_ERR_ARG; }
  if (T <= 0) return JB200_OK;
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  int rc = gmm_launch_states(h, d_feats, T, d_rows, h->row_stride, st, nullptr, nullptr, 0);
  if (rc) return rc;
  return jb200_gmm_cdsets_device(h, d_rows, T, st);
}

static int ensure_scratch(jb200_gmm *h, int T) {
  if ((size_t)T <= h->cap_frames) return JB200_OK;
  cudaFree(h->d_feats); cudaFree(h->d_rows); h->d_feats = h->d_rows = nullptr; h->cap_frames = 0;
  JB_CUDA(cudaMalloc(&h->d_feats, (size_t)T * h->D * sizeof(float)));
  JB_CUDA(cudaMalloc(&h->d_rows, (size_t)T * h->row_stride * sizeof(float)));
  h->cap_frames = T;
  return JB200_OK;
}

extern "C" int jb200_gmm_score_rows_host(jb200_gmm *h, const float *feats, int T, float *rows) {
  if (!h || !feats || !rows) { set_error("jb200_gmm_score_rows_host: null argument"); return JB200_ERR_ARG; }
  if (T <= 0) return JB200_OK;
  JB_CUDA(cudaSetDevice(h->device));
  int rc = ensure_scratch(h, T); if (rc) return rc;
  JB_CUDA(cudaMemcpyAsync(h->d_feats, feats, (size_t)T * h->D * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  rc = jb200_gmm_score_device(h, h->d_feats, T, h->d_rows, h->stream); if (rc) return rc;
  JB_CUDA(cudaMemcpyAsync(rows, h->d_rows, (size_t)T * h->row_stride * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  JB_CUDA(cudaStreamSynchronize(h->stream));
  return JB200_OK;
}

extern "C" int jb200_gmm_score_host(jb200_gmm *h, const float *feats, int T, float *scores) {
  if (!h || !feats || !scores) { set_error("jb200_gmm_score_host: null argument"); return JB200_ERR_ARG; }
  if (T <= 0) return JB200_OK;
  JB_CUDA(cudaSetDevice(h->device));
  int rc = ensure_scratch(h, T); if (rc) return rc;
  JB_CUDA(cudaMemcpyAsync(h->d_feats, feats, (size_t)T * h->D * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  rc = jb200_gmm_score_device(h, h->d_feats, T, h->d_rows, h->stream); if (rc) return rc;
  JB_CUDA(cudaMemcpy2DAsync(scores, (size_t)h->S * sizeof(float), h->d_rows, (size_t)h->row_stride * sizeof(float),
                            (size_t)h->S * sizeof(float), T, cudaMemcpyDeviceToHost, h->stream));
  JB_CUDA(cudaStreamSynchronize(h->stream));
  return JB200_OK;
}

extern "C" int jb200_gmm_gauss_host(jb200_gmm *h, const float *feat, float *gauss) {
  if (!h || !feat || !gauss) { set_error("jb200_gmm_gauss_host: null argument"); return JB200_ERR_ARG; }
  JB_CUDA(cudaSetDevice(h->device));
  float *d_f = nullptr, *d_o = nullptr;
  JB_CUDA(cudaMalloc(&d_f, sizeof(float) * h->D));
  JB_CUDA(cudaMalloc(&d_o, sizeof(float) * (h->G + 1)));
  JB_CUDA(cudaMemcpyAsync(d_f, feat, sizeof(float) * h->D, cudaMemcpyHostToDevice, h->stream));
  gauss_frame_kernel<<<(h->G + 255) / 256, 256, 0, h->stream>>>(h->d_pk, h->stride, h->D, h->G, d_f, d_o);
  JB_LAUNCH_CHECK();
  JB_CUDA(cudaMemcpyAsync(gauss, d_o, sizeof(float) * h->G, cudaMemcpyDeviceToHost, h->stream));
  JB_CUDA(cudaStreamSynchronize(h->stream));
  cudaFree(d_f); cudaFree(d_o);
  return JB200_OK;
}
