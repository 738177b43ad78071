// Per-scan feature covariance of a sparse tensor's N x C feature matrix, forward and backward: the statistic of
// RobustNet's instance-selective whitening (ISW) loss, one of the normalisation baselines next to LiDOG (SURVEY.md
// 2.2).  Scan b = the rows whose batch index (coordinate column 0) is b; rows need not be sorted by batch.
//
//   cov_b = X_b^T X_b / (n_b - 1) + eps * I        (X_b not centred; n_b <= 1: cov_b = eps * I)
//   dx_r  = x_r S_b(r),  S_b = (G_b + G_b^T) / (n_b - 1)   (n_b <= 1: S_b = 0)
//
// Forward, five launches:
//   k_cov_rank<false>   per (row chunk, scan) row counts                    hist [B][n_h]
//   k_scan_partials     exclusive scan of hist in (scan, chunk) order       -> where each chunk's rows of b go
//   k_cov_rank<true>    stable scatter of the row ids, grouped by scan     perm [n_valid]
//   k_cov_gram          per (position chunk, upper C x C tile): Gram sums of the chunk's rows, one partial per
//                       (chunk, scan) segment, float over 32 rows then double
//   k_cov_tail          fixed-order double sum of a scan's partials, scale, eps, mirror -> cov [B][C][C], counts [B]
// Backward, two launches: k_cov_bwd_s forms S_b once per scan; k_cov_bwd_apply is one pass over rows.
// Integer atomics only (shared-memory row counts); every float result is bit-identical run to run.
// Work: forward C(C+1)/2 FMA per row (plus the lower halves of the diagonal tiles), backward C^2.  Measured on a B200
// (DESIGN.md 4.7): the forward reaches at most 6 % of either the HBM or the FP32 bound (latency: the grouping passes and
// 32-row slabs of a few hundred blocks); the backward 20-27 % of the FP32 bound and less of the HBM bound.
#include <climits>

#include "common.cuh"
#include "runtime.cuh"
#include "scan.cuh"

namespace lg {

constexpr int kCovMaxB = 256;      // scans per call (LG_ERR_UNSUPPORTED above)
constexpr int kCovMaxC = 256;      // channels (LG_ERR_UNSUPPORTED above)
constexpr int kCovRankWarps = 4;   // row chunks per rank block, one warp each
constexpr int kCovRankRows = 512;  // rows per rank chunk (more when (scan, chunk) counts would pass kCovHistMax)
constexpr int kCovHistMax = 16384;
constexpr int kCovSlab = 32;       // rows staged in shared memory per step; float sums over a slab, double across
constexpr int kCovThreads = 256;
constexpr int kCovTargetBlocks = 148 * 4;

// ------------------------------------------------------------------ grouping rows by scan

// One warp per chunk of H rows, in row order.  Counting pass: hist[b * n_h + k] = rows of scan b in chunk k.
// Scatter pass (hist scanned): the rows of scan b in chunk k go to perm[hist[b * n_h + k] ...] in row order, so
// perm lists every valid row grouped by scan, rows of a scan in ascending order.  Rows outside [0, B) are left out.
template <bool SCATTER>
__global__ void __launch_bounds__(32 * kCovRankWarps)
    k_cov_rank(const int32_t* __restrict__ coords, int64_t n, int B, int64_t H, int n_h, int* __restrict__ hist,
               int* __restrict__ perm) {
  __shared__ int s_cnt[kCovRankWarps][kCovMaxB];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int k = blockIdx.x * kCovRankWarps + w;
  if (k >= n_h) return;  // warp-uniform; the kernel has no block barrier
  int* cnt = s_cnt[w];
  for (int b = lane; b < B; b += 32) cnt[b] = SCATTER ? hist[(int64_t)b * n_h + k] : 0;
  __syncwarp();
  const int64_t r0 = (int64_t)k * H, r1 = min(n, r0 + H);
  const unsigned lt = (1u << lane) - 1u;
  for (int64_t g0 = r0; g0 < r1; g0 += 4 * 32) {
    int bv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t r = g0 + u * 32 + lane;
      bv[u] = r < r1 ? __ldg(coords + r * 4) : -1;
      if ((unsigned)bv[u] >= (unsigned)B) bv[u] = -1;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int b = bv[u];
      const unsigned same = __match_any_sync(0xffffffffu, b);
      const int rank = __popc(same & lt);
      if (SCATTER && b >= 0) perm[cnt[b] + rank] = (int)(g0 + u * 32 + lane);
      __syncwarp();
      if (b >= 0 && rank == 0) cnt[b] += __popc(same);
      __syncwarp();
    }
  }
  if (!SCATTER)
    for (int b = lane; b < B; b += 32) hist[(int64_t)b * n_h + k] = cnt[b];
}

// Segment table of the scan-grouped order: start[b] = first position of scan b (start[B] = valid rows), and
// slot(k, b) = k + inner[b] numbers the (position chunk k, scan b) segments consecutively, with
// inner[b] = #{b' <= b : n_b' > 0, start[b'] % R != 0} (a scan that begins inside a chunk opens one more segment).
struct CovSeg {
  int start[kCovMaxB + 1];
  int inner[kCovMaxB];
};

__device__ void cov_seg_load(CovSeg& s, const int* __restrict__ hist, const int64_t* __restrict__ total, int n_h,
                             int B, int64_t R) {
  for (int b = threadIdx.x; b < B; b += blockDim.x) s.start[b] = hist[(int64_t)b * n_h];
  if (threadIdx.x == 0) s.start[B] = (int)*total;
  __syncthreads();
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    int carry = 0;
    for (int b0 = 0; b0 < B; b0 += 32) {
      const int b = b0 + lane;
      const bool f = b < B && s.start[b + 1] > s.start[b] && s.start[b] % R != 0;
      const unsigned m = __ballot_sync(0xffffffffu, f);
      if (b < B) s.inner[b] = carry + __popc(m & ((2u << lane) - 1u));
      carry += __popc(m);
    }
  }
  __syncthreads();
}

// ------------------------------------------------------------------ forward: Gram partials and tail

__device__ __forceinline__ void upper_tile(int t, int nt, int& ti, int& tj) {
  ti = 0;
  while (t >= nt - ti) t -= nt - ti, ++ti;
  tj = ti + t;
}

// Stages rows [p, p + kCovSlab) of the grouped order (clipped at `end`), columns c0 .. c0 + T, of x into dst[slab][T]
// (zeros outside).  V = 4: float4 loads (C % 4 == 0).
template <int T, int V>
struct CovStage {
  static constexpr int kPer = (kCovSlab * T / V + kCovThreads - 1) / kCovThreads;
  float v[kPer][V];
  __device__ __forceinline__ void load(const float* __restrict__ x, const int* __restrict__ perm, int64_t p,
                                       int64_t end, int C, int c0) {
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
      const int idx = q * kCovThreads + threadIdx.x;
      const int row = idx / (T / V), col = c0 + (idx % (T / V)) * V;
#pragma unroll
      for (int j = 0; j < V; ++j) v[q][j] = 0.f;
      if (idx < kCovSlab * T / V && p + row < end && col < C) {
        const int64_t r = __ldg(perm + p + row);
        if constexpr (V == 4) {
          const float4 f = __ldg(reinterpret_cast<const float4*>(x + r * C + col));
          v[q][0] = f.x, v[q][1] = f.y, v[q][2] = f.z, v[q][3] = f.w;
        } else {
          v[q][0] = __ldg(x + r * C + col);
        }
      }
    }
  }
  __device__ __forceinline__ void store(float* dst) const {
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
      const int idx = q * kCovThreads + threadIdx.x;
      if (idx < kCovSlab * T / V)
#pragma unroll
        for (int j = 0; j < V; ++j) dst[idx * V + j] = v[q][j];
    }
  }
};

// grid (n_pc, n_tiles), block 256.  Block (k, t) owns positions [k R, k R + R) of the grouped order and the upper
// tile t = (ti, tj) of T x T channels.  Threads form G = 256 / (T/4)^2 groups; a thread's 4 x 4 outputs are
// rows ti*T + 4 ty + u, columns tj*T + 4 tx + v; group g takes rows g, g + G, ... of each slab.  Per segment
// (rows of one scan inside the chunk) the groups' double sums are added in group order and written to
//   part[(slot(k, b) * n_tiles + t) * T * T + i * T + j]   (double, the whole tile).
template <int T, int V>
__global__ void __launch_bounds__(kCovThreads)
    k_cov_gram(const float* __restrict__ x, const int* __restrict__ perm, const int* __restrict__ hist,
               const int64_t* __restrict__ total, int n_h, int C, int B, int64_t R, int nt,
               int* __restrict__ segtab, double* __restrict__ part) {
  constexpr int TPG = (T / 4) * (T / 4), G = kCovThreads / TPG;
  __shared__ CovSeg seg;
  __shared__ __align__(16) float sa[kCovSlab * T];
  __shared__ __align__(16) float sb[kCovSlab * T];
  __shared__ double red[G > 1 ? TPG * 16 : 1];  // group sums in flight (T = 32: four groups)
  cov_seg_load(seg, hist, total, n_h, B, R);
  if (blockIdx.x == 0 && blockIdx.y == 0) {  // the tail reads the table from here
    for (int b = threadIdx.x; b <= B; b += blockDim.x) segtab[b] = seg.start[b];
    for (int b = threadIdx.x; b < B; b += blockDim.x) segtab[B + 1 + b] = seg.inner[b];
  }
  const int64_t k = blockIdx.x, p0 = k * R, p1 = min((int64_t)seg.start[B], p0 + R);
  if (p0 >= p1) return;  // block-uniform
  int ti, tj;
  upper_tile(blockIdx.y, nt, ti, tj);
  const bool diag = ti == tj;
  const int n_tiles = nt * (nt + 1) / 2;
  const int g = threadIdx.x / TPG, q = threadIdx.x % TPG, ty = q / (T / 4), tx = q % (T / 4);
  const float* sbr = diag ? sa : sb;
  int64_t p = p0;
  while (p < p1) {
    int lo = 0, hi = B;  // the scan of position p: start[b] <= p < start[b + 1]
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (seg.start[mid] <= p) lo = mid; else hi = mid;
    }
    const int b = lo;
    const int64_t end = min(p1, (int64_t)seg.start[b + 1]);
    double dacc[4][4] = {};
    CovStage<T, V> ra, rb;
    ra.load(x, perm, p, end, C, ti * T);
    if (!diag) rb.load(x, perm, p, end, C, tj * T);
    for (int64_t s = p; s < end; s += kCovSlab) {
      __syncthreads();  // the previous slab (or segment) is consumed
      ra.store(sa);
      if (!diag) rb.store(sb);
      __syncthreads();
      if (s + kCovSlab < end) {  // next slab in flight during the FMAs
        ra.load(x, perm, s + kCovSlab, end, C, ti * T);
        if (!diag) rb.load(x, perm, s + kCovSlab, end, C, tj * T);
      }
      float acc[4][4] = {};
#pragma unroll 4
      for (int kk = g; kk < kCovSlab; kk += G) {
        const float4 a = *reinterpret_cast<const float4*>(sa + kk * T + 4 * ty);
        const float4 c = *reinterpret_cast<const float4*>(sbr + kk * T + 4 * tx);
        const float av[4] = {a.x, a.y, a.z, a.w}, cv[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < 4; ++v) acc[u][v] = fmaf(av[u], cv[v], acc[u][v]);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) dacc[u][v] += (double)acc[u][v];
    }
    const int64_t slot = k + seg.inner[b];
    double* out = part + (slot * n_tiles + blockIdx.y) * (int64_t)(T * T);
    for (int gg = 0; gg < G; ++gg) {  // groups in order: red = ((g0 + g1) + g2) + ...
      if (g == gg) {
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            const double d = gg == 0 ? dacc[u][v] : red[q * 16 + u * 4 + v] + dacc[u][v];
            if (gg == G - 1) out[(4 * ty + u) * T + 4 * tx + v] = d;
            else red[q * 16 + u * 4 + v] = d;
          }
      }
      if (G > 1) __syncthreads();
    }
    p = end;
  }
}

// grid (n_tiles, B), block 256.  Element (i, j), i <= j, of tile t for scan b: the partials of b's segments in chunk
// order, summed in double, / (n_b - 1), + eps on the diagonal; written to cov[b][i][j] and cov[b][j][i].
template <int T>
__global__ void __launch_bounds__(kCovThreads)
    k_cov_tail(const double* __restrict__ part, const int* __restrict__ segtab, int C, int B, int64_t R, int nt,
               float eps, float* __restrict__ cov, int* __restrict__ counts) {
  const int b = blockIdx.y;
  const int n_tiles = nt * (nt + 1) / 2;
  int ti, tj;
  upper_tile(blockIdx.x, nt, ti, tj);
  const int64_t st = segtab[b], nb = segtab[b + 1] - st;
  const int inner = segtab[B + 1 + b];
  if (blockIdx.x == 0 && threadIdx.x == 0) counts[b] = (int)nb;
  const int64_t kf = st / R, kl = nb > 0 ? (st + nb - 1) / R : kf - 1;
  float* cb = cov + (int64_t)b * C * C;
  for (int e = threadIdx.x; e < T * T; e += blockDim.x) {
    const int i = ti * T + e / T, j = tj * T + e % T;
    if (i >= C || j >= C || i > j) continue;
    double s = 0.0;
    if (nb > 1) {
      for (int64_t kk = kf; kk <= kl; ++kk) s += __ldg(part + ((kk + inner) * n_tiles + blockIdx.x) * (int64_t)(T * T) + e);
      s /= (double)(nb - 1);
    }
    if (i == j) s += (double)eps;
    cb[(int64_t)i * C + j] = (float)s;
    if (i != j) cb[(int64_t)j * C + i] = (float)s;
  }
}

// ------------------------------------------------------------------ backward

// grid (ceil(C*C / 256), B): S[b][i][j] = (G[b][i][j] + G[b][j][i]) / (n_b - 1), 0 when n_b <= 1.
__global__ void __launch_bounds__(256)
    k_cov_bwd_s(const float* __restrict__ G, const int* __restrict__ counts, int C, float* __restrict__ S) {
  const int b = blockIdx.y;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, CC = (int64_t)C * C;
  if (e >= CC) return;
  const int i = (int)(e / C), j = (int)(e % C);
  const int nb = __ldg(counts + b);
  const float* g = G + b * CC;
  S[b * CC + e] = nb > 1 ? (float)(((double)__ldg(g + e) + (double)__ldg(g + (int64_t)j * C + i)) / (double)(nb - 1)) : 0.f;
}

// grid (ceil(n / RT), ceil(C / JT)), block 256, RT = 4096 / JT rows.  Thread (ty, tx) computes rows r0 + 4 ty + u,
// columns j0 + 4 tx + v: dx = sum_i x[r][i] S_b[i][j], i ascending, one fmaf chain in float.  A block whose rows
// span several scans runs once per scan present (ascending), each time with S of that scan, and keeps the result of
// the rows of that scan: a row's arithmetic does not depend on its neighbours.  Rows outside [0, B): NaN.
template <int JT, int V>
__global__ void __launch_bounds__(256)
    k_cov_bwd_apply(const float* __restrict__ x, const int32_t* __restrict__ coords, const float* __restrict__ S,
                    int64_t n, int C, int B, float* __restrict__ dx) {
  constexpr int RT = 4096 / JT, KI = 32, TX = JT / 4;
  __shared__ float xs[KI][RT + 1];  // x transposed: xs[i][row]
  __shared__ __align__(16) float ss[KI][JT];
  __shared__ int s_b[RT];
  __shared__ int s_next;
  const int tx = threadIdx.x % TX, ty = threadIdx.x / TX;
  const int64_t r0 = (int64_t)blockIdx.x * RT;
  const int j0 = blockIdx.y * JT;
  for (int rr = threadIdx.x; rr < RT; rr += blockDim.x) {
    const int64_t r = r0 + rr;
    int b = r < n ? __ldg(coords + r * 4) : -1;
    s_b[rr] = (unsigned)b < (unsigned)B ? b : -1;
  }
  __syncthreads();
  int rb[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) rb[u] = s_b[4 * ty + u];
  float out[4][4];
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) out[u][v] = __int_as_float(0x7fffffff);
  int cur = -1;
  for (;;) {
    if (threadIdx.x == 0) s_next = INT_MAX;
    __syncthreads();
    for (int rr = threadIdx.x; rr < RT; rr += blockDim.x)
      if (s_b[rr] > cur) atomicMin(&s_next, s_b[rr]);
    __syncthreads();
    const int b = s_next;
    __syncthreads();  // s_next is re-armed at the top of the next pass
    if (b == INT_MAX) break;
    cur = b;
    const float* Sb = S + (int64_t)b * C * C;
    float acc[4][4] = {};
    for (int i0 = 0; i0 < C; i0 += KI) {
      for (int idx = threadIdx.x; idx < RT * KI / V; idx += blockDim.x) {  // x rows of scan b, columns i0 ..
        const int rr = idx / (KI / V), ii = (idx % (KI / V)) * V;
        const int64_t r = r0 + rr;
        float f[V] = {};
        if (s_b[rr] == b && i0 + ii < C) {
          if constexpr (V == 4) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(x + r * C + i0 + ii));
            f[0] = t.x, f[1] = t.y, f[2] = t.z, f[3] = t.w;
          } else {
            f[0] = __ldg(x + r * C + i0 + ii);
          }
        }
#pragma unroll
        for (int j = 0; j < V; ++j) xs[ii + j][rr] = f[j];
      }
      for (int idx = threadIdx.x; idx < KI * JT / V; idx += blockDim.x) {  // S_b rows i0 .., columns j0 ..
        const int ii = idx / (JT / V), jj = (idx % (JT / V)) * V;
        float f[V] = {};
        if (i0 + ii < C && j0 + jj < C) {
          if constexpr (V == 4) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(Sb + (int64_t)(i0 + ii) * C + j0 + jj));
            f[0] = t.x, f[1] = t.y, f[2] = t.z, f[3] = t.w;
          } else {
            f[0] = __ldg(Sb + (int64_t)(i0 + ii) * C + j0 + jj);
          }
        }
#pragma unroll
        for (int j = 0; j < V; ++j) ss[ii][jj + j] = f[j];
      }
      __syncthreads();
      const int kmax = min(KI, C - i0);
      for (int kk = 0; kk < kmax; ++kk) {
        const float4 s4 = *reinterpret_cast<const float4*>(&ss[kk][4 * tx]);
        const float sv[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float a = xs[kk][4 * ty + u];
#pragma unroll
          for (int v = 0; v < 4; ++v) acc[u][v] = fmaf(a, sv[v], acc[u][v]);
        }
      }
      __syncthreads();
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (rb[u] == b)
#pragma unroll
        for (int v = 0; v < 4; ++v) out[u][v] = acc[u][v];
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int64_t r = r0 + 4 * ty + u;
    const int j = j0 + 4 * tx;
    if (r >= n || j >= C) continue;
    if constexpr (V == 4) {
      *reinterpret_cast<float4*>(dx + r * C + j) = make_float4(out[u][0], out[u][1], out[u][2], out[u][3]);
    } else {
#pragma unroll
      for (int v = 0; v < 4; ++v)
        if (j + v < C) dx[r * C + j + v] = out[u][v];
    }
  }
}

// ------------------------------------------------------------------ host

struct CovPlan {
  int T, nt, n_tiles, n_h, n_pc;
  int64_t H, R;
  size_t hist_bytes, perm_bytes, seg_bytes, part_bytes;
};

static CovPlan cov_plan(int64_t n, int C, int B) {
  CovPlan p;
  p.T = C <= 32 ? 32 : 64;
  p.nt = (int)ceil_div(C, p.T);
  p.n_tiles = p.nt * (p.nt + 1) / 2;
  int64_t nh = ceil_div(n, kCovRankRows);
  const int64_t cap = kCovHistMax / B;
  if (nh > cap) nh = cap;
  if (nh < 1) nh = 1;
  p.H = n > 0 ? ceil_div(n, nh) : 1;
  p.n_h = n > 0 ? (int)ceil_div(n, p.H) : 1;
  int64_t pc = ceil_div(kCovTargetBlocks, p.n_tiles);
  const int64_t by_rows = ceil_div(n, 256);  // at least 256 positions (8 slabs) per block
  if (pc > by_rows) pc = by_rows;
  if (pc < 1) pc = 1;
  p.R = n > 0 ? round_up(ceil_div(n, pc), kCovSlab) : kCovSlab;
  p.n_pc = n > 0 ? (int)ceil_div(n, p.R) : 1;
  p.hist_bytes = sizeof(int) * (size_t)B * p.n_h;
  p.perm_bytes = sizeof(int) * (size_t)(n > 0 ? n : 1);
  p.seg_bytes = sizeof(int) * (size_t)(2 * B + 1);
  // segments: one per position chunk, plus one per scan that begins inside a chunk
  p.part_bytes = sizeof(double) * (size_t)(p.n_pc + B) * p.n_tiles * p.T * p.T;
  return p;
}

static int cov_check(const char* who, const float* x, const int32_t* coords, int64_t n, int C, int B,
                     const void* cov_or_g, const int32_t* counts, const float* dx) {
  LG_CHECK_ARG(n >= 0 && C >= 1 && B >= 1, "%s: needs n >= 0, C >= 1, B >= 1", who);
  LG_CHECK_ARG(n < INT_MAX, "%s: n = %lld rows, fewer than 2^31 - 1 are supported", who, (long long)n);
  LG_CHECK_ARG(x && coords && cov_or_g && counts, "%s: null pointer", who);
  const uintptr_t a = C % 4 == 0 ? 15 : 3;
  LG_CHECK_ARG(((uintptr_t)x & a) == 0 && ((uintptr_t)dx & a) == 0 && ((uintptr_t)coords & 3) == 0 &&
                   ((uintptr_t)cov_or_g & 3) == 0 && ((uintptr_t)counts & 3) == 0,
               "%s: misaligned pointer (features need 16 bytes when C %% 4 == 0, else 4)", who);
  if (B > kCovMaxB || C > kCovMaxC) {
    set_error("%s: B = %d scans, C = %d channels; at most %d and %d are supported", who, B, C, kCovMaxB, kCovMaxC);
    return LG_ERR_UNSUPPORTED;
  }
  return LG_OK;
}

template <int T, int V>
static int cov_launch_gram(const CovPlan& p, const float* x, const int* perm, const int* hist, const int64_t* total,
                           int C, int B, int* segtab, double* part, float eps, float* cov, int* counts,
                           cudaStream_t stream) {
  k_cov_gram<T, V><<<dim3((unsigned)p.n_pc, (unsigned)p.n_tiles), kCovThreads, 0, stream>>>(
      x, perm, hist, total, p.n_h, C, B, p.R, p.nt, segtab, part);
  LG_LAUNCH_OK();
  k_cov_tail<T><<<dim3((unsigned)p.n_tiles, (unsigned)B), kCovThreads, 0, stream>>>(part, segtab, C, B, p.R, p.nt, eps,
                                                                                  cov, counts);
  LG_LAUNCH_OK();
  return LG_OK;
}

}  // namespace lg

using namespace lg;

extern "C" int lg_inst_cov_forward(const float* x, const int32_t* coords, int64_t n, int32_t C, int32_t B, float eps,
                                   float* cov, int32_t* counts, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = cov_check("lg_inst_cov_forward", x, coords, n, C, B, cov, counts, nullptr);
  if (rc) return rc;
  LG_CHECK_ARG(eps >= 0.f, "lg_inst_cov_forward: eps must be >= 0");
  const CovPlan p = cov_plan(n, C, B);
  ArenaCursor ar;
  rc = arena_begin(stream,
                   arena_pad(p.hist_bytes) + arena_pad(sizeof(int64_t)) + arena_pad(p.perm_bytes) +
                       arena_pad(p.seg_bytes) + arena_pad(p.part_bytes),
                   &ar);
  if (rc) return rc;
  int* hist = (int*)arena_take(&ar, p.hist_bytes);
  int64_t* total = (int64_t*)arena_take(&ar, sizeof(int64_t));
  int* perm = (int*)arena_take(&ar, p.perm_bytes);
  int* segtab = (int*)arena_take(&ar, p.seg_bytes);
  double* part = (double*)arena_take(&ar, p.part_bytes);
  // n = 0 runs too (one empty chunk): every scan gets eps * I and a count of 0
  const unsigned rank_blocks = (unsigned)ceil_div(p.n_h, kCovRankWarps);
  k_cov_rank<false><<<rank_blocks, 32 * kCovRankWarps, 0, stream>>>(coords, n, B, p.H, p.n_h, hist, nullptr);
  LG_LAUNCH_OK();
  k_scan_partials<<<1, 1024, 0, stream>>>(hist, B * p.n_h, total);
  LG_LAUNCH_OK();
  k_cov_rank<true><<<rank_blocks, 32 * kCovRankWarps, 0, stream>>>(coords, n, B, p.H, p.n_h, hist, perm);
  LG_LAUNCH_OK();
  const bool v4 = C % 4 == 0;
  if (p.T == 32)
    return v4 ? cov_launch_gram<32, 4>(p, x, perm, hist, total, C, B, segtab, part, eps, cov, counts, stream)
              : cov_launch_gram<32, 1>(p, x, perm, hist, total, C, B, segtab, part, eps, cov, counts, stream);
  return v4 ? cov_launch_gram<64, 4>(p, x, perm, hist, total, C, B, segtab, part, eps, cov, counts, stream)
            : cov_launch_gram<64, 1>(p, x, perm, hist, total, C, B, segtab, part, eps, cov, counts, stream);
}

extern "C" int lg_inst_cov_backward(const float* x, const int32_t* coords, int64_t n, int32_t C, int32_t B,
                                    const float* G, const int32_t* counts, float* dx, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = cov_check("lg_inst_cov_backward", x, coords, n, C, B, G, counts, dx);
  if (rc) return rc;
  LG_CHECK_ARG(dx, "lg_inst_cov_backward: null pointer");
  if (n == 0) return LG_OK;
  const size_t s_bytes = sizeof(float) * (size_t)B * C * C;
  ArenaCursor ar;
  rc = arena_begin(stream, arena_pad(s_bytes), &ar);
  if (rc) return rc;
  float* S = (float*)arena_take(&ar, s_bytes);
  k_cov_bwd_s<<<dim3((unsigned)ceil_div((int64_t)C * C, 256), (unsigned)B), 256, 0, stream>>>(G, counts, C, S);
  LG_LAUNCH_OK();
  const bool v4 = C % 4 == 0;
  if (C <= 32) {
    const dim3 grid((unsigned)ceil_div(n, 128), 1);
    if (v4) k_cov_bwd_apply<32, 4><<<grid, 256, 0, stream>>>(x, coords, S, n, C, B, dx);
    else k_cov_bwd_apply<32, 1><<<grid, 256, 0, stream>>>(x, coords, S, n, C, B, dx);
  } else {
    const dim3 grid((unsigned)ceil_div(n, 64), (unsigned)ceil_div(C, 64));
    if (v4) k_cov_bwd_apply<64, 4><<<grid, 256, 0, stream>>>(x, coords, S, n, C, B, dx);
    else k_cov_bwd_apply<64, 1><<<grid, 256, 0, stream>>>(x, coords, S, n, C, B, dx);
  }
  LG_LAUNCH_OK();
  return LG_OK;
}
