// Instance normalisation of a sparse tensor's N x C feature matrix, per (scan, channel), with an optional ReLU:
// ME.MinkowskiInstanceNorm as the domain-generalisation baselines next to LiDOG use it (IBN-Net, RobustNet;
// SURVEY.md 2, Appendix C).  Instance b = the rows whose batch index (coordinate column 0) is b; rows need not be
// sorted by batch.
//
//   y = ((x - mean_b) * (var_b + eps)^-1/2) * weight + bias     (biased variance over the rows of instance b)
//
// Three passes each way, modelled on bn.cu (statistics / tail / apply):
//   forward   k_in_stats<true>   per-(chunk, instance, channel) count, mean, M2                (read x, coords)
//             k_in_tail<true>    Chan merge of the chunks in a fixed order, in double -> mean, invstd [B][C]
//             k_in_apply         y = act(xhat * weight + bias) -> fp32 y and the 16-bit operand copy
//   backward  k_in_stats<false>  g = dy * [y > 0]; per-(chunk, instance, channel) sum g, sum g * xhat
//             k_in_tail<false>   fixed-order sums -> dx coefficients; the last block adds dweight, dbias over b
//             k_in_bwd_apply     dx = invstd * weight * (g - mean_b(g) - xhat * mean_b(g * xhat))
// No atomics on data, no reduction whose order depends on scheduling: every output is bit-identical run to run.
// Bound: HBM.  Algorithmic bytes per element: forward 4 (stats) + 4+4+2 (apply), backward 12 + 12+4; plus 4 bytes of
// batch index per row and pass.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "runtime.cuh"

namespace lg {

constexpr int kInMaxB = 256;          // instances per call (LG_ERR_UNSUPPORTED above)
constexpr int kInTile = 32;           // columns per warp: lane = column
constexpr int kInMaxWarps = 8;        // warps per statistics block; they split the block's rows
constexpr int kInSmemMax = 112 << 10;  // statistics block shared memory: two blocks per SM even at B = 256
constexpr int kInUnroll = 8;          // rows whose loads are in flight per warp
constexpr int kInTargetWarps = 148 * 48;
constexpr int kInMinRowsPerWarp = 64;
constexpr int kInTailY = 32;          // chunk slices per tail block

// bn_to16's rounding (bn.cu): equal to what lg_cast_rows makes of the fp32 value
__device__ __forceinline__ unsigned short in_to16(float v, int fmt) {
  if (fmt == LG_FMT_BF16) return __bfloat16_as_ushort(__float2bfloat16_rn(v));
  v = fminf(fmaxf(v, -65504.f), 65504.f);
  return __half_as_ushort(__float2half_rn(v));
}

// x - mean with the double mean split in two floats: x - hi is exact near the mean (Sterbenz), so a feature with a
// large mean and a small spread keeps its precision; xhat = that * invstd.  The backward recomputes it identically.
__device__ __forceinline__ float in_xhat(float x, const double* __restrict__ st, int64_t i, int64_t BC) {
  const double m = __ldg(st + i);
  const float hi = (float)m, lo = (float)(m - (double)hi);
  return ((x - hi) - lo) * (float)__ldg(st + BC + i);
}

__device__ __forceinline__ bool in_batch_ok(int b, int B) { return (unsigned)b < (unsigned)B; }

// Running (count, acc0, acc1) of one (instance, column), folded with a part (nb, p0, p1) of nb > 0 rows.
// Forward: acc = (mean, M2), Chan's parallel update.  Backward: acc = (sum g, sum g * xhat), plain sums.
template <bool FWD>
__device__ __forceinline__ void in_fold(double& n, double& a0, double& a1, double nb, double p0, double p1) {
  if (nb == 0.0) return;
  if (FWD) {
    const double tot = n + nb, d = p0 - a0;
    a0 += d * (nb / tot);
    a1 += p1 + d * d * (n * nb / tot);
    n = tot;
  } else {
    n += nb, a0 += p0, a1 += p1;
  }
}

// Shared memory of one warp: cnt[B] (int), then NACC floats per (instance, lane): [NACC][B][32].
template <bool FWD>
struct InSlab {
  static constexpr int kAcc = FWD ? 3 : 2;  // forward: shift K, sum (x - K), sum (x - K)^2; backward: sum g, sum g*xhat
  static __host__ __device__ size_t bytes(int B) { return ((size_t)B * 4 + (size_t)kAcc * B * kInTile * 4 + 15) & ~(size_t)15; }
};

// grid (n_chunks, n_ctiles), block 32 x W.  Block (chunk, ct) owns rows [chunk * per, ...) and columns ct*32 + lane;
// warp w walks its own contiguous sub-range in row order, so each (instance, column) accumulator has one owner.
// The block then merges its W warps in warp order (double) and writes the partial row
//   part[chunk][b] = [count | acc0 (C) | acc1 (C)]   (double)
// forward acc0 / acc1 = mean / M2 of the chunk's rows of instance b; backward = sum g / sum g * xhat.
// The forward accumulates x - K with K = the first value of that (instance, column) the warp meets, so the float
// sums never carry the mean itself.
template <bool FWD>
__global__ void __launch_bounds__(kInTile* kInMaxWarps)
    k_in_stats(const float* __restrict__ x, const float* __restrict__ dy, const float* __restrict__ y,
               const double* __restrict__ st, const int32_t* __restrict__ coords, int64_t n, int C, int B, int relu,
               int64_t rows_per_chunk, double* __restrict__ part) {
  extern __shared__ __align__(16) unsigned char in_smem[];
  const int lane = threadIdx.x, w = threadIdx.y, W = blockDim.y;
  const size_t slab = InSlab<FWD>::bytes(B);
  int* cnt = reinterpret_cast<int*>(in_smem + slab * w);
  float* acc = reinterpret_cast<float*>(in_smem + slab * w + (size_t)B * 4);
  const int c = blockIdx.y * kInTile + lane;
  const bool col = c < C;
  const int64_t BC = (int64_t)B * C;
  for (int b = lane; b < B; b += kInTile) cnt[b] = 0;
  for (int b = 0; b < B; ++b) {
    acc[b * kInTile + lane] = FWD ? __int_as_float(0x7fffffff) : 0.f;  // forward: K unset (NaN)
    acc[(B + b) * kInTile + lane] = 0.f;
    if (FWD) acc[(2 * B + b) * kInTile + lane] = 0.f;
  }
  __syncwarp();
  const int64_t c0 = (int64_t)blockIdx.x * rows_per_chunk, c1 = min(n, c0 + rows_per_chunk);
  const int64_t per = (c1 - c0 + W - 1) / W;
  const int64_t r0 = min(c1, c0 + per * w), r1 = min(c1, r0 + per);
  for (int64_t g0 = r0; g0 < r1; g0 += kInTile) {
    const int64_t rl = g0 + lane;
    const int bl = rl < r1 ? __ldg(coords + rl * 4) : -1;  // one batch index per lane, broadcast by shuffles
    const int m = (int)min((int64_t)kInTile, r1 - g0);
    for (int t0 = 0; t0 < m; t0 += kInUnroll) {
      float v[kInUnroll], gv[kInUnroll];
#pragma unroll
      for (int u = 0; u < kInUnroll; ++u) {
        v[u] = 0.f, gv[u] = 0.f;
        const int64_t r = g0 + t0 + u;
        if (col && t0 + u < m) {
          v[u] = __ldg(x + r * C + c);
          if (!FWD) {
            gv[u] = __ldg(dy + r * C + c);
            if (relu && !(__ldg(y + r * C + c) > 0.f)) gv[u] = 0.f;
          }
        }
      }
#pragma unroll
      for (int u = 0; u < kInUnroll; ++u) {
        const int b = __shfl_sync(0xffffffffu, bl, (t0 + u) & (kInTile - 1));
        if (t0 + u >= m || !in_batch_ok(b, B)) continue;  // warp-uniform
        if (lane == 0) cnt[b] += 1;
        if (!col) continue;
        float* a = acc + b * kInTile + lane;
        if (FWD) {
          float k = a[0];
          if (k != k) a[0] = k = v[u];
          const float d = v[u] - k;
          a[B * kInTile] += d;
          a[2 * B * kInTile] = fmaf(d, d, a[2 * B * kInTile]);
        } else {
          const float xh = in_xhat(v[u], st, (int64_t)b * C + c, BC);
          a[0] += gv[u];
          a[B * kInTile] = fmaf(gv[u], xh, a[B * kInTile]);
        }
      }
    }
  }
  __syncthreads();
  // merge the W warps in warp order: thread t handles (b, lane) pairs t, t + 32W, ...
  const int64_t width = 1 + 2 * (int64_t)C;
  for (int i = w * kInTile + lane; i < B * kInTile; i += W * kInTile) {
    const int b = i / kInTile, l = i % kInTile, cc = blockIdx.y * kInTile + l;
    double nn = 0.0, a0 = 0.0, a1 = 0.0;
    for (int ww = 0; ww < W; ++ww) {
      const int* cw = reinterpret_cast<const int*>(in_smem + slab * ww);
      const float* aw = reinterpret_cast<const float*>(in_smem + slab * ww + (size_t)B * 4) + b * kInTile + l;
      const double nb = (double)cw[b];
      if (FWD && nb > 0.0) {  // this warp's (count, mean, M2) from its shifted sums
        const double s = aw[B * kInTile], ss = aw[2 * B * kInTile];
        in_fold<true>(nn, a0, a1, nb, (double)aw[0] + s / nb, fmax(ss - s * s / nb, 0.0));
      } else if (!FWD) {
        in_fold<false>(nn, a0, a1, nb, aw[0], aw[B * kInTile]);
      }
    }
    double* row = part + ((int64_t)blockIdx.x * B + b) * width;
    if (blockIdx.y == 0 && l == 0) row[0] = nn;
    if (cc < C) row[1 + cc] = a0, row[1 + C + cc] = a1;
  }
}

struct InBwdOut {
  float* coef;     // [2][B][C]: mean_b(g), mean_b(g * xhat) (per unit weight)
  double* sums;    // [2][B][C]: sum g, sum g * xhat
  float *dweight, *dbias;
  int* ticket;
};

// grid (n_ctiles, B), block 32 x kInTailY.  Thread (lane, ty) folds chunks ty, ty + 32, ... of instance blockIdx.y,
// column ct*32 + lane (4 partial rows in flight); row 0 then folds the 32 slices in order.
// Forward: stats [2][B][C] double = mean, invstd (0, 0 for an instance without rows: nothing reads them).
// Backward: coefficients; the block that finishes last sums dweight / dbias over the instances in order.
template <bool FWD>
__global__ void __launch_bounds__(kInTile* kInTailY)
    k_in_tail(const double* __restrict__ part, int n_chunks, int C, int B, float eps, double* __restrict__ st,
              InBwdOut bo) {
  __shared__ double sm[3][kInTailY][kInTile];
  __shared__ int s_last;
  const int lane = threadIdx.x, ty = threadIdx.y, b = blockIdx.y;
  const int c = blockIdx.x * kInTile + lane;
  const int64_t width = 1 + 2 * (int64_t)C;
  double nn = 0.0, a0 = 0.0, a1 = 0.0;
  if (c < C) {
    int p = ty;
    for (; p + 3 * kInTailY < n_chunks; p += 4 * kInTailY) {
      double r[4][3];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const double* row = part + ((int64_t)(p + u * kInTailY) * B + b) * width;
        r[u][0] = __ldg(row), r[u][1] = __ldg(row + 1 + c), r[u][2] = __ldg(row + 1 + C + c);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) in_fold<FWD>(nn, a0, a1, r[u][0], r[u][1], r[u][2]);
    }
    for (; p < n_chunks; p += kInTailY) {
      const double* row = part + ((int64_t)p * B + b) * width;
      in_fold<FWD>(nn, a0, a1, __ldg(row), __ldg(row + 1 + c), __ldg(row + 1 + C + c));
    }
  }
  sm[0][ty][lane] = nn, sm[1][ty][lane] = a0, sm[2][ty][lane] = a1;
  __syncthreads();
  const int64_t BC = (int64_t)B * C, i = (int64_t)b * C + c;
  if (ty == 0 && c < C) {
    nn = 0.0, a0 = 0.0, a1 = 0.0;
    for (int s = 0; s < kInTailY; ++s) in_fold<FWD>(nn, a0, a1, sm[0][s][lane], sm[1][s][lane], sm[2][s][lane]);
    if (FWD) {
      st[i] = nn > 0.0 ? a0 : 0.0;
      st[BC + i] = nn > 0.0 ? 1.0 / sqrt(a1 / nn + (double)eps) : 0.0;
    } else {
      bo.sums[i] = a0, bo.sums[BC + i] = a1;
      bo.coef[i] = nn > 0.0 ? (float)(a0 / nn) : 0.f;
      bo.coef[BC + i] = nn > 0.0 ? (float)(a1 / nn) : 0.f;
    }
  }
  if (FWD) return;
  __threadfence();
  __syncthreads();
  if (lane == 0 && ty == 0) {
    const int t = atomicAdd(bo.ticket, 1);
    s_last = (t == (int)(gridDim.x * gridDim.y) - 1);
    if (s_last) *bo.ticket = 0;  // the slot is zero again for the next launch that draws it
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int cc = ty * kInTile + lane; cc < C; cc += kInTile * kInTailY) {
    double sg = 0.0, sgx = 0.0;
    for (int bb = 0; bb < B; ++bb) sg += __ldcg(bo.sums + (int64_t)bb * C + cc), sgx += __ldcg(bo.sums + BC + (int64_t)bb * C + cc);
    bo.dbias[cc] = (float)sg;
    bo.dweight[cc] = (float)sgx;
  }
}

// One thread per V consecutive elements of a row (V = 4 when C % 4 == 0: float4 loads and stores).
template <int V>
struct InVec;
template <>
struct InVec<4> {
  using T = float4;
  static __device__ __forceinline__ float get(const T& v, int j) { return j == 0 ? v.x : j == 1 ? v.y : j == 2 ? v.z : v.w; }
  static __device__ __forceinline__ void set(T& v, int j, float f) {
    if (j == 0) v.x = f; else if (j == 1) v.y = f; else if (j == 2) v.z = f; else v.w = f;
  }
};
template <>
struct InVec<1> {
  using T = float;
  static __device__ __forceinline__ float get(const T& v, int) { return v; }
  static __device__ __forceinline__ void set(T& v, int, float f) { v = f; }
};

template <int V>
__global__ void __launch_bounds__(256)
    k_in_apply(const float* __restrict__ x, const int32_t* __restrict__ coords, const double* __restrict__ st,
               const float* __restrict__ weight, const float* __restrict__ bias, int relu, int64_t n, int C, int B,
               float* __restrict__ y, unsigned short* __restrict__ y16, int fmt) {
  using VT = typename InVec<V>::T;
  const int CV = C / V;
  const int64_t nv = n * CV;
  const int64_t BC = (int64_t)B * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / CV;
    const int c = (int)(i - r * CV) * V;
    const VT xv = __ldg(reinterpret_cast<const VT*>(x) + i);
    const int b = __ldg(coords + r * 4);
    VT o;
    unsigned short h[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float f = __int_as_float(0x7fffffff);  // a row outside [0, B): NaN, never a silent value
      if (in_batch_ok(b, B)) {
        f = fmaf(in_xhat(InVec<V>::get(xv, j), st, (int64_t)b * C + c + j, BC), __ldg(weight + c + j), __ldg(bias + c + j));
        if (relu) f = fmaxf(f, 0.f);
      }
      InVec<V>::set(o, j, f);
      h[j] = in_to16(f, fmt);
    }
    reinterpret_cast<VT*>(y)[i] = o;
    if (y16) {
      if constexpr (V == 4) {
        uint2 p;
        p.x = h[0] | ((unsigned)h[1] << 16);
        p.y = h[2] | ((unsigned)h[3] << 16);
        *reinterpret_cast<uint2*>(y16 + i * V) = p;
      } else {
        y16[i] = h[0];
      }
    }
  }
}

template <int V>
__global__ void __launch_bounds__(256)
    k_in_bwd_apply(const float* __restrict__ dy, const float* __restrict__ y, const float* __restrict__ x,
                   const int32_t* __restrict__ coords, const double* __restrict__ st, const float* __restrict__ coef,
                   const float* __restrict__ weight, int relu, int64_t n, int C, int B, float* __restrict__ dx) {
  using VT = typename InVec<V>::T;
  const int CV = C / V;
  const int64_t nv = n * CV;
  const int64_t BC = (int64_t)B * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / CV;
    const int c = (int)(i - r * CV) * V;
    const VT xv = __ldg(reinterpret_cast<const VT*>(x) + i);
    const VT gv = __ldg(reinterpret_cast<const VT*>(dy) + i);
    VT yv = gv;
    if (relu) yv = __ldg(reinterpret_cast<const VT*>(y) + i);
    const int b = __ldg(coords + r * 4);
    VT o;
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float f = __int_as_float(0x7fffffff);
      if (in_batch_ok(b, B)) {
        const int64_t k = (int64_t)b * C + c + j;
        const float g = (relu && !(InVec<V>::get(yv, j) > 0.f)) ? 0.f : InVec<V>::get(gv, j);
        const float xh = in_xhat(InVec<V>::get(xv, j), st, k, BC);
        const float a = (float)__ldg(st + BC + k) * __ldg(weight + c + j);
        f = a * fmaf(-xh, __ldg(coef + BC + k), g - __ldg(coef + k));
      }
      InVec<V>::set(o, j, f);
    }
    reinterpret_cast<VT*>(dx)[i] = o;
  }
}

struct InPlan {
  int W, n_ct, n_chunks;
  int64_t rows_per_chunk;
  size_t smem;
};

template <bool FWD>
static InPlan in_plan(int64_t n, int C, int B) {
  InPlan p;
  const size_t slab = InSlab<FWD>::bytes(B);
  int64_t W = (int64_t)(kInSmemMax / slab);
  p.W = (int)(W < 1 ? 1 : (W > kInMaxWarps ? kInMaxWarps : W));
  p.n_ct = (int)ceil_div(C, kInTile);
  int64_t ch = ceil_div(kInTargetWarps, (int64_t)p.W * p.n_ct);
  const int64_t by_rows = ceil_div(n, (int64_t)p.W * kInMinRowsPerWarp);
  const int64_t by_bytes = (int64_t)4096 / B;  // partial rows: at most 4096 (chunk, instance) pairs
  if (ch > by_rows) ch = by_rows;
  if (ch > by_bytes) ch = by_bytes;
  if (ch < 1) ch = 1;
  p.rows_per_chunk = ceil_div(n, ch);
  p.n_chunks = (int)ceil_div(n, p.rows_per_chunk);
  p.smem = slab * p.W;
  return p;
}

static size_t in_part_bytes(const InPlan& p, int C, int B) {
  return sizeof(double) * (size_t)p.n_chunks * B * (1 + 2 * (size_t)C);
}

static int in_apply_grid(int64_t nv) {
  const int64_t g = ceil_div(nv, 256);
  return (int)(g < 1 ? 1 : (g > 148 * 16 ? 148 * 16 : g));
}

static int in_check(const char* who, const float* x, const int32_t* coords, int64_t n, int C, int B,
                    const double* stats) {
  LG_CHECK_ARG(n >= 0 && C >= 1 && B >= 1, "%s: needs n >= 0, C >= 1, B >= 1", who);
  LG_CHECK_ARG(x && coords && stats, "%s: null pointer", who);
  const uintptr_t a = C % 4 == 0 ? 15 : 3;
  LG_CHECK_ARG(((uintptr_t)x & a) == 0 && ((uintptr_t)coords & 3) == 0 && ((uintptr_t)stats & 7) == 0,
               "%s: misaligned pointer (features need 16 bytes when C %% 4 == 0, else 4)", who);
  if (B > kInMaxB) {
    set_error("%s: B = %d instances, at most %d are supported", who, B, kInMaxB);
    return LG_ERR_UNSUPPORTED;
  }
  return LG_OK;
}

}  // namespace lg

using namespace lg;

extern "C" int lg_instnorm_forward(const float* x, const int32_t* coords, int64_t n, int32_t C, int32_t B,
                                   const float* weight, const float* bias, float eps, int32_t relu, float* y,
                                   void* y16, int32_t fmt, double* stats, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = in_check("lg_instnorm_forward", x, coords, n, C, B, stats);
  if (rc) return rc;
  LG_CHECK_ARG(weight && bias && y, "lg_instnorm_forward: null pointer");
  LG_CHECK_ARG(!y16 || fmt == LG_FMT_BF16 || fmt == LG_FMT_FP16, "lg_instnorm_forward: bad 16-bit format");
  LG_CHECK_ARG(eps >= 0.f, "lg_instnorm_forward: eps must be >= 0");
  const uintptr_t a = C % 4 == 0 ? 15 : 3;
  LG_CHECK_ARG(((uintptr_t)y & a) == 0 && ((uintptr_t)y16 & (C % 4 == 0 ? 7 : 1)) == 0 &&
                   ((uintptr_t)weight & 3) == 0 && ((uintptr_t)bias & 3) == 0,
               "lg_instnorm_forward: misaligned pointer");
  if (n == 0) return LG_OK;
  const InPlan p = in_plan<true>(n, C, B);
  ArenaCursor ar;
  rc = arena_begin(stream, arena_pad(in_part_bytes(p, C, B)), &ar);
  if (rc) return rc;
  double* part = (double*)arena_take(&ar, in_part_bytes(p, C, B));
  LG_CUDA_OK(cudaFuncSetAttribute(k_in_stats<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  k_in_stats<true><<<dim3((unsigned)p.n_chunks, (unsigned)p.n_ct), dim3(kInTile, p.W), p.smem, stream>>>(
      x, nullptr, nullptr, nullptr, coords, n, C, B, 0, p.rows_per_chunk, part);
  LG_LAUNCH_OK();
  InBwdOut none = {};
  k_in_tail<true><<<dim3((unsigned)p.n_ct, (unsigned)B), dim3(kInTile, kInTailY), 0, stream>>>(part, p.n_chunks, C, B,
                                                                                              eps, stats, none);
  LG_LAUNCH_OK();
  if (C % 4 == 0)
    k_in_apply<4><<<in_apply_grid(n * C / 4), 256, 0, stream>>>(x, coords, stats, weight, bias, relu, n, C, B, y,
                                                               (unsigned short*)y16, fmt);
  else
    k_in_apply<1><<<in_apply_grid(n * C), 256, 0, stream>>>(x, coords, stats, weight, bias, relu, n, C, B, y,
                                                            (unsigned short*)y16, fmt);
  LG_LAUNCH_OK();
  return LG_OK;
}

extern "C" int lg_instnorm_backward(const float* dy, const float* x, const float* y, const int32_t* coords, int64_t n,
                                    int32_t C, int32_t B, const float* weight, int32_t relu, const double* stats,
                                    float* dx, float* dweight, float* dbias, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = in_check("lg_instnorm_backward", x, coords, n, C, B, stats);
  if (rc) return rc;
  LG_CHECK_ARG(dy && weight && dx && dweight && dbias && (!relu || y), "lg_instnorm_backward: null pointer");
  const uintptr_t a = C % 4 == 0 ? 15 : 3;
  LG_CHECK_ARG(((uintptr_t)dy & a) == 0 && ((uintptr_t)y & a) == 0 && ((uintptr_t)dx & a) == 0 &&
                   ((uintptr_t)weight & 3) == 0 && ((uintptr_t)dweight & 3) == 0 && ((uintptr_t)dbias & 3) == 0,
               "lg_instnorm_backward: misaligned pointer");
  const InPlan p = in_plan<false>(n > 0 ? n : 1, C, B);
  const size_t BC = (size_t)B * C;
  ArenaCursor ar;
  rc = arena_begin(stream,
                   arena_pad(in_part_bytes(p, C, B)) + arena_pad(sizeof(double) * 2 * BC) + arena_pad(sizeof(float) * 2 * BC),
                   &ar);
  if (rc) return rc;
  double* part = (double*)arena_take(&ar, in_part_bytes(p, C, B));
  InBwdOut bo;
  bo.sums = (double*)arena_take(&ar, sizeof(double) * 2 * BC);
  bo.coef = (float*)arena_take(&ar, sizeof(float) * 2 * BC);
  bo.dweight = dweight, bo.dbias = dbias;
  rc = counter_slot(&bo.ticket);
  if (rc) return rc;
  // n = 0 still runs the statistics (one empty chunk) and the tail: dweight = dbias = 0
  LG_CUDA_OK(cudaFuncSetAttribute(k_in_stats<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  k_in_stats<false><<<dim3((unsigned)p.n_chunks, (unsigned)p.n_ct), dim3(kInTile, p.W), p.smem, stream>>>(
      x, dy, y, stats, coords, n, C, B, relu, p.rows_per_chunk, part);
  LG_LAUNCH_OK();
  k_in_tail<false><<<dim3((unsigned)p.n_ct, (unsigned)B), dim3(kInTile, kInTailY), 0, stream>>>(part, p.n_chunks, C, B,
                                                                                               0.f, nullptr, bo);
  LG_LAUNCH_OK();
  if (n == 0) return LG_OK;
  if (C % 4 == 0)
    k_in_bwd_apply<4><<<in_apply_grid(n * C / 4), 256, 0, stream>>>(dy, y, x, coords, stats, bo.coef, weight, relu, n,
                                                                    C, B, dx);
  else
    k_in_bwd_apply<1><<<in_apply_grid(n * C), 256, 0, stream>>>(dy, y, x, coords, stats, bo.coef, weight, relu, n, C, B,
                                                                dx);
  LG_LAUNCH_OK();
  return LG_OK;
}
