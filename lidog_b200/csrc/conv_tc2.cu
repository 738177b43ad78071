// Sparse convolution on tcgen05: gather-GEMM (forward / dgrad) and wgrad pipelines.
//
// Measured on B200 (profiles/r01_conv_bench_v1.txt): tile::gather4 TMA moves 256 B per instruction and
// sustains ~100 SM cycles per instruction, 2.7x slower than LDGSTS (cp.async) row gathers; and a
// producer that waits for its own copies keeps only two stages in flight.  This pipeline therefore
//   * gathers operand rows with cp.async (16 B per lane, 4 lanes per 64-byte row segment, so every
//     request is a full 32 B sector pair) and lets the copies themselves arrive on the stage's
//     mbarrier (cp.async.mbarrier.arrive.noinc): producers never wait for data, the whole ring is in
//     flight;
//   * gives each of the 4 producer warps whole stages (unit u -> warp u % 4), so the index fetch of
//     one stage overlaps the copies of three others;
//   * forward / dgrad (k_gemm2): a CTA owns a SUPER-TILE of T row tiles whose T accumulators live in
//     TMEM together (T * N <= 512 columns); the loop runs kernel offset outermost, so one TMA load of
//     the weight panel W[k] feeds up to T gathered tiles (weight traffic / T);
//   * wgrad (k_wgrad2): a CTA owns a group of G kernel offsets (G * Cout <= 512 TMEM columns) and a
//     chunk of tiles; the dY tile is staged once and reused by every offset of the group.
// Shared-memory operand tiles use the SWIZZLE_64B layout (64-byte rows = 32 channels).
// Results are deterministic: every output row / weight element is written once in a fixed order.
// Reference contract: MinkowskiConvolution(+Transpose) forward/backward, utils/models/minkunet_bev.py:57-123.
// Inference (k_gemm2<PC, true>): the epilogue also applies the eval-mode batch norm, the residual and the ReLU that
// follow the convolution, with k_bn_apply's expression, and writes the 16-bit operand copy (lg_conv_layer_infer).
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "runtime.cuh"
#include "tc_ptx.cuh"

namespace lg {

int launch_reduce_partials(const float* partial, int n_chunks, int64_t n_elems, const float* out_scale, float* dW,
                           cudaStream_t stream);

namespace v2 {
using namespace ptx;

constexpr int kRowB = 64;            // bytes per smem operand row (32 x 16-bit)
constexpr int kSub = 128 * kRowB;    // one [128 rows x 32 channels] sub-tile = 8 KB
constexpr int kEpiWarps = 4;         // warps 0..3
constexpr int kMmaWarp = 4;
constexpr int kBWarp = 5;            // weight-panel TMA producer (forward) / unused (wgrad)
constexpr int kProdWarp0 = 6;
constexpr int kProdWarps = 4;        // warps 6..9
constexpr int kIdxWarp = kProdWarp0 + kProdWarps;  // warp 10: row-id ring (bulk copies of 512 B id rows)
constexpr int kThreads = (kIdxWarp + 1) * 32;
constexpr int kIdxSlotBytes = LG_TILE_ROWS * 4;
// Row-id ring of k_gemm2.  The ncu source view of the lean kernel (profiles/r01_s4_gemm2_source_stalls.txt) shows the
// MMA warp polling the stage-full barrier ~17 times per unit and the producers waiting for free stages a quarter of
// the time -- a latency-bound ring -- so shared memory goes to operand stages first: 16 id slots (8 KB instead of 16).
constexpr int kGemmIdxSlots = 4 * kProdWarps;
constexpr int kSchedSlots = 4;                                   // super-tile hand-out ring
constexpr int kSchedWords = 12;  // ring entry: [0] super-tile, [1] "tile has any offset" bits, [2..9] mask word 0 of its tiles
constexpr int kSchedConsumers = kEpiWarps + 2 + kProdWarps;      // warps that read every ring entry
constexpr int kStgPitch = 36;                                    // floats per staged row (32 + 4: conflict-free v4)
constexpr int kStgBytes = kEpiWarps * 32 * kStgPitch * 4;        // epilogue transposition buffers

__device__ __forceinline__ uint32_t sw64(uint32_t r, uint32_t j) { return r * kRowB + ((j ^ ((r >> 1) & 3u)) << 4); }

// 1D bulk copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_copy_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ int lds32(uint32_t saddr) {
  int v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(saddr) : "memory");
  return v;
}

__device__ __forceinline__ void cp_async_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Dynamic super-tile schedule.  The id warp draws super-tiles from a global counter (largest index first:
// with mask-sorted plans the expensive tiles sit at the end, so the tail of the launch is made of cheap
// ones) and publishes them through a 4-entry shared-memory ring; every other warp reads each entry once.
struct SchedCursor {
  int slot;
  uint32_t phase;
};
// tile-mask words of the (<= 8) tiles of a super-tile, kept in registers; word 0 travels with the ring entry
// (every layer on the tensor-core path has K <= 27 offsets = one word), further words are reloaded every 32 offsets
struct TileMasks {
  uint32_t w[8];
};
struct SchedItem {
  int64_t st;    // super-tile index, < 0 = no more work
  uint32_t any;  // bit t = tile t has at least one offset
  TileMasks tm;  // mask word 0 of the tiles
};
// All helpers below are called by fully active warps and broadcast lane 0's value, so everything derived from
// them (unit sequence, stage counters, descriptors) is warp-uniform for ptxas.
__device__ __forceinline__ void sched_next(SchedItem& it, SchedCursor& c, uint64_t* fullS, uint64_t* emptyS,
                                           const int* ring, int lane, int* err) {
  mbar_wait(&fullS[c.slot], c.phase, err, 20);
  const volatile int* e = ring + c.slot * kSchedWords;
  it.st = (int)bcast0((uint32_t)e[0]);
  it.any = bcast0((uint32_t)e[1]);
#pragma unroll
  for (int t = 0; t < 8; ++t) it.tm.w[t] = bcast0((uint32_t)e[2 + t]);
  __syncwarp();
  if (lane == 0) mbar_arrive(&emptyS[c.slot]);
  if (++c.slot == kSchedSlots) {
    c.slot = 0;
    c.phase ^= 1;
  }
}

__device__ __forceinline__ void load_masks(TileMasks& tm, const lgConvPlan& p, int64_t tile0, int nt, int word) {
#pragma unroll
  for (int t = 0; t < 8; ++t)
    tm.w[t] = (t < nt) ? bcast0(__ldg(p.tile_mask + (tile0 + t) * p.mask_words + word)) : 0u;
}
__device__ __forceinline__ uint32_t present_bits(const TileMasks& tm, int k) {
  uint32_t m = 0;
#pragma unroll
  for (int t = 0; t < 8; ++t) m |= ((tm.w[t] >> (k & 31)) & 1u) << t;
  return m;
}
// offsets present in ANY tile of the super-tile, for mask word `word` (word 0 came with the ring entry)
__device__ __forceinline__ uint32_t offset_bits(TileMasks& tm, const lgConvPlan& p, int64_t tile0, int nt, int word) {
  if (word) load_masks(tm, p, tile0, nt, word);
  return ((tm.w[0] | tm.w[1]) | (tm.w[2] | tm.w[3])) | ((tm.w[4] | tm.w[5]) | (tm.w[6] | tm.w[7]));
}
// Every role walks the same (offset k, tile bits m) sequence: set bits only -- the one-thread roles used to spend
// ~100 cycles per ABSENT offset on the shift/or chains of a plain k = 0..K-1 scan.
// Lane j of the warp computes the tile bits of offset 32 w + j once per mask word (the 32 shift/or instructions of
// present_bits run in parallel across the lanes); inside the walk an offset's bits are one shuffle away.
#define LG_FOR_EACH_OFFSET(tm, plan, tile0, nt, k, m)                                                  \
  for (int _w = 0; _w < (plan).mask_words; ++_w)                                                       \
    for (uint32_t _kb = offset_bits(tm, plan, tile0, nt, _w), _mk = present_bits(tm, lane); _kb;       \
         _kb &= _kb - 1)                                                                               \
      if (const int _j = __ffs(_kb) - 1; true)                                                         \
        if (const int k = 32 * _w + _j; true)                                                          \
          if (const uint32_t m = __shfl_sync(0xffffffffu, _mk, _j); true)

__device__ __forceinline__ uint32_t any_mask(const lgConvPlan& p, int64_t tile0, int nt) {
  uint32_t m = 0;
  for (int t = 0; t < nt; ++t) {
    uint32_t w = 0;
    for (int i = 0; i < p.mask_words; ++i) w |= __ldg(p.tile_mask + (tile0 + t) * p.mask_words + i);
    m |= (w != 0 ? 1u : 0u) << t;
  }
  return bcast0(m);
}

// Gather 128 rows x (PC * 32) channels of a row-major 16-bit matrix into `dst` (PC sub-tiles of 8 KB,
// SWIZZLE_64B).  One warp does the whole stage: lane = (row % 8, 16-byte piece), 16 rows per lane
// (rows[i] = id of row 8*i + lane/4, negative = zero fill); PC copies per row are issued back to back;
// byte offsets stay in 32 bits (host checks rows * ld * 2 < 2^32).
template <int PC>
__device__ __forceinline__ void gather_rows(uint8_t* dst, const uint8_t* __restrict__ src, uint32_t ld_bytes,
                                            const int (&rows)[16], int lane) {
  const int piece = lane & 3, rsub = lane >> 2;
  const uint8_t* base = src + piece * 16;
  uint8_t* d0 = dst + sw64(rsub, piece);  // row 8*i + rsub sits 512*i bytes further (same swizzle phase)
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int row = rows[i];
    const bool ok = row >= 0;
    const uint8_t* s = base + (size_t)((uint32_t)(ok ? row : 0) * ld_bytes);
#pragma unroll
    for (int c = 0; c < PC; ++c) cp_async16(d0 + i * 512 + c * kSub, s + c * 64, ok);
  }
}

__device__ __forceinline__ void gather_stage(uint8_t* dst, const uint16_t* src, int ld, int col0, int pc,
                                             const int (&rows)[16], int lane) {
  const uint8_t* s = reinterpret_cast<const uint8_t*>(src + col0);
  const uint32_t ldb = (uint32_t)ld * 2u;
  switch (pc) {
    case 1: gather_rows<1>(dst, s, ldb, rows, lane); break;
    case 2: gather_rows<2>(dst, s, ldb, rows, lane); break;
    case 3: gather_rows<3>(dst, s, ldb, rows, lane); break;
    default: gather_rows<4>(dst, s, ldb, rows, lane); break;
  }
}

// row ids of a stage from the shared-memory id ring (filled by the id warp's bulk copies)
__device__ __forceinline__ void ids_from_ring(int (&rows)[16], uint32_t slot_saddr, int lane) {
#pragma unroll
  for (int i = 0; i < 16; ++i) rows[i] = lds32(slot_saddr + 4 * (8 * i + (lane >> 2)));
}

// ------------------------------------------------------------------------------------ forward / dgrad
struct Gemm2Args {
  lgConvPlan plan;
  const uint16_t* A;  // [n_in][Ck]
  float* Y;           // [n_out][N]
  float* stats;       // nullable: [n_tiles * 4][2N] per-(tile, epilogue warp) column sums / sums of squares of Y
  const float* out_scale;
  const float* bias;
  int Ck, N, n_blk, flip, umma_fmt;
  int T, pc, n_panels, sa, sb, np;  // np = active producer warps (<= sa, see the ring-phase note)
  int64_t n_tiles, n_super;
  int* err;
  int* sched;  // [0..3] next super-tile per blockIdx.y, [4] finished CTAs (self-resetting)
};

// Epilogue of the inference instantiations: Y = act(fmaf(acc, scale, shift) [+ res]), Y16 = 16-bit copy of Y.
// A separate kernel parameter after the tensor map, so the training instantiations keep their parameter layout.
struct InferEpi {
  const float* scale;  // [N] = bn_stats + 2N (lg_bn_apply layout)
  const float* shift;  // [N] = bn_stats + 3N
  const float* res;    // nullable [n_out][N]
  uint16_t* Y16;       // nullable [n_out][N]
  int relu, fmt;
};

// same rounding as bn_to16 (bn.cu): the 16-bit copy equals the one lg_bn_apply writes
__device__ __forceinline__ uint16_t epi_to16(float v, int fmt) {
  if (fmt == LG_FMT_BF16) return __bfloat16_as_ushort(__float2bfloat16_rn(v));
  v = fminf(fmaxf(v, -65504.f), 65504.f);
  return __half_as_ushort(__float2half_rn(v));
}

// One 32-column block of 32 rows of the inference epilogue.  Lane = (row (lane >> 3) + 4 j, columns 4 (lane & 7)..+3):
// every warp instruction reads / writes 4 rows x 128 contiguous bytes (Y, res) or 4 x 64 bytes (Y16), like the staged
// Y store of the training epilogue.  `stg` holds the accumulators transposed through shared memory, or nothing when
// the tile has no neighbour at all (acc = 0: fmaf(0, s, h) is what k_bn_apply computes on the zeros the training
// epilogue writes there).  The expression is k_bn_apply's, operation by operation, so the result is bit-identical
// to lg_conv_layer_forward followed by lg_bn_apply.
// The loads (scale, shift, the 8 residual rows) are issued by infer_loads before the accumulators are read from TMEM:
// the compiler cannot move them above the stores to Y (res and Y may alias as far as it knows), so loaded inside the
// row loop each row would wait for its own residual load in series.
struct InferIn {
  float4 sc, sh, r[8];
};
__device__ __forceinline__ void infer_loads(const InferEpi& e, InferIn& in, const int (&srow)[8], int N, int c) {
  in.sc = __ldg(reinterpret_cast<const float4*>(e.scale + c));
  in.sh = __ldg(reinterpret_cast<const float4*>(e.shift + c));
  if (e.res) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (srow[j] >= 0) in.r[j] = __ldg(reinterpret_cast<const float4*>(e.res + (int64_t)srow[j] * N + c));
  }
}
__device__ __forceinline__ void infer_block(const InferEpi& e, const InferIn& in, const float* stg, bool have,
                                            const int (&srow)[8], float* Y, int N, int c, int lane) {
  const float4 sc = in.sc, sh = in.sh;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (srow[j] < 0) continue;
    const int64_t off = (int64_t)srow[j] * N + c;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    if (have) a = *reinterpret_cast<const float4*>(stg + ((lane >> 3) + 4 * j) * kStgPitch + 4 * (lane & 7));
    float4 o = make_float4(fmaf(a.x, sc.x, sh.x), fmaf(a.y, sc.y, sh.y), fmaf(a.z, sc.z, sh.z), fmaf(a.w, sc.w, sh.w));
    if (e.res) {
      const float4 r = in.r[j];
      o.x += r.x, o.y += r.y, o.z += r.z, o.w += r.w;
    }
    if (e.relu) o = make_float4(fmaxf(o.x, 0.f), fmaxf(o.y, 0.f), fmaxf(o.z, 0.f), fmaxf(o.w, 0.f));
    *reinterpret_cast<float4*>(Y + off) = o;
    if (e.Y16) {
      uint2 h;
      h.x = epi_to16(o.x, e.fmt) | ((uint32_t)epi_to16(o.y, e.fmt) << 16);
      h.y = epi_to16(o.z, e.fmt) | ((uint32_t)epi_to16(o.w, e.fmt) << 16);
      *reinterpret_cast<uint2*>(e.Y16 + off) = h;
    }
  }
}

// PC: 32-channel chunks per operand stage (= g.pc).  TMEM holds two accumulator sets of T tiles (2 * T * n_blk <= 512
// columns): the epilogue of one super-tile overlaps the MMAs of the next.
// INFER: the inference epilogue (InferEpi; no statistics, no bias, no out_scale, n_blk % 32 == 0 -- host-checked).
template <int PC, bool INFER>
__global__ void __launch_bounds__(kThreads, 1)
    k_gemm2(const Gemm2Args g, const __grid_constant__ CUtensorMap tmB, const InferEpi e) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int stageA = PC * kSub, stageB = PC * g.n_blk * kRowB;
  uint8_t* smA = smem;
  uint8_t* smB = smem + (size_t)g.sa * stageA;
  uint8_t* smI = smB + (size_t)g.sb * stageB;  // id ring: ni slots of 128 row ids
  constexpr int ni = kGemmIdxSlots;
  float* smStg = (float*)(smI + (size_t)ni * kIdxSlotBytes);  // epilogue transposition buffers
  uint64_t* fullA = (uint64_t*)((uint8_t*)smStg + kStgBytes);
  uint64_t* emptyA = fullA + g.sa;
  uint64_t* fullB = emptyA + g.sa;
  uint64_t* emptyB = fullB + g.sb;
  uint64_t* fullI = emptyB + g.sb;
  uint64_t* emptyI = fullI + ni;
  uint64_t* acc_full = emptyI + ni;
  uint64_t* acc_empty = acc_full + 2;  // one per accumulator: [set * T + tile slot]
  uint64_t* fullS = acc_empty + 8;
  uint64_t* emptyS = fullS + kSchedSlots;
  uint32_t* tmem_slot = (uint32_t*)(emptyS + kSchedSlots);
  int* sched_ring = (int*)(tmem_slot + 2);
  SchedCursor sc{0, 0};
  const int n0 = blockIdx.y * g.n_blk;
  const int K = g.plan.kernel_volume;

  if (threadIdx.x == 0) {
    for (int s = 0; s < g.sa; ++s) {
      mbar_init(&fullA[s], 32);
      mbar_init(&emptyA[s], 1);
    }
    for (int s = 0; s < g.sb; ++s) {
      mbar_init(&fullB[s], 1);
      mbar_init(&emptyB[s], 1);
    }
    for (int s = 0; s < ni; ++s) {
      mbar_init(&fullI[s], 1);
      mbar_init(&emptyI[s], 1);
    }
    mbar_init(&acc_full[0], 1);
    mbar_init(&acc_full[1], 1);
    for (int t = 0; t < 8; ++t) mbar_init(&acc_empty[t], kEpiWarps * 32);
    for (int t = 0; t < kSchedSlots; ++t) {
      mbar_init(&fullS[t], 1);
      mbar_init(&emptyS[t], kSchedConsumers);
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_slot, 512);
  if (warp == kBWarp && lane == 0) prefetch_tmap(&tmB);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kIdxWarp) {
    // ===================================================================== id ring (runs ahead; one elected lane issues)
    int slot = 0;
    uint32_t iphase = 0;
    for (;;) {
      mbar_wait(&emptyS[sc.slot], sc.phase ^ 1, g.err, 21);
      int drawn = 0;
      if (lane == 0) drawn = atomicAdd(g.sched + blockIdx.y, 1);
      drawn = (int)bcast0((uint32_t)drawn);
      const int64_t st = drawn < g.n_super ? g.n_super - 1 - drawn : -1;
      const int64_t tile0 = st * g.T;
      const int nt = st < 0 ? 0 : (int)min((int64_t)g.T, g.n_tiles - tile0);
      // the entry carries the tiles' mask words, so the other nine warps never go to global memory for them
      uint32_t w0 = 0;
      if (lane < nt) w0 = __ldg(g.plan.tile_mask + (tile0 + lane) * g.plan.mask_words);
      uint32_t any = __ballot_sync(0xffffffffu, w0 != 0);
      if (g.plan.mask_words > 1 && st >= 0) any = any_mask(g.plan, tile0, nt);
      int* entry = sched_ring + sc.slot * kSchedWords;
      if (lane < 8) entry[2 + lane] = (int)w0;
      if (lane == 0) {
        entry[0] = (int)st;
        entry[1] = (int)any;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&fullS[sc.slot]);
      __syncwarp();
      if (++sc.slot == kSchedSlots) {
        sc.slot = 0;
        sc.phase ^= 1;
      }
      if (st < 0) break;
      TileMasks tm;
#pragma unroll
      for (int t = 0; t < 8; ++t) tm.w[t] = __shfl_sync(0xffffffffu, w0, t);
      LG_FOR_EACH_OFFSET(tm, g.plan, tile0, nt, k, m) {
        for (int p = 0; p < g.n_panels; ++p) {
          for (uint32_t mm = m; mm; mm &= mm - 1) {
            const int t = __ffs(mm) - 1;
            mbar_wait(&emptyI[slot], iphase ^ 1, g.err, 7);
            if (elect_one()) {
              mbar_arrive_expect_tx(&fullI[slot], kIdxSlotBytes);
              bulk_copy_g2s(smI + (size_t)slot * kIdxSlotBytes,
                            g.plan.nbr + (int64_t)k * g.plan.k_stride + (tile0 + t) * LG_TILE_ROWS, kIdxSlotBytes,
                            &fullI[slot]);
            }
            __syncwarp();
            if (++slot == ni) {
              slot = 0;
              iphase ^= 1;
            }
          }
        }
      }
    }
  } else if (warp >= kProdWarp0 && warp < kProdWarp0 + kProdWarps) {
    // ===================================================================== A producers (cp.async gather)
    const int pw = warp - kProdWarp0;
    int stage = 0, turn = 0, slot = 0;
    uint32_t phase = 0, iphase = 0;
    SchedItem item;
    for (;;) {
      sched_next(item, sc, fullS, emptyS, sched_ring, lane, g.err);
      const int64_t st = item.st;
      if (st < 0) break;
      const int64_t tile0 = st * g.T;
      const int nt = (int)min((int64_t)g.T, g.n_tiles - tile0);
      TileMasks& tm = item.tm;
      LG_FOR_EACH_OFFSET(tm, g.plan, tile0, nt, k, m) {
        for (int p = 0; p < g.n_panels; ++p) {
          for (int t = 0; t < nt; ++t) {
            if (!((m >> t) & 1u)) continue;
            if (turn == pw) {
              int rows[16];
              mbar_wait(&fullI[slot], iphase, g.err, 8);
              ids_from_ring(rows, smem_u32(smI) + slot * kIdxSlotBytes, lane);
              __syncwarp();
              if (lane == 0) mbar_arrive(&emptyI[slot]);
              if (lane == 0) mbar_wait(&emptyA[stage], phase ^ 1, g.err, 1);
              __syncwarp();
              gather_rows<PC>(smA + (size_t)stage * stageA, reinterpret_cast<const uint8_t*>(g.A + p * PC * 32), (uint32_t)g.Ck * 2u, rows, lane);
              cp_async_arrive_noinc(&fullA[stage]);
            }
            turn = (turn + 1 == g.np) ? 0 : turn + 1;
            if (++stage == g.sa) {
              stage = 0;
              phase ^= 1;
            }
            if (++slot == ni) {
              slot = 0;
              iphase ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == kBWarp) {
    // ===================================================================== B producer (weight panels, TMA)
    int bs = 0;
    uint32_t bphase = 0;
    SchedItem item;
    for (;;) {
      sched_next(item, sc, fullS, emptyS, sched_ring, lane, g.err);
      const int64_t st = item.st;
      if (st < 0) break;
      const int64_t tile0 = st * g.T;
      const int nt = (int)min((int64_t)g.T, g.n_tiles - tile0);
      TileMasks& tm = item.tm;
      LG_FOR_EACH_OFFSET(tm, g.plan, tile0, nt, k, m) {
        (void)m;
        const int wk = g.flip ? (K - 1 - k) : k;
        for (int p = 0; p < g.n_panels; ++p) {
          mbar_wait(&emptyB[bs], bphase ^ 1, g.err, 2);
          if (elect_one()) {
            mbar_arrive_expect_tx(&fullB[bs], (uint32_t)stageB);
            uint8_t* dst = smB + (size_t)bs * stageB;
#pragma unroll
            for (int c = 0; c < PC; ++c)
              tma_load_2d(dst + c * g.n_blk * kRowB, &tmB, (p * PC + c) * 32, wk * g.N + n0, &fullB[bs]);
          }
          __syncwarp();
          if (++bs == g.sb) {
            bs = 0;
            bphase ^= 1;
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ===================================================================== MMA issuer
    // The loop runs warp-uniformly (every lane computes the same unit sequence; the masks are broadcast), and
    // one elected lane issues the tcgen05 instructions: descriptors are a constant high word plus
    // (address >> 4) held in uniform registers, so a unit costs two barrier waits, a proxy fence and 2*pc
    // back-to-back UTCHMMAs.  Accumulators are handed back by the epilogue tile by tile (acc_empty[t]), so
    // the first offsets of the next super-tile overlap the drain of the previous one.
    const uint32_t idesc = make_idesc(g.umma_fmt, 0, 0, LG_TILE_ROWS, g.n_blk);
    const uint64_t desc_hi = make_smem_desc(0, 16, 8 * kRowB, kLayoutSw64);
    const uint32_t a_base = smem_u32(smA) >> 4, b_base = smem_u32(smB) >> 4;
    const uint32_t a_stage16 = (uint32_t)stageA >> 4, b_stage16 = (uint32_t)stageB >> 4;
    const uint32_t b_sub16 = (uint32_t)(g.n_blk * kRowB) >> 4;
    // everything the loop needs lives in registers: no parameter loads, no 64-bit index arithmetic in the hot path
    const int sa = g.sa, sb = g.sb, T = g.T, n_panels = g.n_panels, n_blk = g.n_blk;
    int stage = 0, bs = 0;
    uint32_t phase = 0, bphase = 0, it = 0;
    SchedItem item;
    for (;;) {
      sched_next(item, sc, fullS, emptyS, sched_ring, lane, g.err);
      const int64_t st = item.st;
      if (st < 0) break;
      const int64_t tile0 = st * T;
      const int nt = (int)min((int64_t)T, g.n_tiles - tile0);
      if (!item.any) continue;
      const int set = (int)(it & 1);
      const uint32_t eparity = ((it >> 1) & 1) ^ 1;
      const uint32_t d_base = tmem_base + (uint32_t)(set * T) * (uint32_t)n_blk;  // first accumulator of this set
      ++it;
      // all T accumulators of the set are taken up front (the epilogue hands them back tile by tile; the last one
      // arrives a few hundred cycles after the first) -- the inner loop then has no hand-off test per unit
      for (int t = 0; t < T; ++t) mbar_wait(&acc_empty[set * T + t], eparity, g.err, 3);
      uint32_t started = 0;
      TileMasks& tm = item.tm;
      LG_FOR_EACH_OFFSET(tm, g.plan, tile0, nt, k, m) {
        for (int p = 0; p < n_panels; ++p) {
          mbar_wait(&fullB[bs], bphase, g.err, 4);
          const uint32_t db_lo = b_base + bs * b_stage16;
          // The units of this (offset, panel) -- at most T <= ring depth (host-checked) -- are handled together:
          // wait for their stages, ONE proxy fence, issue their MMAs back to back, release the stages.
          {
            int s = stage;
            uint32_t ph = phase;
            for (uint32_t bb = m; bb; bb &= bb - 1) {
              mbar_wait(&fullA[s], ph, g.err, 5);
              if (++s == sa) {
                s = 0;
                ph ^= 1;
              }
            }
          }
          fence_proxy_async();  // cp.async (generic proxy) writes -> tcgen05 (async proxy) reads
          tc_fence_after();
          if (elect_one()) {
            int s = stage;
            for (uint32_t bb = m; bb; bb &= bb - 1) {
              const int t = __ffs(bb) - 1;
              const uint64_t da0 = desc_hi | (uint64_t)(a_base + s * a_stage16);
              const uint64_t db0 = desc_hi | (uint64_t)db_lo;
              const uint32_t d_tmem = d_base + (uint32_t)t * (uint32_t)n_blk;
              const uint32_t acc0 = (started >> t) & 1u;
#pragma unroll
              for (int c = 0; c < PC; ++c) {
                umma_f16(d_tmem, da0 + c * (kSub >> 4), db0 + c * b_sub16, idesc, c == 0 ? acc0 : 1u);
                umma_f16(d_tmem, da0 + c * (kSub >> 4) + 2, db0 + c * b_sub16 + 2, idesc, 1u);
              }
              umma_commit(&emptyA[s]);
              if (++s == sa) s = 0;
            }
            umma_commit(&emptyB[bs]);
          }
          __syncwarp();
          started |= m;
          stage += __popc(m);
          if (stage >= sa) {
            stage -= sa;
            phase ^= 1;
          }
          if (++bs == sb) {
            bs = 0;
            bphase ^= 1;
          }
        }
      }
      if (elect_one()) umma_commit(&acc_full[set]);
      __syncwarp();
    }
  } else {
    // ===================================================================== epilogue (warps 0..3)
    const float scale = g.out_scale ? g.out_scale[0] : 1.f;
    uint32_t it = 0;
    SchedItem item;
    for (;;) {
      sched_next(item, sc, fullS, emptyS, sched_ring, lane, g.err);
      const int64_t st = item.st;
      if (st < 0) break;
      const int64_t tile0 = st * g.T;
      const int nt = (int)min((int64_t)g.T, g.n_tiles - tile0);
      const uint32_t am = item.any;
      int a0 = 0;
      if (am) {
        const int set = (int)(it & 1);
        a0 = set * g.T;
        mbar_wait(&acc_full[set], (it >> 1) & 1, g.err, 6);
        ++it;
        tc_fence_after();
      }
      for (int t = 0; t < g.T; ++t) {
        if (t < nt) {
          const int64_t s = (tile0 + t) * LG_TILE_ROWS + warp * 32 + lane;
          int64_t row = g.plan.out_row ? (int64_t)g.plan.out_row[s] : s;
          const bool row_ok = row >= 0 && row < g.plan.n_out;
          if constexpr (INFER) {
            const bool have = (am >> t) & 1u;
            const uint32_t taddr = tmem_base + (a0 + t) * g.n_blk + ((uint32_t)(warp * 32) << 16);
            float* stg = smStg + warp * 32 * kStgPitch;
            int srow[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) srow[j] = __shfl_sync(0xffffffffu, row_ok ? (int)row : -1, (lane >> 3) + 4 * j);
            for (int n = 0; n < g.n_blk; n += 32) {
              const int c = n0 + n + 4 * (lane & 7);
              InferIn in;
              infer_loads(e, in, srow, g.N, c);
              if (have) {
                uint32_t v[32];
                tmem_ld32(taddr + n, v);
                tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < 8; ++q)
                  *reinterpret_cast<float4*>(stg + lane * kStgPitch + 4 * q) =
                      make_float4(__uint_as_float(v[4 * q + 0]), __uint_as_float(v[4 * q + 1]),
                                  __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
                __syncwarp();
              }
              infer_block(e, in, stg, have, srow, g.Y, g.N, c, lane);
              __syncwarp();
            }
            if (am) {  // hand accumulator t back
              tc_fence_before();
              mbar_arrive(&acc_empty[a0 + t]);
            }
            continue;
          }
          float* yrow = g.Y + (row_ok ? row : 0) * g.N + n0;
          // BN statistics of the layer that follows (SURVEY.md 8f-1): this warp's 32 rows contribute one partial
          // row [sum | sum of squares] per tile; a fixed shuffle order and a fixed (tile, warp) slot keep the later
          // reduction deterministic although tiles are handed out dynamically.
          float* strow = g.stats ? g.stats + ((tile0 + t) * kEpiWarps + warp) * 2 * (int64_t)g.N + n0 : nullptr;
          if (!((am >> t) & 1u)) {  // no neighbour at all: bias / zeros
            if (row_ok)
              for (int n = 0; n < g.n_blk; n += 4) {
                float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
                if (g.bias) o = *reinterpret_cast<const float4*>(g.bias + n0 + n);
                *reinterpret_cast<float4*>(yrow + n) = o;
              }
            if (strow) {
              const int valid = __popc(__ballot_sync(0xffffffffu, row_ok));
              for (int n = 4 * lane; n < g.n_blk; n += 128) {
                float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (g.bias) b4 = *reinterpret_cast<const float4*>(g.bias + n0 + n);
                const float v = (float)valid;
                *reinterpret_cast<float4*>(strow + n) = make_float4(v * b4.x, v * b4.y, v * b4.z, v * b4.w);
                *reinterpret_cast<float4*>(strow + g.N + n) =
                    make_float4(v * b4.x * b4.x, v * b4.y * b4.y, v * b4.z * b4.z, v * b4.w * b4.w);
              }
            }
          } else {
            // TMEM lane = tile row, so a thread holds 32 consecutive columns of ONE row; storing them directly
            // makes every warp store touch 32 different lines (measured: the epilogue was store-bound).  The
            // 32x32 block goes through shared memory instead and leaves as 4 rows x 128 contiguous bytes per
            // warp instruction.
            const uint32_t taddr = tmem_base + (a0 + t) * g.n_blk + ((uint32_t)(warp * 32) << 16);
            float* stg = smStg + warp * 32 * kStgPitch;
            int srow[8];  // result rows this lane stores: tile rows (lane >> 3) + 4 j
#pragma unroll
            for (int j = 0; j < 8; ++j) srow[j] = __shfl_sync(0xffffffffu, row_ok ? (int)row : -1, (lane >> 3) + 4 * j);
            int n = 0;
            for (; n + 32 <= g.n_blk; n += 32) {
              uint32_t v[32];
              tmem_ld32(taddr + n, v);
              tmem_ld_wait();
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                float4 o;
                o.x = __uint_as_float(v[4 * q + 0]) * scale;
                o.y = __uint_as_float(v[4 * q + 1]) * scale;
                o.z = __uint_as_float(v[4 * q + 2]) * scale;
                o.w = __uint_as_float(v[4 * q + 3]) * scale;
                if (g.bias) {
                  const float4 bb = *reinterpret_cast<const float4*>(g.bias + n0 + n + 4 * q);
                  o.x += bb.x, o.y += bb.y, o.z += bb.z, o.w += bb.w;
                }
                *reinterpret_cast<float4*>(stg + lane * kStgPitch + 4 * q) = o;
              }
              __syncwarp();
              float4 cs = make_float4(0.f, 0.f, 0.f, 0.f), cq = cs;
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float4 o = *reinterpret_cast<const float4*>(stg + ((lane >> 3) + 4 * j) * kStgPitch + 4 * (lane & 7));
                if (srow[j] >= 0) {
                  // (Summing the gradient of a multi-consumer tensor here -- read-modify-write instead of a store --
                  // was measured: the 31 separate adds it removes cost 0.6 ms per step, the loads in this epilogue
                  // 2.8 ms (k_gemm2 8.39 -> 11.17 ms, profiles/r02_c_launch_summary_grad_accum_experiment.txt): the
                  // accumulators drain late and the MMA warp stalls.  Not kept.)
                  *reinterpret_cast<float4*>(g.Y + (int64_t)srow[j] * g.N + n0 + n + 4 * (lane & 7)) = o;
                  cs.x += o.x, cs.y += o.y, cs.z += o.z, cs.w += o.w;
                  cq.x = fmaf(o.x, o.x, cq.x), cq.y = fmaf(o.y, o.y, cq.y), cq.z = fmaf(o.z, o.z, cq.z),
                  cq.w = fmaf(o.w, o.w, cq.w);
                }
              }
              if (strow) {  // lanes l, l+8, l+16, l+24 hold the same 4 columns of different rows
#pragma unroll
                for (int d = 8; d <= 16; d <<= 1) {
                  cs.x += __shfl_xor_sync(0xffffffffu, cs.x, d), cs.y += __shfl_xor_sync(0xffffffffu, cs.y, d);
                  cs.z += __shfl_xor_sync(0xffffffffu, cs.z, d), cs.w += __shfl_xor_sync(0xffffffffu, cs.w, d);
                  cq.x += __shfl_xor_sync(0xffffffffu, cq.x, d), cq.y += __shfl_xor_sync(0xffffffffu, cq.y, d);
                  cq.z += __shfl_xor_sync(0xffffffffu, cq.z, d), cq.w += __shfl_xor_sync(0xffffffffu, cq.w, d);
                }
                if (lane < 8) {
                  *reinterpret_cast<float4*>(strow + n + 4 * lane) = cs;
                  *reinterpret_cast<float4*>(strow + g.N + n + 4 * lane) = cq;
                }
              }
              __syncwarp();
            }
            for (; n < g.n_blk; n += 16) {  // 16-column remainder (N % 32 == 16): direct stores
              uint32_t v[16];
              tmem_ld16(taddr + n, v);
              tmem_ld_wait();
              if (row_ok) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  float4 o;
                  o.x = __uint_as_float(v[4 * q + 0]) * scale;
                  o.y = __uint_as_float(v[4 * q + 1]) * scale;
                  o.z = __uint_as_float(v[4 * q + 2]) * scale;
                  o.w = __uint_as_float(v[4 * q + 3]) * scale;
                  if (g.bias) {
                    const float4 bb = *reinterpret_cast<const float4*>(g.bias + n0 + n + 4 * q);
                    o.x += bb.x, o.y += bb.y, o.z += bb.z, o.w += bb.w;
                  }
                  *reinterpret_cast<float4*>(yrow + n + 4 * q) = o;
                }
              }
            }
          }
        }
        if (am) {  // hand accumulator t back (tcgen05.ld of it have completed: wait::ld above)
          tc_fence_before();
          mbar_arrive(&acc_empty[a0 + t]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem_base, 512);
  if (threadIdx.x == 0) {  // the last CTA to finish rewinds the counters for the launch that reuses this slot
    __threadfence();
    const int done = atomicAdd(g.sched + 4, 1);
    if (done == (int)(gridDim.x * gridDim.y) - 1) {
      for (int y = 0; y < 5; ++y) g.sched[y] = 0;
      __threadfence();
    }
  }
}

// ------------------------------------------------------------------------------------ wgrad
// dW[k] (Cin x Cout) = sum_s X16[nbr[k][s], :]^T dY16[out_row[s] (or s), :].
// CTA = (group of G kernel offsets, 128-channel block of Cin, chunk of tiles).
// A stage: gathered X rows [128 pairs x 4 sub-blocks of 32 channels]; B stage: dY rows [128 pairs x Cout].
struct Wgrad2Args {
  lgConvPlan plan;
  const uint16_t* X;
  const uint16_t* dY;
  float* partial;  // [chunks][K][Cin][Cout]
  int Cin, Cout, m_blocks, G, n_groups, tiles_per_chunk, umma_fmt, sa, sb, np, bmax;
  int strided;  // offsets of a group are grp + j * n_groups (load balance) instead of a contiguous range
  int64_t n_tiles;
  int* err;
};

__global__ void __launch_bounds__(kThreads, 1) k_wgrad2(const Wgrad2Args g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int grp = blockIdx.x / g.m_blocks, mb = blockIdx.x % g.m_blocks;
  const int chunk = blockIdx.y;
  const int K = g.plan.kernel_volume;
  // The offsets of a group are STRIDED: group grp owns offsets grp, grp + n_groups, grp + 2 n_groups, ...  Contiguous
  // ranges put the whole centre plane of a 3x3x3 kernel (offsets 9..17: 60 % of all pairs of a LiDAR map) into one or
  // two groups: on the bench batch the heaviest CTA had 2.8x the mean number of units (190 vs 69,
  // profiles/r02_d_wgrad_balance.txt); strided groups bring that to 1.4x for 1.5x more dY tile loads.
  const int ng = g.strided ? g.n_groups : 1;
  const int k0 = g.strided ? grp : grp * g.G;                                  // first offset of the group
  const int gcount = g.strided ? (K - grp + ng - 1) / ng : min(K, k0 + g.G) - k0;  // number of offsets
  const int m0 = mb * 128;
  const int na = min(4, (g.Cin - m0) / 32);  // real 32-channel sub-blocks of the A operand
  const int nb = g.Cout / 32;
  // (the MMA always reads 4 sub-blocks = 128 accumulator lanes; lanes of sub-blocks that are not staged hold whatever
  // the stage held before and are never read back: the epilogue stops at Cin)
  const int stageA = 4 * kSub, stageB = nb * kSub;
  uint8_t* smA = smem;
  uint8_t* smB = smem + (size_t)g.sa * stageA;
  uint8_t* smI = smB + (size_t)g.sb * stageB;  // id ring: ni slots of 128 row ids
  const int ni = 8 * g.np;
  uint64_t* fullA = (uint64_t*)(smI + (size_t)ni * kIdxSlotBytes);
  uint64_t* emptyA = fullA + g.sa;
  uint64_t* fullB = emptyA + g.sa;
  uint64_t* emptyB = fullB + g.sb;
  uint64_t* fullI = emptyB + g.sb;
  uint64_t* emptyI = fullI + ni;
  uint64_t* done = emptyI + ni;
  uint32_t* tmem_slot = (uint32_t*)(done + 1);
  // chunk c owns tiles c, c + chunks, c + 2 chunks, ...: with mask-sorted plans neighbouring tiles have the
  // same offsets, so interleaving gives every CTA of an offset group the same amount of work
  const int64_t t0 = chunk, t1 = g.n_tiles, tstep = gridDim.y;

  if (threadIdx.x == 0) {
    for (int s = 0; s < g.sa; ++s) {
      mbar_init(&fullA[s], 32);
      mbar_init(&emptyA[s], 1);
    }
    for (int s = 0; s < g.sb; ++s) {
      mbar_init(&fullB[s], 32);
      mbar_init(&emptyB[s], 1);
    }
    for (int s = 0; s < ni; ++s) {
      mbar_init(&fullI[s], 1);
      mbar_init(&emptyI[s], 1);
    }
    mbar_init(done, 1);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // bit j of group_mask(tile) = offset k0 + j * ng present in the tile (K <= 64, host-checked)
  auto group_mask = [&](int64_t tile) -> uint32_t {
    const uint32_t* mw = g.plan.tile_mask + tile * g.plan.mask_words;
    uint64_t bits = (uint64_t)__ldg(mw) | (g.plan.mask_words > 1 ? (uint64_t)__ldg(mw + 1) << 32 : 0ull);
    bits >>= k0;
    uint32_t m;
    if (ng == 1) {
      m = (uint32_t)bits;
    } else {
      m = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < gcount) m |= (uint32_t)((bits >> (j * ng)) & 1ull) << j;
    }
    return bcast0(m & ((1u << gcount) - 1u));
  };

  if (warp == kIdxWarp) {
    // ---------------------------------------------------------------- id ring (runs ahead; one elected lane issues)
    int slot = 0;
    uint32_t iphase = 0;
    for (int64_t tile = t0; tile < t1; tile += tstep) {
      for (uint32_t mm = group_mask(tile); mm; mm &= mm - 1) {
        const int k = k0 + (__ffs(mm) - 1) * ng;
        mbar_wait(&emptyI[slot], iphase ^ 1, g.err, 16);
        if (elect_one()) {
          mbar_arrive_expect_tx(&fullI[slot], kIdxSlotBytes);
          bulk_copy_g2s(smI + (size_t)slot * kIdxSlotBytes,
                        g.plan.nbr + (int64_t)k * g.plan.k_stride + tile * LG_TILE_ROWS, kIdxSlotBytes, &fullI[slot]);
        }
        __syncwarp();
        if (++slot == ni) {
          slot = 0;
          iphase ^= 1;
        }
      }
    }
  } else if (warp >= kProdWarp0) {
    // ---------------------------------------------------------------- X producers
    const int pw = warp - kProdWarp0;
    int stage = 0, turn = 0, slot = 0;
    uint32_t phase = 0, iphase = 0;
    for (int64_t tile = t0; tile < t1; tile += tstep) {
      for (uint32_t mm = group_mask(tile); mm; mm &= mm - 1) {
        if (turn == pw) {
          int rows[16];
          mbar_wait(&fullI[slot], iphase, g.err, 17);
          ids_from_ring(rows, smem_u32(smI) + slot * kIdxSlotBytes, lane);
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(&emptyI[slot]);
            mbar_wait(&emptyA[stage], phase ^ 1, g.err, 11);
          }
          __syncwarp();
          gather_stage(smA + (size_t)stage * stageA, g.X, g.Cin, m0, na, rows, lane);
          cp_async_arrive_noinc(&fullA[stage]);
        }
        turn = (turn + 1 == g.np) ? 0 : turn + 1;
        if (++stage == g.sa) {
          stage = 0;
          phase ^= 1;
        }
        if (++slot == ni) {
          slot = 0;
          iphase ^= 1;
        }
      }
    }
  } else if (warp == kBWarp) {
    // ---------------------------------------------------------------- dY producer (one warp, whole tiles)
    // ncu (profiles/r02_a_wgrad2_source_stalls.txt): the MMA warp polled this ring 41 times per tile -- two stages and
    // two dependent global latencies per tile (out_row, then the rows) could not keep it fed.  The row ids of the NEXT
    // tile are now loaded before the wait for a free stage, and the ring is as deep as shared memory allows.
    int bs = 0;
    uint32_t bphase = 0;
    const int lim = (int)g.plan.n_out;
    auto next_tile = [&](int64_t t) {
      while (t < t1 && !group_mask(t)) t += tstep;
      return t;
    };
    auto load_rows = [&](int (&rows)[16], int64_t tile) {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int sl = (int)(tile * LG_TILE_ROWS) + 8 * i + (lane >> 2);
        const int r = g.plan.out_row ? __ldg(g.plan.out_row + sl) : sl;
        rows[i] = (r < lim) ? r : -1;
      }
    };
    int64_t tile = next_tile(t0);
    int rows[16], rows_n[16];
    if (tile < t1) load_rows(rows, tile);
    while (tile < t1) {
      const int64_t nxt = next_tile(tile + tstep);
      if (nxt < t1) load_rows(rows_n, nxt);
      if (lane == 0) mbar_wait(&emptyB[bs], bphase ^ 1, g.err, 12);
      __syncwarp();
      uint8_t* dst = smB + (size_t)bs * stageB;
      for (int c0 = 0; c0 < nb; c0 += 4)
        gather_stage(dst + c0 * kSub, g.dY, g.Cout, c0 * 32, min(4, nb - c0), rows, lane);
      cp_async_arrive_noinc(&fullB[bs]);
      if (++bs == g.sb) {
        bs = 0;
        bphase ^= 1;
      }
#pragma unroll
      for (int i = 0; i < 16; ++i) rows[i] = rows_n[i];
      tile = nxt;
    }
  } else if (warp == kMmaWarp) {
    // warp-uniform loop, one elected lane issues (see k_gemm2)
    const uint32_t idesc = make_idesc(g.umma_fmt, 1, 1, 128, g.Cout);
    // MN-major SWIZZLE_64B: LBO = pitch between 32-channel sub-blocks, SBO = 8 rows * 64 B
    const uint64_t desc_hi = make_smem_desc(0, kSub, 8 * kRowB, kLayoutSw64);
    const uint32_t a_base = smem_u32(smA) >> 4, b_base = smem_u32(smB) >> 4;
    const uint32_t a_stage16 = (uint32_t)stageA >> 4, b_stage16 = (uint32_t)stageB >> 4;
    int stage = 0, bs = 0;
    uint32_t phase = 0, bphase = 0, started = 0;
    for (int64_t tile = t0; tile < t1; tile += tstep) {
      const uint32_t m = group_mask(tile);
      if (!m) continue;
      mbar_wait(&fullB[bs], bphase, g.err, 13);
      const uint64_t db0 = desc_hi | (uint64_t)(b_base + bs * b_stage16);
      // the offsets of this tile in batches of <= bmax (<= ring depth): all waits, one proxy fence, then the MMAs
      uint32_t mm = m;
      while (mm) {
        uint32_t batch = 0;
        {
          uint32_t x = mm;
          for (int i = 0; i < g.bmax && x; ++i) {
            batch |= x & (0u - x);
            x &= x - 1;
          }
        }
        mm &= ~batch;
        {
          int s = stage;
          uint32_t ph = phase;
          for (uint32_t bb = batch; bb; bb &= bb - 1) {
            mbar_wait(&fullA[s], ph, g.err, 14);
            if (++s == g.sa) {
              s = 0;
              ph ^= 1;
            }
          }
        }
        fence_proxy_async();
        tc_fence_after();
        if (elect_one()) {
          int s = stage;
          for (uint32_t bb = batch; bb; bb &= bb - 1) {
            const int j = __ffs(bb) - 1;
            const uint64_t da0 = desc_hi | (uint64_t)(a_base + s * a_stage16);
            const uint32_t d_tmem = tmem_base + j * g.Cout;
            const uint32_t acc0 = (started >> j) & 1u;
            umma_f16(d_tmem, da0, db0, idesc, acc0);
#pragma unroll
            for (int q = 1; q < LG_TILE_ROWS / 16; ++q)  // K = 16 gathered rows per MMA
              umma_f16(d_tmem, da0 + q * (16 * kRowB >> 4), db0 + q * (16 * kRowB >> 4), idesc, 1u);
            umma_commit(&emptyA[s]);
            if (++s == g.sa) s = 0;
          }
        }
        __syncwarp();
        started |= batch;
        for (int i = __popc(batch); i > 0; --i) {
          if (++stage == g.sa) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
      if (elect_one()) umma_commit(&emptyB[bs]);
      __syncwarp();
      if (++bs == g.sb) {
        bs = 0;
        bphase ^= 1;
      }
    }
    if (elect_one()) {
      if (started)
        umma_commit(done);
      else
        mbar_arrive(done);
    }
    __syncwarp();
  } else {
    // ---------------------------------------------------------------- epilogue: lane = input channel
    uint32_t started = 0;
    for (int64_t tile = t0; tile < t1; tile += tstep) started |= group_mask(tile);
    const int ci = m0 + warp * 32 + lane;
    mbar_wait(done, 0, g.err, 15);
    tc_fence_after();
    for (int j = 0; j < gcount; ++j) {
      const int k = k0 + j * ng;
      const bool have = (started >> j) & 1u;
      float* prow = g.partial + (((int64_t)chunk * K + k) * g.Cin + (ci < g.Cin ? ci : 0)) * g.Cout;
      const uint32_t taddr = tmem_base + j * g.Cout + ((uint32_t)(warp * 32) << 16);
      for (int n = 0; n < g.Cout; n += 16) {
        uint32_t v[16];
        if (have) {
          tmem_ld16(taddr + n, v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int q = 0; q < 16; ++q) v[q] = 0u;
        }
        if (ci < g.Cin) {
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<float4*>(prow + n + 4 * q) =
                make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]),
                            __uint_as_float(v[4 * q + 3]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem_base, 512);
}

constexpr size_t kSmemBudget = 225 * 1024;

static inline size_t wgrad_tail_bytes(int sa, int sb) {  // id ring + barriers + tmem slot + alignment slack
  const int ni = 8 * kProdWarps;
  return (size_t)ni * kIdxSlotBytes + (size_t)(2 * sa + 2 * sb + 2 * ni + 2) * 8 + 16 + 1024;
}
static inline size_t tail_bytes(int sa, int sb) {  // + epilogue staging + schedule ring
  const int ni = kGemmIdxSlots;
  return (size_t)ni * kIdxSlotBytes + kStgBytes + (size_t)(2 * sa + 2 * sb + 2 * ni + 11 + 2 * kSchedSlots) * 8 + 16 +
         4 * kSchedWords * kSchedSlots + 1024;
}

// Launch shape of k_gemm2, a pure function of the problem: grid (min(n_super, sm_count), n_split) x kThreads, smem bytes.
struct Gemm2Shape {
  int n_split, n_blk;  // column blocks of N (blockIdx.y) and their width
  int T, pc, n_panels, sa, sb, np;  // see Gemm2Args
  int64_t n_super;
  size_t smem;
};

// column-block width of k_gemm2 for N output columns (blocks of <= 256 columns, equal widths)
static inline int gemm2_n_blk(int N) { return N / ((N + 255) / 256); }

static int gemm2_shape(int64_t n_tiles, int Ck, int N, int sm_count, bool stats, Gemm2Shape* s) {
  s->n_split = (N + 255) / 256;
  s->n_blk = gemm2_n_blk(N);
  if (s->n_blk % 16 != 0 || s->n_blk * s->n_split != N) {
    set_error("lg_conv_gemm_tc: N=%d cannot be split into equal multiples of 16", N);
    return LG_ERR_UNSUPPORTED;
  }
  if (stats && s->n_blk % 32 != 0) {
    set_error("lg_conv_layer_forward: epilogue statistics need column blocks that are multiples of 32 (N=%d)", N);
    return LG_ERR_UNSUPPORTED;
  }
  if (s->n_split > 4) {
    set_error("lg_conv_gemm_tc: N=%d needs more than 4 column blocks", N);
    return LG_ERR_UNSUPPORTED;
  }
  const int n_chunks = Ck / 32;
  s->n_panels = (n_chunks + 3) / 4;
  while (n_chunks % s->n_panels != 0) ++s->n_panels;
  s->pc = n_chunks / s->n_panels;
  // Tiles per super-tile.  TMEM holds two accumulator sets of T tiles, 2 * T * n_blk <= 512 columns (n_blk <= 256 by
  // the split above, so T >= 1 always fits), and 2 * T <= 8 accumulator barriers; but keep >= ~3 super-tiles per SM.
  int T = 256 / s->n_blk < 4 ? 256 / s->n_blk : 4;
  while (T > 1 && ceil_div(n_tiles, T) * s->n_split < 3 * (int64_t)sm_count) --T;
  // Pipeline shape.  The weight-panel ring gets 3 stages whenever 4 operand stages still fit next to it (with 2,
  // the TMA load of the next panel cannot start before the MMAs of the current one retire: the 256-channel
  // layers waited 22 % of the time for weights); the rest of the budget goes to operand (gather) stages.
  size_t stageA, stageB;
  for (;;) {
    stageA = (size_t)s->pc * kSub, stageB = (size_t)s->pc * s->n_blk * kRowB;
    s->sb = (3 * stageB + 4 * stageA + tail_bytes(4, 3) <= kSmemBudget) ? 3 : 2;
    s->sa = 12;
    while (s->sa > 2 && s->sa * stageA + s->sb * stageB + tail_bytes(s->sa, s->sb) > kSmemBudget) --s->sa;
    // would 2 weight stages buy an operand stage?  Only where a weight stage is no bigger than an operand stage:
    // measured (profiles/r01_s4_sweep_n_ring.txt) -17 % / -12 % on the 128-channel layers at tensor stride 8 / 4,
    // but +2 ... +5 % on the 256-channel single-tile layers, whose 32 KB panels want the third stage.
    if (s->sb == 3 && s->sa < 12 && stageB <= stageA) {
      int sa2 = 12;
      while (sa2 > 2 && sa2 * stageA + 2 * stageB + tail_bytes(sa2, 2) > kSmemBudget) --sa2;
      if (sa2 > s->sa) {
        s->sa = sa2;
        s->sb = 2;
      }
    }
    if (s->sa >= kProdWarps || s->pc == 1) break;
    // deeper ring with smaller panels (pc must divide the chunk count)
    int pc = s->pc - 1;
    while (n_chunks % pc != 0) --pc;
    s->pc = pc;
    s->n_panels = n_chunks / pc;
  }
  s->T = T < s->sa ? T : s->sa;  // the MMA warp waits for up to T stages at once: they must all fit in the ring
  s->n_super = ceil_div(n_tiles, s->T);
  // Ring-phase rule: a producer warp revisits a stage only after the consumer freed it once, which the
  // parity wait can tell only when consecutive units of one warp are < one ring wrap apart: np <= sa.
  s->np = s->sa < kProdWarps ? s->sa : kProdWarps;
  s->smem = s->sa * stageA + s->sb * stageB + tail_bytes(s->sa, s->sb);
  if (s->smem > kSmemBudget) {
    set_error("lg_conv_gemm_tc: shared memory %zu exceeds the budget (Ck=%d N=%d)", s->smem, Ck, N);
    return LG_ERR_UNSUPPORTED;
  }
  return LG_OK;
}

}  // namespace v2

// host launcher: forward / dgrad
// infer (nullable): run the inference epilogue (k_gemm2<PC, true>); out_scale, bias and stats must then be null
int launch_gemm_tc2(const lgConvPlan* plan, const void* A16, int Ck, const void* B16, int N, int flip_k, int fmt,
                    const float* out_scale, const float* bias, float* Y, float* stats, cudaStream_t stream,
                    const v2::InferEpi* infer = nullptr) {
  using namespace v2;
  // the inference epilogue has no bias, no output scale and no statistics, and no 16-column remainder path
  LG_CHECK_ARG(!infer || (!out_scale && !bias && !stats && gemm2_n_blk(N) % 32 == 0),
               "launch_gemm_tc2: the inference epilogue takes no bias / out_scale / statistics and 32-column blocks");
  int sm_count = 0;
  int* err = nullptr;
  int rc = tc_runtime(&sm_count, &err);
  if (rc) return rc;
  const int64_t n_tiles = plan->n_slots / LG_TILE_ROWS;
  Gemm2Shape s;
  rc = gemm2_shape(n_tiles, Ck, N, sm_count, stats != nullptr, &s);
  if (rc) return rc;
  Gemm2Args g;
  g.plan = *plan;
  g.A = (const uint16_t*)A16;
  g.Y = Y;
  g.stats = stats;
  g.out_scale = out_scale;
  g.bias = bias;
  g.Ck = Ck;
  g.N = N;
  g.n_blk = s.n_blk;
  g.flip = flip_k;
  g.umma_fmt = (fmt == LG_FMT_BF16) ? 1 : 0;
  g.T = s.T;
  g.pc = s.pc;
  g.n_panels = s.n_panels;
  g.sa = s.sa;
  g.sb = s.sb;
  g.np = s.np;
  g.n_tiles = n_tiles;
  g.n_super = s.n_super;
  g.err = err;
  rc = counter_slot(&g.sched);
  if (rc) return rc;
  CUtensorMap tmB;
  memset(&tmB, 0, sizeof(tmB));
  rc = tc_make_tmap(&tmB, B16, (int64_t)plan->kernel_volume * N, Ck, g.n_blk);
  if (rc) return rc;
  const dim3 grid((unsigned)(s.n_super < sm_count ? s.n_super : sm_count), (unsigned)s.n_split);
  const size_t smem = s.smem;
  InferEpi e;
  memset(&e, 0, sizeof(e));
  if (infer) e = *infer;
#define LG_LAUNCH_GEMM2(PCV, INF)                                                                                 \
  do {                                                                                                            \
    LG_CUDA_OK(cudaFuncSetAttribute(k_gemm2<PCV, INF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  \
    k_gemm2<PCV, INF><<<grid, kThreads, smem, stream>>>(g, tmB, e);                                               \
  } while (0)
  if (infer) {
    switch (g.pc) {
      case 1: LG_LAUNCH_GEMM2(1, true); break;
      case 2: LG_LAUNCH_GEMM2(2, true); break;
      case 3: LG_LAUNCH_GEMM2(3, true); break;
      default: LG_LAUNCH_GEMM2(4, true); break;
    }
  } else {
    switch (g.pc) {
      case 1: LG_LAUNCH_GEMM2(1, false); break;
      case 2: LG_LAUNCH_GEMM2(2, false); break;
      case 3: LG_LAUNCH_GEMM2(3, false); break;
      default: LG_LAUNCH_GEMM2(4, false); break;
    }
  }
#undef LG_LAUNCH_GEMM2
  LG_LAUNCH_OK();
  return LG_OK;
}

static int wgrad2_shape(const lgConvPlan* plan, int Cin, int Cout, int* G, int* n_groups, int* tiles_per_chunk) {
  const int K = plan->kernel_volume;
  int gmax = 512 / Cout;
  if (gmax > 8) gmax = 8;
  if (gmax > K) gmax = K;
  *n_groups = (K + gmax - 1) / gmax;
  *G = (K + *n_groups - 1) / *n_groups;
  const int m_blocks = (Cin + 127) / 128;
  const int64_t n_tiles = plan->n_slots / LG_TILE_ROWS;
  // Chunks of tiles per (offset group, channel block).  Every chunk costs one partial dW (written by the epilogue,
  // re-read by the reduction) and one pipeline ramp, so a chunk should own >= ~32 tiles; but the launch wants at
  // least one wave of 148 CTAs and gains nothing beyond four.  Measured (profiles/r01_s4_sweep_a.txt): the layers at
  // tensor stride >= 4 ran 1.3-1.8x faster with 148 CTAs than with 592, the stride-1 layers 1.3x slower.
  const int64_t per = (int64_t)*n_groups * m_blocks;
  const int64_t hi = 592 / per, lo = ceil_div((int64_t)148, per);
  int64_t want = n_tiles / 32;
  if (want < lo) want = lo;
  if (want > hi) want = hi;
  if (want < 1) want = 1;
  int64_t chunks = n_tiles < want ? n_tiles : want;
  if (chunks < 1) chunks = 1;
  *tiles_per_chunk = (int)ceil_div(n_tiles > 0 ? n_tiles : 1, chunks);
  return (int)ceil_div(n_tiles > 0 ? n_tiles : 1, *tiles_per_chunk);
}

size_t wgrad_tc2_workspace(const lgConvPlan* plan, int Cin, int Cout) {
  int G, ng, tpc;
  const int chunks = wgrad2_shape(plan, Cin, Cout, &G, &ng, &tpc);
  return (size_t)chunks * plan->kernel_volume * Cin * Cout * sizeof(float) + 256;
}

int launch_wgrad_tc2(const lgConvPlan* plan, const void* X16, int Cin, const void* dY16, int Cout, int fmt,
                     const float* out_scale, float* dW, void* workspace, cudaStream_t stream) {
  using namespace v2;
  int sm_count = 0;
  int* err = nullptr;
  int rc = tc_runtime(&sm_count, &err);
  if (rc) return rc;
  Wgrad2Args g;
  g.plan = *plan;
  g.X = (const uint16_t*)X16;
  g.dY = (const uint16_t*)dY16;
  g.partial = (float*)workspace;
  g.Cin = Cin;
  g.Cout = Cout;
  g.m_blocks = (Cin + 127) / 128;
  const int chunks = wgrad2_shape(plan, Cin, Cout, &g.G, &g.n_groups, &g.tiles_per_chunk);
  g.umma_fmt = (fmt == LG_FMT_BF16) ? 1 : 0;
  g.n_tiles = plan->n_slots / LG_TILE_ROWS;
  g.err = err;
  // strided groups where there are enough groups for the imbalance to matter: measured -7 ... -20 % on the 96- / 128- /
  // 256-channel layers (5 ... 14 groups), +15 % on the 32-channel ones (4 groups of 7 offsets, already balanced, and
  // every extra dY tile load is pure HBM cost there) -- profiles/r02_d_layer_table_strided.txt
  g.strided = g.n_groups >= 5 ? 1 : 0;
  if (plan->kernel_volume > 64) {
    set_error("lg_conv_wgrad_tc: kernel volume %d > 64 is not on the tensor-core path", plan->kernel_volume);
    return LG_ERR_UNSUPPORTED;
  }
  // An X stage always holds 4 sub-blocks (32 KB) although a 96-channel layer fills 3 and a 32-channel layer 1.
  // Packing the stages tighter is WRONG: the M = 128 MMA then reads its unused sub-blocks out of the neighbouring
  // stages, and the full-scale parity test (tests/test_gpu_fullscale.py) measured 0.3-2.5 % error in dW -- bisected
  // on hardware (profiles/r02_b_wgrad_bisect.log).
  const size_t stageA = 4 * kSub, stageB = (size_t)(Cout / 32) * kSub;
  // dY ring: 3 stages when 4 X stages still fit next to them (the MMA warp waited on this ring, see the dY producer)
  g.sb = (4 * stageA + 3 * stageB + wgrad_tail_bytes(4, 3) <= kSmemBudget) ? 3 : 2;
  g.sa = 6;
  while (g.sa > 2 && g.sa * stageA + g.sb * stageB + wgrad_tail_bytes(g.sa, g.sb) > kSmemBudget) --g.sa;
  g.np = g.sa < kProdWarps ? g.sa : kProdWarps;
  g.bmax = g.sa < 4 ? g.sa : 4;  // offsets of a tile per batch of the MMA warp
  const size_t smem = g.sa * stageA + g.sb * stageB + wgrad_tail_bytes(g.sa, g.sb);
  if (smem > kSmemBudget) {
    set_error("lg_conv_wgrad_tc: shared memory %zu exceeds the budget (Cin=%d Cout=%d)", smem, Cin, Cout);
    return LG_ERR_UNSUPPORTED;
  }
  dim3 grid((unsigned)(g.n_groups * g.m_blocks), (unsigned)chunks);
  LG_CUDA_OK(cudaFuncSetAttribute(k_wgrad2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_wgrad2<<<grid, kThreads, smem, stream>>>(g);
  LG_LAUNCH_OK();
  return launch_reduce_partials((const float*)workspace, chunks, (int64_t)plan->kernel_volume * Cin * Cout, out_scale,
                                dW, stream);
}

static int check_tc_plan(const lgConvPlan* p, const char* who) {
  LG_CHECK_ARG(p != nullptr, "%s: null plan", who);
  LG_CHECK_ARG(p->n_slots > 0 && p->n_slots % LG_TILE_ROWS == 0, "%s: n_slots must be a positive multiple of 128", who);
  LG_CHECK_ARG(p->kernel_volume >= 1 && p->kernel_volume <= 128 && p->mask_words == (p->kernel_volume + 31) / 32,
               "%s: bad kernel_volume/mask_words", who);
  LG_CHECK_ARG(p->k_stride == 0 || p->k_stride == p->n_slots, "%s: k_stride must be 0 or n_slots", who);
  LG_CHECK_ARG(p->nbr && p->tile_mask, "%s: null plan arrays", who);
  LG_CHECK_ARG(p->n_in < ((int64_t)1 << 31) && p->n_out < ((int64_t)1 << 31), "%s: more than 2^31 rows", who);
  return LG_OK;
}

static int check_gemm(const lgConvPlan* plan, int Ck, int N, int fmt, const char* who) {
  int rc = check_tc_plan(plan, who);
  if (rc) return rc;
  if (Ck % 32 != 0 || N % 16 != 0 || N < 16 || N > 512) {
    set_error("%s: Ck=%d must be a multiple of 32 and N=%d a multiple of 16 in [16,512]", who, Ck, N);
    return LG_ERR_UNSUPPORTED;
  }
  // the gather kernels keep row byte offsets in 32 bits
  if ((uint64_t)plan->n_in * (uint64_t)Ck * 2ull >= ((uint64_t)1 << 32)) {
    set_error("%s: operand matrix of %lld x %d 16-bit elements exceeds the 4 GiB row-offset range", who,
              (long long)plan->n_in, Ck);
    return LG_ERR_UNSUPPORTED;
  }
  LG_CHECK_ARG(fmt == LG_FMT_BF16 || fmt == LG_FMT_FP16, "%s: bad format", who);
  return LG_OK;
}

static int check_wgrad(const lgConvPlan* plan, int Cin, int Cout, int fmt, const char* who) {
  int rc = check_tc_plan(plan, who);
  if (rc) return rc;
  if (Cin % 32 != 0 || Cout % 32 != 0 || Cout > 256 || Cin < 32) {
    set_error("%s: Cin=%d, Cout=%d must be multiples of 32 with Cout <= 256", who, Cin, Cout);
    return LG_ERR_UNSUPPORTED;
  }
  if ((uint64_t)plan->n_in * (uint64_t)Cin * 2ull >= ((uint64_t)1 << 32) ||
      (uint64_t)plan->n_out * (uint64_t)Cout * 2ull >= ((uint64_t)1 << 32)) {
    set_error("%s: operand matrix exceeds the 4 GiB row-offset range", who);
    return LG_ERR_UNSUPPORTED;
  }
  LG_CHECK_ARG(fmt == LG_FMT_BF16 || fmt == LG_FMT_FP16, "%s: bad format", who);
  return LG_OK;
}

}  // namespace lg

using namespace lg;

extern "C" int lg_conv_gemm_tc(const lgConvPlan* plan, const void* A16, int32_t Ck, const void* B16, int32_t N,
                               int32_t flip_k, int32_t fmt, const float* out_scale, const float* bias, float* Y,
                               void* stream_) {
  int rc = check_gemm(plan, Ck, N, fmt, "lg_conv_gemm_tc");
  if (rc) return rc;
  LG_CHECK_ARG(A16 && B16 && Y, "lg_conv_gemm_tc: null pointer");
  return launch_gemm_tc2(plan, A16, Ck, B16, N, flip_k, fmt, out_scale, bias, Y, nullptr, (cudaStream_t)stream_);
}

extern "C" size_t lg_conv_wgrad_tc_workspace(const lgConvPlan* plan, int32_t Cin, int32_t Cout) {
  if (!plan || Cout < 32 || Cout > 256) return 0;
  return wgrad_tc2_workspace(plan, Cin, Cout);
}

extern "C" int lg_conv_wgrad_tc(const lgConvPlan* plan, const void* X16, int32_t Cin, const void* dY16, int32_t Cout,
                                int32_t fmt, const float* out_scale, float* dW, void* workspace, size_t workspace_bytes,
                                void* stream_) {
  int rc = check_wgrad(plan, Cin, Cout, fmt, "lg_conv_wgrad_tc");
  if (rc) return rc;
  LG_CHECK_ARG(X16 && dY16 && dW && workspace, "lg_conv_wgrad_tc: null pointer");
  LG_CHECK_ARG(workspace_bytes >= lg_conv_wgrad_tc_workspace(plan, Cin, Cout), "lg_conv_wgrad_tc: workspace too small");
  return launch_wgrad_tc2(plan, X16, Cin, dY16, Cout, fmt, out_scale, dW, workspace, (cudaStream_t)stream_);
}

/* One MinkowskiConvolution forward on the tensor-core path in one host call (see include/lidog_b200.h). */
extern "C" int lg_conv_layer_forward(const lgConvPlan* plan, const void* X16, int32_t Cin, const float* W, int32_t Cout,
                                     void* w16, void* w16t, int32_t prep, int32_t fmt, const float* bias, float* Y,
                                     float* stat_partials, void* stream_) {
  int rc = check_gemm(plan, Cin, Cout, fmt, "lg_conv_layer_forward");
  if (rc) return rc;
  LG_CHECK_ARG(X16 && w16t && Y && (!prep || W), "lg_conv_layer_forward: null pointer");
  if (prep) {
    rc = lg_prep_weights(W, plan->kernel_volume, Cin, Cout, w16, w16t, fmt, stream_);
    if (rc) return rc;
  }
  return launch_gemm_tc2(plan, X16, Cin, w16t, Cout, 0, fmt, nullptr, bias, Y, stat_partials, (cudaStream_t)stream_);
}

/* Inference form of lg_conv_layer_forward: convolution -> eval-mode batch norm [-> + res] [-> ReLU] in one launch
 * (see include/lidog_b200.h). */
extern "C" int lg_conv_layer_infer(const lgConvPlan* plan, const void* X16, int32_t Cin, const float* W, int32_t Cout,
                                   void* w16, void* w16t, int32_t prep, int32_t fmt, const float* bn_stats,
                                   const float* res, int32_t relu, float* Y, void* Y16, void* stream_) {
  int rc = check_gemm(plan, Cin, Cout, fmt, "lg_conv_layer_infer");
  if (rc) return rc;
  LG_CHECK_ARG(X16 && w16t && Y && bn_stats && (!prep || (W && w16)), "lg_conv_layer_infer: null pointer");
  const auto misaligned = [](const void* p, uintptr_t a) { return ((uintptr_t)p & (a - 1)) != 0; };
  LG_CHECK_ARG(!misaligned(Y, 16) && !misaligned(bn_stats, 16) && !misaligned(res, 16) && !misaligned(Y16, 8),
               "lg_conv_layer_infer: Y, bn_stats and res must be 16-byte aligned, Y16 8-byte aligned");
  if (v2::gemm2_n_blk(Cout) % 32 != 0) {
    set_error("lg_conv_layer_infer: Cout=%d gives column blocks that are not multiples of 32", Cout);
    return LG_ERR_UNSUPPORTED;
  }
  if (prep) {
    rc = lg_prep_weights(W, plan->kernel_volume, Cin, Cout, w16, w16t, fmt, stream_);
    if (rc) return rc;
  }
  v2::InferEpi e;
  e.scale = bn_stats + 2 * Cout;
  e.shift = bn_stats + 3 * Cout;
  e.res = res;
  e.Y16 = (uint16_t*)Y16;
  e.relu = relu ? 1 : 0;
  e.fmt = fmt;
  return launch_gemm_tc2(plan, X16, Cin, w16t, Cout, 0, fmt, nullptr, nullptr, Y, nullptr, (cudaStream_t)stream_, &e);
}

/* dgrad and wgrad of one MinkowskiConvolution in one host call; the split-K partials live in the library arena. */
extern "C" int lg_conv_layer_backward(const lgConvPlan* plan_dgrad, const lgConvPlan* plan_wgrad, int32_t flip_dgrad,
                                      const void* X16, int32_t Cin, const void* dY16, int32_t Cout, const void* w16,
                                      int32_t fmt, const float* inv_scale, float* dX, float* dW, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc;
  LG_CHECK_ARG(dY16, "lg_conv_layer_backward: null gradient");
  if (dX) {
    rc = check_gemm(plan_dgrad, Cout, Cin, fmt, "lg_conv_layer_backward(dgrad)");
    if (rc) return rc;
    LG_CHECK_ARG(w16, "lg_conv_layer_backward: null weights");
    rc = launch_gemm_tc2(plan_dgrad, dY16, Cout, w16, Cin, flip_dgrad, fmt, inv_scale, nullptr, dX, nullptr, stream);
    if (rc) return rc;
  }
  if (dW) {
    rc = check_wgrad(plan_wgrad, Cin, Cout, fmt, "lg_conv_layer_backward(wgrad)");
    if (rc) return rc;
    LG_CHECK_ARG(X16, "lg_conv_layer_backward: null operand");
    ArenaCursor ar;
    const size_t ws = wgrad_tc2_workspace(plan_wgrad, Cin, Cout);
    rc = arena_begin(stream, ws, &ar);
    if (rc) return rc;
    rc = launch_wgrad_tc2(plan_wgrad, X16, Cin, dY16, Cout, fmt, inv_scale, dW, arena_take(&ar, ws), stream);
    if (rc) return rc;
  }
  return LG_OK;
}
