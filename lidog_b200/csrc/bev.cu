// Fused point-to-BEV projection (forward + backward).
// Reference: MinkUNetBaseBEV.sparse2super + filter_bounds, utils/models/minkunet_bev.py:158-230 --
// scatter of voxel features into a dense (H, W, C) image, a raw re-view of that memory as (C, H, W)
// and MaxPool2d(5, 3, 1).  The dense tensor (1.5 GB per sample at H = W = 2000, C = 96) is never
// materialised: a pixel -> row map (4 B per pixel) is built by one scatter, then one CTA per output
// row (b, c', i) rebuilds the pk scrambled input rows it needs in shared memory -- in flat terms
// they are ONE contiguous run of pk*W floats of the dense buffer, i.e. a run of ~pk*W/C consecutive
// pixels -- and reduces them.  Output rows are written exactly once, coalesced, without atomics;
// rows whose pixel run is empty are stored as zeros without touching the features.
// Pixel maths replicates the reference's three separately rounded float32 operations.
//
// Round 2 (ncu, profiles/r02_a_ncu_bev.txt): both pooling kernels were INSTRUCTION-bound, not memory-bound -- 1.2 G warp
// instructions for 42 k tiles (28 k per tile): every tile looked up 832 pixel runs one 4-byte load at a time, walked
// all 256 (channel, row) lines and moved its 8 192 results with scalar shared / global accesses although ~90 % of
// the lines pool zeros only.  Now an occupancy word per scrambled row (`rowbits`, built by one scatter over the
// voxels: bit jt = "this row holds a voxel inside tile column block jt") answers the emptiness question with 32
// coalesced loads per tile, only occupied rows touch the pixel map, only non-empty lines are scanned, and tiles move
// as float4.  While it scans, the forward records the winning cell of every window that can hold a voxel in a
// one-byte-per-window table (`argpos`).  The backward is one pass over the voxel rows, a warp per row and a lane per
// channel: each (row, channel) cell adds up the <= ceil(pk/ps)^2 windows the table says it won, in ascending (i, j)
// order -- the order of torch's CPU max_pool2d backward, so the gradient is reproduced bit for bit -- and every element
// of the gradient is written by exactly one thread: no atomics, no memset, run-to-run deterministic.
// Geometry envelope (bev_check): 1 <= pk <= 15 (a window position fits the table's byte with 255 to spare),
// 1 <= ps <= 16, 0 <= 2 pp <= pk, any C, H, W within int32 flat indices.  The tile height follows from ps so that a
// tile's scrambled rows fit one 32-bit row mask, and images wider than 32 tile column blocks share one occupancy bit
// between neighbouring blocks.
#include "common.cuh"

namespace lg {

struct BevWorkspace {
  int* pix_of_row;  // [n]      flat pixel (b*H*W + py*W + px) or -1
  int* next;        // [n]      chain of rows sharing a pixel (LG_BEV_MAX)
  int* pixmap;      // [B*H*W]  winner row (LAST) / chain head (MAX) / -1
  uint32_t* rowbits;  // [B*C*H]  bit jt >> grp_shift: scrambled row (c', h') holds a voxel inside tile column block jt
  unsigned char* argpos;  // [B*C*h_out*w_out] winning cell of a window ((h - h0) * pk + w - w0; 255 = an empty cell);
                          // written only for the (c', i) lines that can hold a voxel, which every voxel's window is on
  size_t total;
};

static BevWorkspace carve_bev(void* base, int64_t n, int64_t pixels, int64_t rows, int64_t windows) {
  BevWorkspace w;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    void* p = base ? (char*)base + off : nullptr;
    off += (bytes + 255) & ~(size_t)255;
    return p;
  };
  w.pix_of_row = (int*)take(sizeof(int) * (size_t)(n > 0 ? n : 1));
  w.next = (int*)take(sizeof(int) * (size_t)(n > 0 ? n : 1));
  w.pixmap = (int*)take(sizeof(int) * (size_t)pixels);
  w.rowbits = (uint32_t*)take(sizeof(uint32_t) * (size_t)rows);
  w.argpos = (unsigned char*)take((size_t)windows);
  w.total = off;
  return w;
}

__global__ void __launch_bounds__(256)
    k_bev_pixels(const int4* __restrict__ coords, int64_t n, int batch_size, float bound, float vs, int H, int W,
                 int policy, int* __restrict__ pix_of_row, int* __restrict__ next, int* __restrict__ pixmap) {
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int4 c = coords[r];
  const float lo = -bound, hi = bound;
  const float x = __fmul_rn((float)c.y, vs), y = __fmul_rn((float)c.z, vs);
  int pix = -1;
  if ((unsigned)c.x < (unsigned)batch_size && lo < x && x < hi && lo < y && y < hi) {
    int px = (int)floorf(__fdiv_rn(__fsub_rn(x, lo), vs));
    int py = (int)floorf(__fsub_rn((float)H, __fdiv_rn(__fsub_rn(y, lo), vs))) - 1;
    if (py < 0) py += H;  // python negative-index wrap
    if (px >= 0 && px < W && py >= 0 && py < H) pix = (c.x * H + py) * W + px;
  }
  pix_of_row[r] = pix;
  next[r] = -1;
  if (pix >= 0) {
    if (policy == LG_BEV_LAST)
      atomicMax(&pixmap[pix], (int)r);
    else
      next[r] = atomicExch(&pixmap[pix], (int)r);
  }
}

// Occupancy of the scrambled rows.  Voxel row r sits at pixel pix; its C channels are the dense cells
// m = pix_local * C .. + C - 1, i.e. a run inside scrambled row R = m / W (R = c' * H + h') that may continue on the next
// row.  For every piece of the run the bits of the tile column blocks whose cell range contains it are set
// (block jt covers cells jt * bw - pp <= w < jt * bw - pp + cover).
__global__ void __launch_bounds__(256)
    k_bev_rowbits(const int* __restrict__ pix_of_row, int64_t n, int C, int H, int W, int bw, int cover, int pp, int n_jc,
                  uint32_t* __restrict__ rowbits) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int pix = pix_of_row[r];
  if (pix < 0) return;
  const int hw = H * W;
  const int b = pix / hw;
  int m = (pix - b * hw) * C;
  const int m_end = m + C;
  while (m < m_end) {
    const int R = m / W, wa = m - R * W;
    const int len = min(m_end - m, W - wa), wb = wa + len - 1;
    int jt_lo = wa + pp - cover + 1;
    jt_lo = jt_lo <= 0 ? 0 : (jt_lo + bw - 1) / bw;
    const int jt_hi = min(n_jc - 1, (wb + pp) / bw);
    if (jt_lo <= jt_hi) {
      const uint32_t bits = (jt_hi - jt_lo == 31) ? 0xffffffffu : (((1u << (jt_hi - jt_lo + 1)) - 1u) << jt_lo);
      atomicOr(&rowbits[(int64_t)b * C * H + R], bits);
    }
    m += len;
  }
}

// value of dense cell (pixel p, channel ch): LAST -> winner row, MAX -> max over the chain
__device__ __forceinline__ float cell_value(int head, int ch, int C, int policy, const float* __restrict__ feats,
                                            const int* __restrict__ next) {
  if (head < 0) return 0.f;
  float v = __ldg(feats + (int64_t)head * C + ch);
  if (policy == LG_BEV_MAX) {
    for (int r = next[head]; r >= 0; r = next[r]) v = fmaxf(v, __ldg(feats + (int64_t)r * C + ch));
  }
  return v;
}

// first (smallest) row of the chain attaining the max for channel ch
__device__ __forceinline__ int cell_argrow(int head, int ch, int C, int policy, const float* __restrict__ feats,
                                           const int* __restrict__ next) {
  if (policy == LG_BEV_LAST || head < 0) return head;
  float best = __ldg(feats + (int64_t)head * C + ch);
  int arg = head;
  for (int r = next[head]; r >= 0; r = next[r]) {
    const float v = __ldg(feats + (int64_t)r * C + ch);
    if (v > best || (v == best && r < arg)) {
      best = v;
      arg = r;
    }
  }
  return arg;
}

// ---------------------------------------------------------------------------------------------
// Tiled pooling.  A CTA owns the output tile (b, 32 scrambled channels c', ib <= kIB rows i, kJC columns j); ib is the
// largest height whose (ib - 1) * ps + pk scrambled rows fit the 32-bit row mask (bev_tile_rows).
// Per (c', h') the cells of its windows are one contiguous run of <= (kJC-1)*ps+pk floats of the
// never-materialised dense buffer, i.e. a handful of consecutive PIXELS, and only ~1-2 % of the pixels
// hold a voxel.  Phase 1 reads one occupancy word per scrambled row (`rowbits`) and looks up the pixels of
// the occupied rows only (pixel -> row heads in shared memory).  Phase 2 evaluates the windows of the
// non-empty (c', i) lines in the reference's scan order (empty cells are zeros; occupied cells read their
// feature value).  Results are staged in shared memory (zero-initialised) and leave as float4 in NHWC
// (channels_last, what cuDNN's tensor-op convolutions consume) or coalesced rows in NCHW.
// No atomics; every output is written exactly once.
constexpr int kCG = 32;   // scrambled channels per CTA
constexpr int kIB = 8;    // most output rows per CTA (collect_lines: 32 channels x 8 rows = 256 threads)
constexpr int kJC = 32;   // output columns per CTA
constexpr int kPitch = kCG + 4;  // floats per staged (i, j) cell group: float4-aligned, conflict-free 128-bit reads

struct TileGeom {
  int b, c0, i0, j0;  // sample, first scrambled channel, first window row / column handled
  int ncg, nib, njc;  // valid extents
  int h_lo, h_hi, w_lo, w_hi;  // cell region (clipped to the image), hi exclusive
  int jt;                      // tile column block
  uint32_t jbits;              // rowbits bit that covers the cell columns of this tile (block group jt >> grp_shift)
};

__device__ __forceinline__ void cell_region(TileGeom& g, int H, int W, int pk, int ps, int pp) {
  g.h_lo = max(g.i0 * ps - pp, 0);
  g.h_hi = min((g.i0 + g.nib - 1) * ps - pp + pk, H);
  g.w_lo = max(g.j0 * ps - pp, 0);
  g.w_hi = min((g.j0 + g.njc - 1) * ps - pp + pk, W);
}

__device__ __forceinline__ TileGeom tile_geom(int C, int H, int W, int h_out, int w_out, int pk, int ps, int pp, int ib,
                                              int grp_shift) {
  TileGeom g;
  const int n_jc = (w_out + kJC - 1) / kJC, n_ib = (h_out + ib - 1) / ib, n_cg = (C + kCG - 1) / kCG;
  int idx = blockIdx.x;
  g.jt = idx % n_jc;
  g.j0 = g.jt * kJC;
  idx /= n_jc;
  g.i0 = (idx % n_ib) * ib;
  idx /= n_ib;
  g.c0 = (idx % n_cg) * kCG;
  g.b = idx / n_cg;
  g.ncg = min(kCG, C - g.c0);
  g.nib = min(ib, h_out - g.i0);
  g.njc = min(kJC, w_out - g.j0);
  g.jbits = 1u << (g.jt >> grp_shift);
  cell_region(g, H, W, pk, ps, pp);
  return g;
}

struct TileSmem {
  float* out;         // staged results: [rows][cols][kPitch]
  int* heads;         // [pairs][max_pix] pixel -> row head (or -1); valid for rows whose rowmask bit is set
  int* plo;           // [pairs] first pixel of the run
  uint32_t* rowmask;  // [kCG] bit (h - h_lo): scrambled row h of channel c' holds a voxel
  unsigned short* lines;  // non-empty (c', i) lines of the tile: (cl << 8) | il; *n_lines = their count
  int* n_lines;
};

// Phase 1.  Returns false (uniformly) when no pixel of the tile is occupied.  One coalesced rowbits load per
// scrambled channel (lane = scrambled row; nrows <= 32 by the choice of the tile height); only rows whose occupancy bit
// is set go to the pixel map.
__device__ __forceinline__ bool tile_lookup(const TileGeom& g, const TileSmem& t, int C, int H, int W, int max_pix,
                                            const int* __restrict__ pixmap, const uint32_t* __restrict__ rowbits) {
  const int nrows = g.h_hi - g.h_lo;
  const int* pm = pixmap + (int64_t)g.b * H * W;
  const uint32_t* rb = rowbits + (int64_t)g.b * C * H;
  int any = 0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int cl = warp; cl < g.ncg; cl += nwarps) {
    const int hr = lane;
    int row_any = 0;
    if (hr < nrows && (__ldg(rb + (g.c0 + cl) * H + g.h_lo + hr) & g.jbits)) {
      const int q = cl * nrows + hr;
      const int m_lo = ((g.c0 + cl) * H + g.h_lo + hr) * W + g.w_lo, m_hi = m_lo + (g.w_hi - g.w_lo);
      const int p_lo = m_lo / C, p_hi = (m_hi - 1) / C;
      t.plo[q] = p_lo;
      for (int d = 0; d < max_pix; ++d) {
        const int head = (p_lo + d <= p_hi) ? __ldg(pm + p_lo + d) : -1;
        t.heads[q * max_pix + d] = head;
        if (head >= 0) row_any = 1;
      }
    }
    const uint32_t bits = __ballot_sync(0xffffffffu, row_any);
    if (lane == 0) t.rowmask[cl] = bits;
    any |= (bits != 0);
  }
  return __syncthreads_or(any) != 0;
}

// Scan of one window in the reference's order (rows, then columns; strict > keeps the first maximum).
// Returns the pooled value; *pos = position (h - h0) * pk + (w - w0) of the winning cell inside the window, 255 when
// an empty cell (a zero) wins.
__device__ __forceinline__ float window_scan(const TileGeom& g, const TileSmem& t, int cl, int i, int j, int C, int H,
                                             int W, int pk, int ps, int pp, int max_pix, int policy,
                                             const float* __restrict__ feats, const int* __restrict__ next, int* pos) {
  const int nrows = g.h_hi - g.h_lo;
  const int h0 = i * ps - pp, w0 = j * ps - pp;
  const int ha = max(h0, 0), hb = min(h0 + pk, H), wa = max(w0, 0), wb = min(w0 + pk, W);
  const uint32_t rbits = (t.rowmask[cl] >> (ha - g.h_lo)) & ((1u << (hb - ha)) - 1u);
  *pos = 255;
  if (!rbits) return 0.f;  // every cell is an empty zero; the first one wins
  float best = -INFINITY;
  for (int h = ha; h < hb; ++h) {
    if (!((rbits >> (h - ha)) & 1u)) {  // an all-empty row: zeros
      if (0.f > best) {
        best = 0.f;
        *pos = 255;
      }
      continue;
    }
    const int q = cl * nrows + (h - g.h_lo);
    const int p_lo = t.plo[q];
    const int x0 = ((g.c0 + cl) * H + h) * W - p_lo * C;  // flat index of column 0 relative to pixel p_lo
    int ch = x0 + wa, d = 0;
    while (ch >= C) {  // <= max_pix - 1 steps, once per row
      ch -= C;
      ++d;
    }
    for (int w = wa; w < wb;) {  // the <= pk cells of this row lie in <= ceil(pk / C) + 1 pixels: one head test each
      const int span = min(wb - w, C - ch);
      const int head = t.heads[q * max_pix + d];
      if (head < 0) {  // a run of empty zeros; only its first cell can take the lead
        if (0.f > best) {
          best = 0.f;
          *pos = 255;
        }
      } else {
        for (int k = 0; k < span; ++k) {
          const float v = cell_value(head, ch + k, C, policy, feats, next);
          if (v > best) {
            best = v;
            *pos = (h - h0) * pk + (w + k - w0);
          }
        }
      }
      w += span;
      ch = 0;
      ++d;
    }
  }
  return best;
}

// staged tile <-> global.  NHWC with C % 4 == 0: one float4 = 4 scrambled channels of one output pixel (8 lanes cover
// the pixel's 128 bytes; the staging pitch keeps the 128-bit shared accesses conflict-free).  Otherwise a warp moves
// one 32-element line per iteration (NHWC: lane = c'; NCHW: lane = column).  `rows` x `cols` windows starting at
// (i_first, j_first); staged cell (il, jl) sits at (il * cols_pitch + jl) * kPitch.
template <bool STORE>
__device__ __forceinline__ void tile_transfer(const TileGeom& g, float* s_out, float* gptr, int layout, int C, int h_out,
                                              int w_out, int i_first, int j_first, int rows, int cols, int cols_pitch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  if (layout && (C & 3) == 0) {
    // thread = (column jl0 = tid / 8, float4 part = tid % 8); rows and the 33rd halo column are walked by loops --
    // the flat-index form of this loop spent ~30 instructions per element on divisions by a run-time column count and
    // was 60 % of all instructions of both pooling kernels (profiles/r02_b_ncu_bev.txt)
    const int parts = g.ncg >> 2;  // float4 per pixel (ncg is a multiple of 4 when C is)
    const int part = threadIdx.x & 7;
    if (part < parts) {
      for (int il = 0; il < rows; ++il) {
        float* grow = gptr + (((int64_t)g.b * h_out + i_first + il) * w_out + j_first) * C + g.c0 + 4 * part;
        float* srow = s_out + il * cols_pitch * kPitch + 4 * part;
        for (int jl = threadIdx.x >> 3; jl < cols; jl += 32) {
          float4* ge = reinterpret_cast<float4*>(grow + (int64_t)jl * C);
          float4* se = reinterpret_cast<float4*>(srow + jl * kPitch);
          if (STORE)
            *ge = *se;
          else
            *se = *ge;
        }
      }
    }
  } else if (layout) {  // NHWC, odd channel count: line = (il, jl), lane = c'
    if (lane >= g.ncg) return;
    for (int il = 0; il < rows; ++il)
      for (int jl = warp; jl < cols; jl += nwarps) {
        float* ge = gptr + (((int64_t)g.b * h_out + i_first + il) * w_out + j_first + jl) * C + g.c0 + lane;
        float* se = s_out + (il * cols_pitch + jl) * kPitch + lane;
        if (STORE)
          *ge = *se;
        else
          *se = *ge;
      }
  } else {  // NCHW: line = (c', il), lanes = columns
    for (int cl = warp; cl < g.ncg; cl += nwarps)
      for (int il = 0; il < rows; ++il)
      for (int jl = lane; jl < cols; jl += 32) {
        float* ge = gptr + (((int64_t)g.b * C + g.c0 + cl) * h_out + i_first + il) * w_out + j_first + jl;
        float* se = s_out + (il * cols_pitch + jl) * kPitch + cl;
        if (STORE)
          *ge = *se;
        else
          *se = *ge;
      }
  }
}

// bit h - ha of the result: scrambled row h of window row i (channel c') holds a voxel; 0 = every window of this
// (c', i) line pools zeros only.  Independent of the column, so a warp tests it once for its 32 windows.
__device__ __forceinline__ uint32_t line_row_bits(const TileGeom& g, const TileSmem& t, int cl, int i, int H, int pk,
                                                  int ps, int pp) {
  const int h0 = i * ps - pp;
  const int ha = max(h0, 0), hb = min(h0 + pk, H);
  return (t.rowmask[cl] >> (ha - g.h_lo)) & ((1u << (hb - ha)) - 1u);
}

// The lines whose windows can hold a voxel, collected so that ALL warps share them: a voxel occupies one scrambled
// channel, so the non-empty lines of a tile belong to a few c' -- with one warp per c' most warps idled at the barrier.
// `*t.n_lines` must be zero on entry; every thread of the CTA calls this.
__device__ __forceinline__ void collect_lines(const TileGeom& g, const TileSmem& t, int H, int pk, int ps, int pp) {
  const int cl = threadIdx.x >> 3, il = threadIdx.x & 7;
  if (cl < g.ncg && il < g.nib && line_row_bits(g, t, cl, g.i0 + il, H, pk, ps, pp))
    t.lines[atomicAdd(t.n_lines, 1)] = (unsigned short)((cl << 8) | il);
  __syncthreads();
}

// 4 blocks per SM: what the bench shape's ~51 KB of shared memory allows anyway; the register budget that follows
// (64) keeps ptxas from spilling, which it did at its own choice of 48 registers
__global__ void __launch_bounds__(256, 4)
    k_bev_pool_fwd(const float* __restrict__ feats, const int* __restrict__ next, const int* __restrict__ pixmap,
                   const uint32_t* __restrict__ rowbits, int C, int H, int W, int h_out, int w_out, int pk, int ps,
                   int pp, int policy, int layout, int ib, int grp_shift, int max_pix, int pairs_cap,
                   float* __restrict__ out, unsigned char* __restrict__ argpos) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  TileSmem t;
  t.out = reinterpret_cast<float*>(s_dyn);
  t.heads = reinterpret_cast<int*>(t.out + kIB * kJC * kPitch);
  t.plo = t.heads + pairs_cap * max_pix;
  t.rowmask = reinterpret_cast<uint32_t*>(t.plo + pairs_cap);
  t.n_lines = reinterpret_cast<int*>(t.rowmask + kCG);
  t.lines = reinterpret_cast<unsigned short*>(t.n_lines + 1);
  const TileGeom g = tile_geom(C, H, W, h_out, w_out, pk, ps, pp, ib, grp_shift);
  {  // zero the staged tile: most lines pool zeros only and are never touched again
    float4* o4 = reinterpret_cast<float4*>(t.out);
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int u = threadIdx.x; u < kIB * kJC * kPitch / 4; u += blockDim.x) o4[u] = z;
    if (threadIdx.x == 0) *t.n_lines = 0;
  }
  if (tile_lookup(g, t, C, H, W, max_pix, pixmap, rowbits)) {
    collect_lines(g, t, H, pk, ps, pp);
    // a warp takes one non-empty (c', i) line at a time, lane = column: the 32 windows of a line share their
    // scrambled rows and neighbouring lanes read neighbouring cells (and write neighbouring bytes of argpos)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_lines = *t.n_lines;
    for (int e = warp; e < n_lines; e += 8) {
      const int cl = t.lines[e] >> 8, il = t.lines[e] & 255;
      if (lane < g.njc) {
        int pos;
        t.out[(il * kJC + lane) * kPitch + cl] = window_scan(g, t, cl, g.i0 + il, g.j0 + lane, C, H, W, pk, ps, pp,
                                                             max_pix, policy, feats, next, &pos);
        argpos[(((int64_t)g.b * C + g.c0 + cl) * h_out + g.i0 + il) * w_out + g.j0 + lane] = (unsigned char)pos;
      }
    }
    __syncthreads();
  }
  tile_transfer<true>(g, t.out, out, layout, C, h_out, w_out, g.i0, g.j0, g.nib, g.njc, kJC);
}

// Backward.  The gradient of a window goes to its first arg-max in scan order (max_pool2d backward) if that cell
// holds a voxel; the forward left the cell's position in `argpos`.  A warp owns one voxel row, lane = channel, so the
// row's writes are coalesced.  The row's cell (c', h, w) sits in the windows i in [ceil((h + pp - pk + 1) / ps),
// floor((h + pp) / ps)] (clipped to the output), likewise for j, and adds up those whose table entry names it in
// ascending (i, j) order -- the order of torch's CPU max_pool2d backward, so the gradient is bit-equal to it.
// LAST: every row of the pixel computes the same sum (index_put_ backward hands the pixel's gradient to each row that
// wrote it); MAX: only the chain's first row attaining the cell's max receives it.  Every element of grad_feats is
// written exactly once, rows outside the image with 0: no memset, no atomics.
// The pass is latency-bound (each row waits on its pixel, then its table bytes, then its gradient reads), so loads
// are issued in groups.  WIDE = false (pk <= 2 ps: at most 2 x 2 windows per cell): kU channels' windows unrolled
// together.  WIDE = true (up to 15 x 15 windows): one channel at a time, its windows in groups of kG.
template <bool WIDE>
__global__ void __launch_bounds__(256)
    k_bev_pool_bwd(const float* __restrict__ feats, const int* __restrict__ pix_of_row, const int* __restrict__ next,
                   const int* __restrict__ pixmap, const unsigned char* __restrict__ argpos, int64_t n, int C, int H,
                   int W, int h_out, int w_out, int pk, int ps, int pp, int policy, int layout,
                   const float* __restrict__ grad_out, float* __restrict__ grad_feats) {
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n) return;
  const int lane = threadIdx.x & 31;
  float* gf = grad_feats + r * C;
  const int pix = __ldg(pix_of_row + r);
  if (pix < 0) {
    for (int ch = lane; ch < C; ch += 32) gf[ch] = 0.f;
    return;
  }
  const int hw = H * W, b = pix / hw;
  const int head = policy == LG_BEV_MAX ? __ldg(pixmap + pix) : -1;
  const int m0 = (pix - b * hw) * C;  // flat index of the row's first cell in the sample's dense buffer
  const int64_t sample = (int64_t)b * C * h_out * w_out;  // C * h_out * w_out < 2^31 (host-checked)
  const unsigned char* tab = argpos + sample;
  const float* go = grad_out + sample;
  if constexpr (!WIDE) {
    // kU channels per lane at a time, unrolled, so that their table reads and then their gradient reads are in flight
    // together: one channel at a time left a chain of dependent loads per channel (0.77 ms at the bench shape).  3 takes
    // the bench's 96 channels in one pass (0.64 ms); 4 needs 68 registers, keeps fewer warps resident and measured
    // 0.80 ms (profiles/r05_bev_bench.jsonl).
    constexpr int kU = 3;
    for (int base = lane; base < C; base += 32 * kU) {
      bool hit[kU][4];
      int off[kU][4];
#pragma unroll
      for (int k = 0; k < kU; ++k) {
        const int ch = base + 32 * k;
#pragma unroll
        for (int q = 0; q < 4; ++q) hit[k][q] = false, off[k][q] = 0;
        if (ch < C && (policy == LG_BEV_LAST || cell_argrow(head, ch, C, policy, feats, next) == (int)r)) {
          // scrambled cell (c', h, w): the (H, W, C) buffer re-viewed as (C, H, W); m < C * H * W < 2^31 (host-checked)
          const int m = m0 + ch, c = m / hw, h = (m - c * hw) / W, w = m - c * hw - h * W;
          // window rows containing h: qi - 1 (h at row offset ri + ps) and qi (offset ri), where it lies inside them
          const int qi = (unsigned)(h + pp) / (unsigned)ps, ri = h + pp - qi * ps;
          const int qj = (unsigned)(w + pp) / (unsigned)ps, rj = w + pp - qj * ps;
#pragma unroll
          for (int q = 0; q < 4; ++q) {  // ascending (i, j)
            const int di = 1 - (q >> 1), dj = 1 - (q & 1);
            const int i = qi - di, j = qj - dj, oh = ri + di * ps, ow = rj + dj * ps;
            if (i >= 0 && i < h_out && oh < pk && j >= 0 && j < w_out && ow < pk) {
              const int t = (c * h_out + i) * w_out + j;
              hit[k][q] = __ldg(tab + t) == oh * pk + ow;
              off[k][q] = layout ? (i * w_out + j) * C + c : t;
            }
          }
        }
      }
#pragma unroll
      for (int k = 0; k < kU; ++k) {
        const int ch = base + 32 * k;
        float sum = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (hit[k][q]) sum += __ldg(go + off[k][q]);
        if (ch < C) gf[ch] = sum;
      }
    }
  } else {
    // the cell's ni x nj windows, flattened in ascending (i, j) order, kG at a time: their table bytes, then the
    // gradients of the hits, are in flight together
    constexpr int kG = 8;
    for (int ch = lane; ch < C; ch += 32) {
      float sum = 0.f;
      if (policy == LG_BEV_LAST || cell_argrow(head, ch, C, policy, feats, next) == (int)r) {
        const int m = m0 + ch, c = m / hw, h = (m - c * hw) / W, w = m - c * hw - h * W;
        const int i_lo = max(h + pp - pk + 1 + ps - 1, 0) / ps, i_hi = min((h + pp) / ps, h_out - 1);
        const int j_lo = max(w + pp - pk + 1 + ps - 1, 0) / ps, j_hi = min((w + pp) / ps, w_out - 1);
        const int nj = j_hi - j_lo + 1, nwin = i_lo <= i_hi && j_lo <= j_hi ? (i_hi - i_lo + 1) * nj : 0;
        for (int t0 = 0; t0 < nwin; t0 += kG) {
          bool hit[kG];
          int off[kG];
#pragma unroll
          for (int k = 0; k < kG; ++k) {
            hit[k] = false;
            off[k] = 0;
            if (t0 + k < nwin) {
              const int i = i_lo + (t0 + k) / nj, j = j_lo + (t0 + k) % nj;
              const int t = (c * h_out + i) * w_out + j;
              hit[k] = __ldg(tab + t) == (h + pp - i * ps) * pk + (w + pp - j * ps);
              off[k] = layout ? (i * w_out + j) * C + c : t;
            }
          }
#pragma unroll
          for (int k = 0; k < kG; ++k)
            if (hit[k]) sum += __ldg(go + off[k]);
        }
      }
      gf[ch] = sum;
    }
  }
}

}  // namespace lg

using namespace lg;

// output rows per tile: the tile's (ib - 1) * ps + pk scrambled rows must fit the 32-bit row mask (>= 1 as pk <= 15)
static int bev_tile_rows(int pk, int ps) { const int r = (32 - pk) / ps + 1; return r < kIB ? r : kIB; }
// log2 of the tile column blocks per occupancy bit: a row's one 32-bit word covers images wider than 32 blocks
static int bev_col_shift(int w_out) {
  int s = 0;
  while ((32 << s) < ceil_div(w_out, kJC)) ++s;
  return s;
}
// a (c', h') run of a tile spans (cols-1)*ps+pk floats = at most this many pixels of C channels
static int bev_max_pix(int C, int pk, int ps, int cols) { return ((cols - 1) * ps + pk + C - 2) / C + 1; }
static int bev_pairs_cap(int C, int pk, int ps, int rows) { return (C < kCG ? C : kCG) * ((rows - 1) * ps + pk); }
static size_t bev_smem_fwd(int C, int pk, int ps) {  // staged tile + heads + first pixels + row masks
  const size_t pairs = bev_pairs_cap(C, pk, ps, bev_tile_rows(pk, ps));
  return sizeof(float) * kIB * kJC * kPitch + sizeof(int) * pairs * (bev_max_pix(C, pk, ps, kJC) + 1) + sizeof(int) * kCG +
         sizeof(int) + 2 * kCG * kIB + 16;
}
static int64_t bev_tiles(int B, int C, int h_out, int w_out, int ib) {
  return (int64_t)B * ceil_div(C, kCG) * ceil_div(h_out, ib) * ceil_div(w_out, kJC);
}
// pooling windows of the output (entries of the argpos table); 0 for parameters bev_check rejects
static int64_t bev_windows(int B, int C, int H, int W, int pk, int ps, int pp) {
  if (B < 1 || C < 1 || ps < 1 || H + 2 * pp < pk || W + 2 * pp < pk) return 0;
  const int64_t h_out = (H + 2 * pp - pk) / ps + 1, w_out = (W + 2 * pp - pk) / ps + 1;
  return (int64_t)B * C * h_out * w_out;
}

static int bev_check(int64_t n, int C, int B, int H, int W, int pk, int ps, int pp, int policy, const char* who) {
  LG_CHECK_ARG(n >= 0 && C >= 1 && B >= 1 && H >= 1 && W >= 1, "%s: bad sizes", who);
  LG_CHECK_ARG(pk >= 1 && pk <= 15, "%s: pool kernel %d outside 1..15 (the one-byte argpos table)", who, pk);
  LG_CHECK_ARG(ps >= 1 && ps <= 16, "%s: pool stride %d outside 1..16", who, ps);
  LG_CHECK_ARG(pp >= 0 && 2 * pp <= pk, "%s: pool padding %d outside 0..pk/2", who, pp);
  LG_CHECK_ARG(H + 2 * pp >= pk && W + 2 * pp >= pk, "%s: image smaller than the pool window (h_out, w_out < 1)", who);
  LG_CHECK_ARG(policy == LG_BEV_LAST || policy == LG_BEV_MAX, "%s: bad policy", who);
  LG_CHECK_ARG((int64_t)B * H * W < ((int64_t)1 << 31), "%s: batch*H*W exceeds int32", who);
  LG_CHECK_ARG((int64_t)C * H * W < ((int64_t)1 << 31), "%s: C*H*W exceeds int32", who);
  const int h_out = (H + 2 * pp - pk) / ps + 1, w_out = (W + 2 * pp - pk) / ps + 1;
  LG_CHECK_ARG((int64_t)C * h_out * w_out < ((int64_t)1 << 31), "%s: C*h_out*w_out exceeds int32", who);
  // never fires inside the envelope above (at most 108 KB, at C = 31, pk = 15, ps = 16); guards the launch below
  LG_CHECK_ARG(bev_smem_fwd(C, pk, ps) <= 200 * 1024, "%s: forward tile needs more than 200 KB of shared memory", who);
  return LG_OK;
}

extern "C" size_t lg_bev_workspace(int64_t n, int32_t C, int32_t batch_size, int32_t H, int32_t W, int32_t pk,
                                   int32_t ps, int32_t pp) {
  const int64_t windows = bev_windows(batch_size, C, H, W, pk, ps, pp);
  return carve_bev(nullptr, n, (int64_t)batch_size * H * W, (int64_t)batch_size * C * H, windows).total;
}

extern "C" int lg_bev_forward(const int32_t* coords4, const float* feats, int64_t n, int32_t C, int32_t batch_size,
                              float bound, float voxel_size, int32_t H, int32_t W, int32_t pk, int32_t ps, int32_t pp,
                              int32_t policy, int32_t layout, float* out, void* workspace, size_t workspace_bytes,
                              void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = bev_check(n, C, batch_size, H, W, pk, ps, pp, policy, "lg_bev_forward");
  if (rc) return rc;
  const int64_t pixels = (int64_t)batch_size * H * W, rows = (int64_t)batch_size * C * H;
  BevWorkspace w = carve_bev(workspace, n, pixels, rows, bev_windows(batch_size, C, H, W, pk, ps, pp));
  LG_CHECK_ARG(workspace && workspace_bytes >= w.total, "lg_bev_forward: workspace too small");
  LG_CHECK_ARG(out && (n == 0 || (coords4 && feats)), "lg_bev_forward: null pointer");
  LG_CHECK_ARG(layout == 0 || layout == 1, "lg_bev_forward: layout must be 0 (NCHW) or 1 (NHWC)");
  LG_CHECK_ARG(((uintptr_t)out & 15) == 0, "lg_bev_forward: out must be 16-byte aligned");
  const int h_out = (H + 2 * pp - pk) / ps + 1, w_out = (W + 2 * pp - pk) / ps + 1;
  const int ib = bev_tile_rows(pk, ps), grp_shift = bev_col_shift(w_out), grp = 1 << grp_shift;
  LG_CUDA_OK(cudaMemsetAsync(w.pixmap, 0xFF, sizeof(int) * (size_t)pixels, stream));
  LG_CUDA_OK(cudaMemsetAsync(w.rowbits, 0, sizeof(uint32_t) * (size_t)rows, stream));
  if (n > 0) {
    k_bev_pixels<<<(unsigned)ceil_div(n, 256), 256, 0, stream>>>((const int4*)coords4, n, batch_size, bound,
                                                                 voxel_size, H, W, policy, w.pix_of_row, w.next,
                                                                 w.pixmap);
    LG_LAUNCH_OK();
    // an occupancy bit stands for grp neighbouring tile column blocks
    k_bev_rowbits<<<(unsigned)ceil_div(n, 256), 256, 0, stream>>>(w.pix_of_row, n, C, H, W, grp * kJC * ps,
                                                                  (grp * kJC - 1) * ps + pk, pp,
                                                                  (int)ceil_div(ceil_div(w_out, kJC), grp), w.rowbits);
    LG_LAUNCH_OK();
  }
  const size_t smem = bev_smem_fwd(C, pk, ps);
  const int64_t blocks = bev_tiles(batch_size, C, h_out, w_out, ib);
  LG_CHECK_ARG(blocks < ((int64_t)1 << 31), "lg_bev_forward: too many output tiles");
  LG_CUDA_OK(cudaFuncSetAttribute(k_bev_pool_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_bev_pool_fwd<<<(unsigned)blocks, 256, smem, stream>>>(feats, w.next, w.pixmap, w.rowbits, C, H, W, h_out, w_out, pk,
                                                          ps, pp, policy, layout, ib, grp_shift,
                                                          bev_max_pix(C, pk, ps, kJC), bev_pairs_cap(C, pk, ps, ib), out,
                                                          w.argpos);
  LG_LAUNCH_OK();
  return LG_OK;
}

extern "C" int lg_bev_backward(const int32_t* coords4, const float* feats, int64_t n, int32_t C, int32_t batch_size,
                               int32_t H, int32_t W, int32_t pk, int32_t ps, int32_t pp, int32_t policy,
                               int32_t layout, const float* grad_out, float* grad_feats, const void* workspace,
                               size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = bev_check(n, C, batch_size, H, W, pk, ps, pp, policy, "lg_bev_backward");
  if (rc) return rc;
  const int64_t pixels = (int64_t)batch_size * H * W, rows = (int64_t)batch_size * C * H;
  BevWorkspace w = carve_bev(const_cast<void*>(workspace), n, pixels, rows, bev_windows(batch_size, C, H, W, pk, ps, pp));
  LG_CHECK_ARG(workspace && workspace_bytes >= w.total, "lg_bev_backward: workspace too small");
  if (n == 0) return LG_OK;
  LG_CHECK_ARG(feats && grad_out && grad_feats, "lg_bev_backward: null pointer");
  const int h_out = (H + 2 * pp - pk) / ps + 1, w_out = (W + 2 * pp - pk) / ps + 1;
  LG_CHECK_ARG(layout == 0 || layout == 1, "lg_bev_backward: layout must be 0 (NCHW) or 1 (NHWC)");
  const int64_t blocks = ceil_div(n, 8);  // a warp per voxel row
  LG_CHECK_ARG(blocks < ((int64_t)1 << 31), "lg_bev_backward: too many rows");
  // pk <= 2 ps: a cell lies in at most 2 x 2 windows, which the unrolled variant takes in one go
  auto kernel = pk <= 2 * ps ? k_bev_pool_bwd<false> : k_bev_pool_bwd<true>;
  kernel<<<(unsigned)blocks, 256, 0, stream>>>(feats, w.pix_of_row, w.next, w.pixmap, w.argpos, n, C, H, W, h_out, w_out,
                                               pk, ps, pp, policy, layout, grad_out, grad_feats);
  LG_LAUNCH_OK();
  return LG_OK;
}
