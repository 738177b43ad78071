// Kernel-map generation: neighbour tables by hash probes, per-tile offset masks, ME-format pair
// lists, and the k-sorted stride-2 "up" plan.  Reference contract: the kernel maps implied by every
// MinkowskiConvolution / MinkowskiConvolutionTranspose in utils/models/minkunet_bev.py:57-123,410-442
// (conventions: SURVEY.md Appendix C.7).  A warp owns 32 consecutive output voxels and walks the
// kernel offsets together, so nbr[k][o..o+31] is written coalesced and the tile mask falls out of a
// ballot; the table (16 B slots, load factor <= 0.5) stays L2-resident.
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"
#include "scan.cuh"

namespace lg {

constexpr int kMaxMaskWords = 4;  // K <= 128 (5^3 = 125)

__global__ void __launch_bounds__(LG_TILE_ROWS)
    k_neighbors(const HashSlot* __restrict__ table, unsigned long long mask, const int4* __restrict__ out_coords,
                int64_t n_out, int ksize, int scale, int row_offset, int K, int mask_words, int32_t* __restrict__ nbr,
                int64_t n_slots, uint32_t* __restrict__ tile_mask, uint32_t* __restrict__ row_mask,
                unsigned int* __restrict__ k_count) {
  __shared__ uint32_t s_mask[kMaxMaskWords];
  if (threadIdx.x < kMaxMaskWords) s_mask[threadIdx.x] = 0;
  __syncthreads();
  const int64_t o = (int64_t)blockIdx.x * LG_TILE_ROWS + threadIdx.x;
  const bool valid = o < n_out;
  int4 c = valid ? out_coords[o] : make_int4(0, 0, 0, 0);
  const int base = (ksize & 1) ? -(ksize / 2) : 0;
  uint32_t wmask[kMaxMaskWords] = {0, 0, 0, 0};
  uint32_t rmask = 0;  // this row's offsets (sorted plans only, K <= 32)
  // (Issuing the first probes of a whole kernel x-row together was tried: 64 instead of 32 registers halved the
  // occupancy and the 125-offset map went 567 -> 736 us.  ncu: 360 M warp instructions for 81 M probes -- the
  // kernel is issue-bound, so the instruction count per probe is what matters; see hash_key in common.cuh.)
  int k = 0;
  for (int iz = 0; iz < ksize; ++iz)
    for (int iy = 0; iy < ksize; ++iy)
      for (int ix = 0; ix < ksize; ++ix, ++k) {
        int r = -1;
        if (valid) {
          int x = c.y + (base + ix) * scale, y = c.z + (base + iy) * scale, z = c.w + (base + iz) * scale;
          if (coord_in_range(c.x, x, y, z)) r = hash_lookup(table, mask, pack_key(c.x, x, y, z));
          if (r >= 0) r -= row_offset;  // the table may index a larger set this one is a contiguous slice of
        }
        nbr[(int64_t)k * n_slots + o] = r;
        const uint32_t bal = __ballot_sync(0xffffffffu, r >= 0);
        if (bal) wmask[k >> 5] |= 1u << (k & 31);
        if (row_mask) {
          rmask |= (r >= 0 ? 1u : 0u) << (k & 31);
          if (bal && (threadIdx.x & 31) == 0) atomicAdd(&k_count[k], (unsigned)__popc(bal));
        }
      }
  if (row_mask) row_mask[o] = rmask;
  if ((threadIdx.x & 31) == 0) {
    for (int w = 0; w < mask_words; ++w)
      if (wmask[w]) atomicOr(&s_mask[w], wmask[w]);
  }
  __syncthreads();
  if (threadIdx.x < mask_words) tile_mask[(int64_t)blockIdx.x * mask_words + threadIdx.x] = s_mask[threadIdx.x];
}

// Same-set maps (odd kernel, output set == the set the table indexes): pair (k, o -> i) exists iff pair
// (K-1-k, i -> o) does, so only the first half of the offsets is probed and every hit also writes its mirror entry.
// k_neighbors is issue-bound on the probes (ncu: ~4.5 warp instructions per probe-lane), so half the probes is close
// to half the time; the mirror entries cost one scattered 4-byte store and an atomicOr on the tile / row masks per
// hit.  Requires: nbr[(K/2+1..K-1)][*] preset to -1, tile_mask and row_mask preset to 0 (the launcher does it).
// Every table entry is written exactly once with a value that does not depend on the schedule: deterministic.
__global__ void __launch_bounds__(LG_TILE_ROWS)
    k_neighbors_sym(const HashSlot* __restrict__ table, unsigned long long mask, const int4* __restrict__ out_coords,
                    int64_t n_out, int ksize, int scale, int row_offset, int K, int mask_words,
                    int32_t* __restrict__ nbr, int64_t n_slots, uint32_t* __restrict__ tile_mask,
                    uint32_t* __restrict__ row_mask, unsigned int* __restrict__ k_count) {
  __shared__ uint32_t s_mask[kMaxMaskWords];
  if (threadIdx.x < kMaxMaskWords) s_mask[threadIdx.x] = 0;
  __syncthreads();
  const int64_t o = (int64_t)blockIdx.x * LG_TILE_ROWS + threadIdx.x;
  const bool valid = o < n_out;
  const int4 c = valid ? out_coords[o] : make_int4(0, 0, 0, 0);
  const int base = -(ksize / 2), half = K / 2;
  uint32_t wmask[kMaxMaskWords] = {0, 0, 0, 0};
  uint32_t rmask = 0;
  int k = 0;
  for (int iz = 0; iz < ksize && k < half; ++iz)
    for (int iy = 0; iy < ksize && k < half; ++iy)
      for (int ix = 0; ix < ksize && k < half; ++ix, ++k) {
        int r = -1;
        if (valid) {
          const int x = c.y + (base + ix) * scale, y = c.z + (base + iy) * scale, z = c.w + (base + iz) * scale;
          if (coord_in_range(c.x, x, y, z)) r = hash_lookup(table, mask, pack_key(c.x, x, y, z));
          if (r >= 0) r -= row_offset;
        }
        nbr[(int64_t)k * n_slots + o] = r;
        const int km = K - 1 - k;
        if (r >= 0) {  // the mirror pair: voxel r sees o through offset K-1-k
          nbr[(int64_t)km * n_slots + r] = (int32_t)o;
          if (row_mask) {
            atomicOr(&row_mask[r], 1u << (km & 31));  // (mask-sorted plans rebuild the tile masks after the sort)
          } else {
            // one atomic per distinct tile of the warp's hits: consecutive voxels mostly hit consecutive rows
            const int tile = r / LG_TILE_ROWS;
            const unsigned peers = __match_any_sync(__activemask(), tile);
            if ((int)(__ffs(peers) - 1) == (int)(threadIdx.x & 31))
              atomicOr(&tile_mask[(int64_t)tile * mask_words + (km >> 5)], 1u << (km & 31));
          }
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, r >= 0);
        if (bal) wmask[k >> 5] |= 1u << (k & 31);
        if (row_mask) {
          rmask |= (r >= 0 ? 1u : 0u) << (k & 31);
          // (k_count of the mirror offset equals this one: k_sort_keys reads count[min(k, K-1-k)])
          if (bal && (threadIdx.x & 31) == 0) atomicAdd(&k_count[k], (unsigned)__popc(bal));
        }
      }
  // centre offset: the voxel itself
  nbr[(int64_t)half * n_slots + o] = valid ? (int32_t)o : -1;
  {
    const uint32_t bal = __ballot_sync(0xffffffffu, valid);
    if (bal) wmask[half >> 5] |= 1u << (half & 31);
    if (row_mask) {
      rmask |= (valid ? 1u : 0u) << (half & 31);
      if (bal && (threadIdx.x & 31) == 0) atomicAdd(&k_count[half], (unsigned)__popc(bal));
    }
  }
  if (row_mask && rmask) atomicOr(&row_mask[o], rmask);
  if ((threadIdx.x & 31) == 0) {
    for (int w = 0; w < mask_words; ++w)
      if (wmask[w]) atomicOr(&s_mask[w], wmask[w]);
  }
  __syncthreads();
  if (threadIdx.x < mask_words && s_mask[threadIdx.x])
    atomicOr(&tile_mask[(int64_t)blockIdx.x * mask_words + threadIdx.x], s_mask[threadIdx.x]);
}

static bool neighbors_symmetric(int same_set, int kernel_size) {
  return same_set && (kernel_size & 1) && kernel_size >= 3;
}

static int launch_neighbors(const void* table_in, int64_t capacity_in, const int32_t* out_coords4, int64_t n_out,
                            int kernel_size, int offset_scale, int row_offset, int same_set, int K, int words,
                            int32_t* nbr, int64_t n_slots, uint32_t* tile_mask, uint32_t* row_mask,
                            unsigned int* k_count, cudaStream_t stream) {
  const unsigned grid = (unsigned)(n_slots / LG_TILE_ROWS);
  if (neighbors_symmetric(same_set, kernel_size)) {
    const int half = K / 2;
    LG_CUDA_OK(cudaMemsetAsync(nbr + (int64_t)(half + 1) * n_slots, 0xFF, sizeof(int32_t) * (size_t)half * n_slots, stream));
    LG_CUDA_OK(cudaMemsetAsync(tile_mask, 0, sizeof(uint32_t) * (size_t)grid * words, stream));
    if (row_mask) LG_CUDA_OK(cudaMemsetAsync(row_mask, 0, sizeof(uint32_t) * (size_t)n_slots, stream));
    k_neighbors_sym<<<grid, LG_TILE_ROWS, 0, stream>>>((const HashSlot*)table_in, (unsigned long long)(capacity_in - 1),
                                                       (const int4*)out_coords4, n_out, kernel_size, offset_scale,
                                                       row_offset, K, words, nbr, n_slots, tile_mask, row_mask, k_count);
  } else {
    k_neighbors<<<grid, LG_TILE_ROWS, 0, stream>>>((const HashSlot*)table_in, (unsigned long long)(capacity_in - 1),
                                                   (const int4*)out_coords4, n_out, kernel_size, offset_scale, row_offset,
                                                   K, words, nbr, n_slots, tile_mask, row_mask, k_count);
  }
  LG_LAUNCH_OK();
  return LG_OK;
}

// ---- ME-format pair lists: flatten [K][n_slots], keep entries >= 0 (order = (k, out) ascending)
struct PairFlag {
  const int32_t* nbr;
  __device__ bool operator()(int64_t i) const { return nbr[i] >= 0; }
};
struct PairSink {
  const int32_t* nbr;
  int64_t n_slots;
  int32_t* in_rows;
  int32_t* out_rows;
  int64_t* k_offsets;
  __device__ void operator()(int64_t i, int prefix, bool f) const {
    const int64_t k = i / n_slots, o = i - k * n_slots;
    if (o == 0) k_offsets[k] = prefix;
    if (f) {
      in_rows[prefix] = nbr[i];
      out_rows[prefix] = (int32_t)o;
    }
  }
};

// ---- stride-2 "up" plan: fine rows grouped by child index
__device__ __forceinline__ int child_index(int4 c, int ts) {
  return (floor_div(c.y, ts) & 1) | ((floor_div(c.z, ts) & 1) << 1) | ((floor_div(c.w, ts) & 1) << 2);
}
struct ChildFlag {
  const int4* coords;
  int64_t n;
  int ts;
  __device__ bool operator()(int64_t i) const {
    const int64_t k = i / n, r = i - k * n;
    return child_index(coords[r], ts) == (int)k;
  }
};
struct ChildSink {  // pass 1: only the per-k starts
  int64_t n;
  int* k_start;  // [9]
  __device__ void operator()(int64_t i, int prefix, bool f) const {
    const int64_t k = i / n;
    if (i - k * n == 0) k_start[k] = prefix;
  }
};
struct ChildFill {
  const int64_t* parent;
  int64_t parent_offset;  // the parent ids index a larger set this coarse level is a contiguous slice of
  int64_t n;
  const int* k_start;      // [9] (k_start[8] = n)
  const int* k_slot_base;  // [9] padded segment starts
  int32_t* gather;
  int32_t* out_row;
  __device__ void operator()(int64_t i, int prefix, bool f) const {
    if (!f) return;
    const int64_t k = i / n, r = i - k * n;
    const int slot = k_slot_base[k] + (prefix - k_start[k]);
    gather[slot] = (int32_t)(parent[r] - parent_offset);
    out_row[slot] = (int32_t)r;
  }
};

__global__ void k_up2_layout(const int* k_start, int64_t n, int* k_slot_base, uint32_t* tile_mask, int64_t n_tiles_cap,
                             int64_t* slots_used) {
  // single thread: 8 segments
  int base = 0;
  for (int k = 0; k < 8; ++k) {
    int cnt = ((k == 7) ? (int)n : k_start[k + 1]) - k_start[k];
    k_slot_base[k] = base;
    int tiles = (cnt + LG_TILE_ROWS - 1) / LG_TILE_ROWS;
    for (int t = 0; t < tiles; ++t) {
      int64_t tile = base / LG_TILE_ROWS + t;
      if (tile < n_tiles_cap) tile_mask[tile] = 1u << k;
    }
    base += tiles * LG_TILE_ROWS;
  }
  k_slot_base[8] = base;
  *slots_used = base;
}

// ---- mask-sorted plans: rows with the same neighbour pattern share tiles
// Sort key of a row = its offset bits, the RAREST offset (smallest pair count, ties by k) most
// significant: rows that own an unusual neighbour end up together, so far fewer (tile, offset)
// units carry mostly-empty rows (measured on kitti-shaped scans: 0.29 -> 0.69 of the gathered rows real).
__global__ void k_sort_keys(const uint32_t* __restrict__ row_mask, const unsigned int* __restrict__ k_count, int K,
                            int64_t n, uint32_t* __restrict__ keys, int32_t* __restrict__ vals, int sym_counts) {
  __shared__ int s_pos[32];
  // sym_counts: only the first half of the offsets was counted (k_neighbors_sym); count[k] = count[K-1-k]
  auto cnt = [&](int k) { return k_count[sym_counts ? min(k, K - 1 - k) : k]; };
  if (threadIdx.x < 32) {
    const int k = threadIdx.x;
    int rank = 0;  // number of offsets rarer than k
    if (k < K) {
      const unsigned ck = cnt(k);
      for (int j = 0; j < K; ++j) {
        const unsigned cj = cnt(j);
        rank += (cj < ck || (cj == ck && j < k)) ? 1 : 0;
      }
    }
    s_pos[k] = K - 1 - rank;
  }
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t m = row_mask[i];
  uint32_t key = 0;
  for (int k = 0; k < K; ++k) key |= ((m >> k) & 1u) << s_pos[k];
  keys[i] = key;
  vals[i] = (int32_t)i;
}

__global__ void __launch_bounds__(LG_TILE_ROWS)
    k_permute_plan(const int32_t* __restrict__ nbr_nat, const int32_t* __restrict__ perm, int64_t n_out, int K,
                   int64_t n_slots, int32_t* __restrict__ nbr, int32_t* __restrict__ out_row,
                   uint32_t* __restrict__ tile_mask) {
  __shared__ uint32_t s_mask;
  if (threadIdx.x == 0) s_mask = 0;
  __syncthreads();
  const int64_t s = (int64_t)blockIdx.x * LG_TILE_ROWS + threadIdx.x;
  const int r = (s < n_out) ? perm[s] : -1;
  out_row[s] = r;
  uint32_t wmask = 0;
  for (int k = 0; k < K; ++k) {
    const int v = (r >= 0) ? nbr_nat[(int64_t)k * n_slots + r] : -1;
    nbr[(int64_t)k * n_slots + s] = v;
    if (__ballot_sync(0xffffffffu, v >= 0)) wmask |= 1u << k;
  }
  if ((threadIdx.x & 31) == 0 && wmask) atomicOr(&s_mask, wmask);
  __syncthreads();
  if (threadIdx.x == 0) tile_mask[blockIdx.x] = s_mask;
}

__global__ void k_fill_i32(int32_t* p, int64_t n, int32_t v) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

}  // namespace lg

using namespace lg;

extern "C" int lg_kernel_map(const void* table_in, int64_t capacity_in, const int32_t* out_coords4, int64_t n_out,
                             int32_t kernel_size, int32_t offset_scale, int32_t in_row_offset, int32_t same_set,
                             int32_t* nbr, int64_t n_slots, uint32_t* tile_mask, void* stream) {
  LG_CHECK_ARG(kernel_size >= 1 && kernel_size <= 5, "lg_kernel_map: kernel_size %d not in [1,5]", kernel_size);
  LG_CHECK_ARG(n_out >= 0 && n_slots == round_up(n_out, LG_TILE_ROWS), "lg_kernel_map: n_slots must be round_up(n_out,128)");
  LG_CHECK_ARG(capacity_in >= 1024 && (capacity_in & (capacity_in - 1)) == 0, "lg_kernel_map: bad capacity");
  if (n_out == 0) return LG_OK;
  LG_CHECK_ARG(table_in && out_coords4 && nbr && tile_mask, "lg_kernel_map: null pointer");
  const int K = kernel_size * kernel_size * kernel_size;
  const int words = (K + 31) / 32;
  return launch_neighbors(table_in, capacity_in, out_coords4, n_out, kernel_size, offset_scale, in_row_offset, same_set,
                          K, words, nbr, n_slots, tile_mask, nullptr, nullptr, (cudaStream_t)stream);
}

namespace {
struct SortedWs {
  int32_t* nbr_nat;
  uint32_t *row_mask, *keys_in, *keys_out, *nat_tile_mask;
  int32_t *vals_in, *vals_out;
  unsigned int* k_count;
  void* cub_tmp;
  size_t cub_bytes, total;
};
SortedWs carve_sorted(void* base, int64_t n_out, int K) {
  const int64_t n_slots = round_up(n_out > 0 ? n_out : 1, LG_TILE_ROWS);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? (char*)base + off : nullptr;
    off += (bytes + 255) & ~(size_t)255;
    return (void*)p;
  };
  SortedWs w;
  w.nbr_nat = (int32_t*)take(sizeof(int32_t) * (size_t)K * n_slots);
  w.row_mask = (uint32_t*)take(4 * (size_t)n_slots);
  w.keys_in = (uint32_t*)take(4 * (size_t)n_slots);
  w.keys_out = (uint32_t*)take(4 * (size_t)n_slots);
  w.vals_in = (int32_t*)take(4 * (size_t)n_slots);
  w.vals_out = (int32_t*)take(4 * (size_t)n_slots);
  w.nat_tile_mask = (uint32_t*)take(4 * (size_t)(n_slots / LG_TILE_ROWS));
  w.k_count = (unsigned int*)take(4 * 32);
  w.cub_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, w.cub_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                  (const int32_t*)nullptr, (int32_t*)nullptr, (int)n_slots, 0, K);
  w.cub_tmp = take(w.cub_bytes);
  w.total = off + 256;
  return w;
}
}  // namespace

extern "C" size_t lg_kernel_map_sorted_workspace(int64_t n_out, int32_t kernel_size) {
  if (kernel_size < 1 || kernel_size > 3) return 0;
  return carve_sorted(nullptr, n_out, kernel_size * kernel_size * kernel_size).total;
}

extern "C" int lg_kernel_map_sorted(const void* table_in, int64_t capacity_in, const int32_t* out_coords4,
                                    int64_t n_out, int32_t kernel_size, int32_t offset_scale, int32_t in_row_offset,
                                    int32_t same_set, int32_t* nbr, int32_t* out_row, int64_t n_slots,
                                    uint32_t* tile_mask, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  LG_CHECK_ARG(kernel_size >= 1 && kernel_size <= 3, "lg_kernel_map_sorted: kernel_size %d not in [1,3]", kernel_size);
  LG_CHECK_ARG(n_out >= 0 && n_slots == round_up(n_out, LG_TILE_ROWS),
               "lg_kernel_map_sorted: n_slots must be round_up(n_out,128)");
  LG_CHECK_ARG(capacity_in >= 1024 && (capacity_in & (capacity_in - 1)) == 0, "lg_kernel_map_sorted: bad capacity");
  LG_CHECK_ARG(n_out < ((int64_t)1 << 31), "lg_kernel_map_sorted: too many rows");
  if (n_out == 0) return LG_OK;
  LG_CHECK_ARG(table_in && out_coords4 && nbr && out_row && tile_mask && workspace, "lg_kernel_map_sorted: null pointer");
  LG_CHECK_ARG(workspace_bytes >= lg_kernel_map_sorted_workspace(n_out, kernel_size),
               "lg_kernel_map_sorted: workspace too small");
  const int K = kernel_size * kernel_size * kernel_size;
  SortedWs w = carve_sorted(workspace, n_out, K);
  LG_CUDA_OK(cudaMemsetAsync(w.k_count, 0, 4 * 32, stream));
  int rc = launch_neighbors(table_in, capacity_in, out_coords4, n_out, kernel_size, offset_scale, in_row_offset, same_set,
                            K, 1, w.nbr_nat, n_slots, w.nat_tile_mask, w.row_mask, w.k_count, stream);
  if (rc) return rc;
  k_sort_keys<<<(unsigned)ceil_div(n_out, 256), 256, 0, stream>>>(w.row_mask, w.k_count, K, n_out, w.keys_in, w.vals_in,
                                                                  neighbors_symmetric(same_set, kernel_size) ? 1 : 0);
  LG_LAUNCH_OK();
  size_t cub_bytes = w.cub_bytes;
  LG_CUDA_OK(cub::DeviceRadixSort::SortPairs(w.cub_tmp, cub_bytes, (const uint32_t*)w.keys_in, w.keys_out,
                                             (const int32_t*)w.vals_in, w.vals_out, (int)n_out, 0, K, stream));
  k_permute_plan<<<(unsigned)(n_slots / LG_TILE_ROWS), LG_TILE_ROWS, 0, stream>>>(w.nbr_nat, w.vals_out, n_out, K,
                                                                                   n_slots, nbr, out_row, tile_mask);
  LG_LAUNCH_OK();
  return LG_OK;
}

extern "C" size_t lg_scan_workspace(int64_t n_items) { return scan_workspace_bytes(n_items > 0 ? n_items : 1) + 1024; }

extern "C" int lg_kernel_map_pairs(const int32_t* nbr, int32_t K, int64_t n_slots, int32_t* in_rows, int32_t* out_rows,
                                   int64_t* k_offsets, void* workspace, size_t workspace_bytes, void* stream) {
  LG_CHECK_ARG(K >= 1 && n_slots >= 0 && k_offsets, "lg_kernel_map_pairs: bad arguments");
  const int64_t n = (int64_t)K * n_slots;
  LG_CHECK_ARG(workspace_bytes >= lg_scan_workspace(n), "lg_kernel_map_pairs: workspace too small");
  if (n == 0) {
    LG_CUDA_OK(cudaMemsetAsync(k_offsets, 0, sizeof(int64_t) * (K + 1), (cudaStream_t)stream));
    return LG_OK;
  }
  PairFlag flag{nbr};
  PairSink sink{nbr, n_slots, in_rows, out_rows, k_offsets};
  return device_scan(flag, sink, n, k_offsets + K, workspace, (cudaStream_t)stream);
}

extern "C" int lg_kernel_map_up2(const int32_t* fine_coords4, const int64_t* parent_of_fine, int64_t n_fine,
                                 int32_t fine_stride, int64_t parent_offset, int32_t* gather, int32_t* out_row,
                                 uint32_t* tile_mask,
                                 int64_t n_slots, int64_t* slots_used, void* workspace, size_t workspace_bytes,
                                 void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  LG_CHECK_ARG(n_fine >= 0 && fine_stride >= 1, "lg_kernel_map_up2: bad arguments");
  LG_CHECK_ARG(n_slots % LG_TILE_ROWS == 0 && n_slots >= round_up(n_fine, LG_TILE_ROWS) + 8 * LG_TILE_ROWS,
               "lg_kernel_map_up2: n_slots too small");
  const int64_t n = 8 * n_fine;
  const size_t need = lg_scan_workspace(n) + 256;
  LG_CHECK_ARG(workspace_bytes >= need, "lg_kernel_map_up2: workspace too small");
  LG_CHECK_ARG(gather && out_row && tile_mask && slots_used && workspace, "lg_kernel_map_up2: null pointer");
  int* k_start = (int*)workspace;  // [9] + k_slot_base [9]
  int* k_slot_base = k_start + 16;
  void* scan_ws = (char*)workspace + 256;
  LG_CUDA_OK(cudaMemsetAsync(tile_mask, 0, sizeof(uint32_t) * (size_t)(n_slots / LG_TILE_ROWS), stream));
  k_fill_i32<<<(unsigned)ceil_div(n_slots, 256), 256, 0, stream>>>(gather, n_slots, -1);
  k_fill_i32<<<(unsigned)ceil_div(n_slots, 256), 256, 0, stream>>>(out_row, n_slots, -1);
  LG_LAUNCH_OK();
  if (n_fine == 0) {
    LG_CUDA_OK(cudaMemsetAsync(slots_used, 0, sizeof(int64_t), stream));
    return LG_OK;
  }
  ChildFlag flag{(const int4*)fine_coords4, n_fine, fine_stride};
  ChildSink s1{n_fine, k_start};
  int rc = device_scan(flag, s1, n, nullptr, scan_ws, stream);
  if (rc != LG_OK) return rc;
  k_up2_layout<<<1, 1, 0, stream>>>(k_start, n_fine, k_slot_base, tile_mask, n_slots / LG_TILE_ROWS, slots_used);
  LG_LAUNCH_OK();
  ChildFill s2{parent_of_fine, parent_offset, n_fine, k_start, k_slot_base, gather, out_row};
  return device_scan(flag, s2, n, nullptr, scan_ws, stream);
}
