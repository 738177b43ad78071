// Per-device runtime shared by the translation units of liblidog_b200 (see runtime.cu).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

namespace lg {

int tc_runtime(int* sm_count, int** err_word);
int counter_slot(int** out);  // 8 zeroed ints the kernel must leave zeroed (schedule counters, last-block tickets)
int tc_make_tmap(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int box_rows);

// Scratch of one fused call: arena_begin sizes the (device, stream) block for the whole call, arena_take carves it.
struct ArenaCursor {
  char* base;
  size_t cap, off;
};
int arena_begin(cudaStream_t stream, size_t bytes, ArenaCursor* cur);
void* arena_take(ArenaCursor* cur, size_t bytes);
static inline size_t arena_pad(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

}  // namespace lg
