// Evaluation metric on the device: the confusion matrix behind LiDOG's per-class IoU / mIoU.
// Reference: sklearn.metrics.jaccard_score(labels=range(C), average=None) on the CPU in eval / test
// (trainer_lighting_bev.py:265-323) and torchmetrics JaccardIndex(ignore_index) in the training step.  Both are
// functions of one (C + 1) x C matrix of counts: row = target class, row C = any target outside [0, C) (the ignore
// label included), column = predicted class argmax_c logits[i, c] (first maximal index, as torch.argmax).
// Each block counts into a shared-memory histogram and adds it to the int64 matrix with integer atomics: the result
// is exact and the same on every run.  Bound: HBM, one read of the logits and the targets.
#include "common.cuh"
#include "runtime.cuh"

namespace lg {

constexpr int kConfThreads = 256;
constexpr int kConfMaxBlocks = 592;  // 4 per SM
constexpr int kConfMaxC = 32;

__global__ void __launch_bounds__(kConfThreads)
    k_confusion(const float* __restrict__ logits, const long long* __restrict__ target, int64_t n, int C,
                unsigned long long* __restrict__ conf) {
  __shared__ unsigned int hist[(kConfMaxC + 1) * kConfMaxC];
  const int cells = (C + 1) * C;
  for (int i = threadIdx.x; i < cells; i += blockDim.x) hist[i] = 0u;
  __syncthreads();
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const float* z = logits + r * C;
    float m = __ldg(z);
    int best = 0;
    for (int c = 1; c < C; ++c) {
      const float v = __ldg(z + c);
      // torch.argmax: the first maximal index; a NaN counts as the maximum (the first NaN wins)
      if (!(m != m) && (v > m || v != v)) {
        m = v;
        best = c;
      }
    }
    const long long t = __ldg(target + r);
    const int row = (t >= 0 && t < C) ? (int)t : C;
    atomicAdd(&hist[row * C + best], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < cells; i += blockDim.x)
    if (hist[i]) atomicAdd(conf + i, (unsigned long long)hist[i]);
}

}  // namespace lg

using namespace lg;

extern "C" int lg_confusion_matrix(const float* logits, int64_t n, int32_t C, const int64_t* target, int64_t* conf,
                                   void* stream_) {
  LG_CHECK_ARG(C >= 1 && C <= kConfMaxC, "lg_confusion_matrix: 1 <= C <= %d classes", kConfMaxC);
  // a block's shared-memory counters are 32-bit: a block sees at most ceil(n / blocks) rows
  LG_CHECK_ARG(n >= 0 && n < ((int64_t)1 << 40), "lg_confusion_matrix: bad row count");
  if (n == 0) return LG_OK;
  LG_CHECK_ARG(logits && target && conf, "lg_confusion_matrix: null pointer");
  // 64-bit atomics on conf, 64-bit loads of target, 32-bit loads of logits
  LG_CHECK_ARG(((uintptr_t)conf & 7) == 0 && ((uintptr_t)target & 7) == 0 && ((uintptr_t)logits & 3) == 0,
               "lg_confusion_matrix: conf and target must be 8-byte aligned, logits 4-byte aligned");
  int64_t nb = ceil_div(n, (int64_t)kConfThreads * 4);
  if (nb > kConfMaxBlocks) nb = kConfMaxBlocks;
  k_confusion<<<(unsigned)nb, kConfThreads, 0, (cudaStream_t)stream_>>>(logits, (const long long*)target, n, C,
                                                                        (unsigned long long*)conf);
  LG_LAUNCH_OK();
  return LG_OK;
}
