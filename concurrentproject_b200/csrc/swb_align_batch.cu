// swb_align_batch.cu -- instantiates the batch alignment kernels (swb_align_batch.cuh).
#define SWB_ALIGN_BATCH_KERNELS
#include "swb_align_batch.cuh"

namespace swb {

void launch_align_span(const AlignBatchParams& P, int blocks, cudaStream_t s) {
  align_span_kernel<<<blocks, 256, 0, s>>>(P);
}

void launch_align_trace(const AlignBatchParams& P, int blocks, cudaStream_t s) {
  align_trace_kernel<<<blocks, 256, 0, s>>>(P);
}

}  // namespace swb
