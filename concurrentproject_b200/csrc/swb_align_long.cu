// swb_align_long.cu -- instantiates the long-pair batch alignment kernels (swb_align_long.cuh).
#define SWB_ALIGN_LONG_KERNELS
#include "swb_align_long.cuh"

namespace swb {

void launch_align_long_span(const AlignBatchParams& P, int blocks, cudaStream_t s) {
  align_long_span_kernel<<<blocks, 32 * kLongAlignWarps, 0, s>>>(P);
}

void launch_align_long_trace(const AlignBatchParams& P, int blocks, cudaStream_t s) {
  align_long_trace_kernel<<<blocks, 32 * kLongAlignWarps, 0, s>>>(P);
}

const void* align_long_span_kernel_ptr() { return (const void*)align_long_span_kernel; }
const void* align_long_trace_kernel_ptr() { return (const void*)align_long_trace_kernel; }

}  // namespace swb
