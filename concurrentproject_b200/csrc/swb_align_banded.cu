// swb_align_banded.cu -- instantiates the banded batch alignment kernels (swb_align_banded.cuh).
#define SWB_ALIGN_BANDED_KERNELS
#include "swb_align_banded.cuh"

namespace swb {

void launch_align_banded_span(const AlignBandedParams& P, int blocks, cudaStream_t s) {
  align_banded_span_kernel<<<blocks, 32 * kBandAlignWarps, 0, s>>>(P);
}

void launch_align_banded_trace(const AlignBandedParams& P, int blocks, cudaStream_t s) {
  align_banded_trace_kernel<<<blocks, 32 * kBandAlignWarps, 0, s>>>(P);
}

const void* align_banded_trace_kernel_ptr() { return (const void*)align_banded_trace_kernel; }

}  // namespace swb
