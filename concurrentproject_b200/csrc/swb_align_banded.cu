// swb_align_banded.cu -- instantiates the banded batch alignment kernels (swb_align_banded.cuh), K = 1, 2, 4, 8.
#define SWB_ALIGN_BANDED_KERNELS
#include "swb_align_banded.cuh"

namespace swb {

void launch_align_banded_span(const AlignBandedParams& P, int K, int blocks, cudaStream_t s) {
  switch (K) {
    case 1: align_banded_span_kernel<1><<<blocks, 32 * kBandAlignWarps, 0, s>>>(P); break;
    case 2: align_banded_span_kernel<2><<<blocks, 32 * kBandAlignWarps, 0, s>>>(P); break;
    case 4: align_banded_span_kernel<4><<<blocks, 32 * kBandAlignWarps, 0, s>>>(P); break;
    case 8: align_banded_span_kernel<8><<<blocks, 32 * kBandAlignWarps, 0, s>>>(P); break;
  }
}

void launch_align_banded_trace(const AlignBandedParams& P, int K, int blocks, cudaStream_t s) {
  switch (K) {
    case 1: align_banded_trace_kernel<1><<<blocks, 32 * kBandAlignWarps, 0, s>>>(P); break;
    case 2: align_banded_trace_kernel<2><<<blocks, 32 * kBandAlignWarps, 0, s>>>(P); break;
    case 4: align_banded_trace_kernel<4><<<blocks, 32 * kBandAlignWarps, 0, s>>>(P); break;
    case 8: align_banded_trace_kernel<8><<<blocks, 32 * kBandAlignWarps, 0, s>>>(P); break;
  }
}

const void* align_banded_trace_kernel_ptr(int K) {
  switch (K) {
    case 2: return (const void*)align_banded_trace_kernel<2>;
    case 4: return (const void*)align_banded_trace_kernel<4>;
    case 8: return (const void*)align_banded_trace_kernel<8>;
    default: return (const void*)align_banded_trace_kernel<1>;
  }
}

}  // namespace swb
