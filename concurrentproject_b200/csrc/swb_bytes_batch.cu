// swb_bytes_batch.cu -- batch scoring and alignment of pairs in any bytes (swb200_score_batch_bytes,
// swb200_align_batch_bytes, and a batch packed by swb200_batch_pack_device_bytes).
//
// The bodies are those of swb_align_batch.cuh with align_code<8>: one thread per pair, 32-bit arithmetic, symbols compared
// with == exactly as main.cpp:28-33 compares bytes (N matches N, 'a' does not match 'A').  The byte packer
// (swb_batch.cu) lays each sequence out as 8 bytes per 64-bit word at fixed word strides, the shorter sequence of a pair
// first.  Scoring runs pass 1 alone, without the end cell.
#include "swb_align_batch.cuh"

namespace swb {

__global__ void __launch_bounds__(256) bytes_span_kernel(const __grid_constant__ AlignBatchParams P) {
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long cells = 0;
  for (long long k = tid; k < P.npairs; k += P.nthreads) cells += align_span_pair<8>(P, k, tid);
  if (cells) atomicAdd(P.cells, (unsigned long long)cells);
}

__global__ void __launch_bounds__(256) bytes_trace_kernel(const __grid_constant__ AlignBatchParams P) {
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long cells = 0;
  for (long long t = tid; t < P.ntodo; t += P.nthreads) {
    const long long c = align_trace_pair<8>(P, P.todo ? P.todo[t] : t, tid);
    cells += c > 0 ? c : 0;
  }
  if (cells) atomicAdd(P.cells, (unsigned long long)cells);
}

__global__ void __launch_bounds__(256) bytes_score_kernel(const __grid_constant__ AlignBatchParams P) {
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (long long k = tid; k < P.npairs; k += P.nthreads) align_score_pair<8>(P, k, tid);
}

void launch_bytes_span(const AlignBatchParams& P, int blocks, cudaStream_t s) { bytes_span_kernel<<<blocks, 256, 0, s>>>(P); }
void launch_bytes_trace(const AlignBatchParams& P, int blocks, cudaStream_t s) { bytes_trace_kernel<<<blocks, 256, 0, s>>>(P); }
void launch_bytes_score(const AlignBatchParams& P, int blocks, cudaStream_t s) { bytes_score_kernel<<<blocks, 256, 0, s>>>(P); }
const void* bytes_score_kernel_ptr() { return (const void*)bytes_score_kernel; }

}  // namespace swb
