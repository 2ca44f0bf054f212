// swb_batch.cu -- instantiates the batch kernels (swb_batch.cuh) and the batch packer.
#include "swb_batch.cuh"
#include "swb_banded.cuh"

namespace swb {

template <int MODE, int G>
static const void* batch_lookup(int R) {
  switch (R) {
    case 2: return (const void*)sw_batch_kernel<2, MODE, G>;
    case 4: return (const void*)sw_batch_kernel<4, MODE, G>;
    case 6: return (const void*)sw_batch_kernel<6, MODE, G>;
    case 8: return (const void*)sw_batch_kernel<8, MODE, G>;
    case 10: return (const void*)sw_batch_kernel<10, MODE, G>;
    case 12: return (const void*)sw_batch_kernel<12, MODE, G>;
    case 16: return (const void*)sw_batch_kernel<16, MODE, G>;
    default: return nullptr;
  }
}

const void* batch_kernel(int R, int mode, int G) {
  if (mode == 0) return G == 8 ? batch_lookup<0, 8>(R) : (G == 16 ? batch_lookup<0, 16>(R) : batch_lookup<0, 32>(R));
  return G == 8 ? batch_lookup<1, 8>(R) : (G == 16 ? batch_lookup<1, 16>(R) : batch_lookup<1, 32>(R));
}

template <int MODE>
static const void* long_lookup(int R) {
  switch (R) {
    case 2: return (const void*)sw_long_batch_kernel<2, MODE>;
    case 4: return (const void*)sw_long_batch_kernel<4, MODE>;
    case 6: return (const void*)sw_long_batch_kernel<6, MODE>;
    case 8: return (const void*)sw_long_batch_kernel<8, MODE>;
    case 10: return (const void*)sw_long_batch_kernel<10, MODE>;
    case 12: return (const void*)sw_long_batch_kernel<12, MODE>;
    case 16: return (const void*)sw_long_batch_kernel<16, MODE>;
    default: return nullptr;
  }
}

const void* long_batch_kernel(int R, int mode) { return mode == 0 ? long_lookup<0>(R) : long_lookup<1>(R); }

const void* banded_kernel(int mode) {
  return mode == 0 ? (const void*)sw_banded_kernel<0> : (const void*)sw_banded_kernel<1>;
}
const void* banded4_kernel(int mode) {
  return mode == 0 ? (const void*)sw_banded4_kernel<0> : (const void*)sw_banded4_kernel<1>;
}
const void* banded2_kernel(int mode) {
  return mode == 0 ? (const void*)sw_banded2_kernel<0> : (const void*)sw_banded2_kernel<1>;
}
const void* banded8_kernel(int mode) {
  return mode == 0 ? (const void*)sw_banded8_kernel<0> : (const void*)sw_banded8_kernel<1>;
}
const void* banded_wide_kernel(int mode, int width) {
  switch (width) {
    case 128: return mode == 0 ? (const void*)sw_banded_wide_kernel<0, 128> : (const void*)sw_banded_wide_kernel<1, 128>;
    case 256: return mode == 0 ? (const void*)sw_banded_wide_kernel<0, 256> : (const void*)sw_banded_wide_kernel<1, 256>;
    case 512: return mode == 0 ? (const void*)sw_banded_wide_kernel<0, 512> : (const void*)sw_banded_wide_kernel<1, 512>;
    default: return nullptr;
  }
}

// Packs a batch: for every pair the shorter sequence becomes Q, the longer one T; both as 2-bit codes,
// 32 per 64-bit word, fixed word strides per pair.  One thread per output word.
__global__ void pack_batch_kernel(const uint8_t* __restrict__ seq1, const long long* __restrict__ off1,
                                  const int* __restrict__ len1, const uint8_t* __restrict__ seq2,
                                  const long long* __restrict__ off2, const int* __restrict__ len2, long long npairs,
                                  long long q_stride, long long t_stride, uint64_t* __restrict__ q_words,
                                  uint64_t* __restrict__ t_words, int* __restrict__ q_len, int* __restrict__ t_len,
                                  int keep_order, int* status) {
  const long long per_pair = q_stride + t_stride;
  const long long total = npairs * per_pair;
  int bad = 0;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long pair = idx / per_pair;
    const long long wi = idx - pair * per_pair;
    const int l1 = len1[pair], l2 = len2[pair];
    const bool swap = !keep_order && l1 > l2;        // Q = the shorter one, unless the caller's order matters (banded)
    const uint8_t* q = swap ? seq2 + off2[pair] : seq1 + off1[pair];
    const uint8_t* t = swap ? seq1 + off1[pair] : seq2 + off2[pair];
    const int lq = swap ? l2 : l1, lt = swap ? l1 : l2;
    const bool is_q = wi < q_stride;
    const uint8_t* src = is_q ? q : t;
    const int len = is_q ? lq : lt;
    const long long w = is_q ? wi : wi - q_stride;
    uint64_t out = 0;
    const long long base = w * 32;
    for (int k = 0; k < 32 && base + k < len; ++k) {
      const uint32_t c = src[base + k];
      const uint32_t v = (c >> 1) & 3;
      bad |= (c != ((0x47544341u >> (8 * v)) & 0xFFu));
      out |= (uint64_t)v << (2 * k);
    }
    if (is_q) q_words[pair * q_stride + w] = out; else t_words[pair * t_stride + w] = out;
    if (wi == 0) { q_len[pair] = lq; t_len[pair] = lt; }
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(status + 1, STATUS_BAD_SYMBOL);
}

void launch_pack_batch(const uint8_t* seq1, const long long* off1, const int* len1, const uint8_t* seq2,
                       const long long* off2, const int* len2, long long npairs, long long q_stride, long long t_stride,
                       uint64_t* q_words, uint64_t* t_words, int* q_len, int* t_len, int keep_order, int* status,
                       int blocks, cudaStream_t s) {
  pack_batch_kernel<<<blocks, 256, 0, s>>>(seq1, off1, len1, seq2, off2, len2, npairs, q_stride, t_stride, q_words, t_words,
                                           q_len, t_len, keep_order, status);
}

// Packs a byte batch (swb_bytes_batch.cu): the shorter sequence of every pair becomes Q, the longer one T, both as raw
// bytes, 8 per 64-bit word (byte p at bits 8*(p%8)), fixed word strides per pair.  Every byte is kept as it is: no
// check, no remapping.  One thread per output word.
__global__ void pack_bytes_kernel(const uint8_t* __restrict__ seq1, const long long* __restrict__ off1,
                                  const int* __restrict__ len1, const uint8_t* __restrict__ seq2,
                                  const long long* __restrict__ off2, const int* __restrict__ len2, long long npairs,
                                  long long q_stride, long long t_stride, uint64_t* __restrict__ q_words,
                                  uint64_t* __restrict__ t_words, int* __restrict__ q_len, int* __restrict__ t_len) {
  const long long per_pair = q_stride + t_stride;
  const long long total = npairs * per_pair;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long pair = idx / per_pair;
    const long long wi = idx - pair * per_pair;
    const int l1 = len1[pair], l2 = len2[pair];
    const bool swap = l1 > l2;
    const uint8_t* q = swap ? seq2 + off2[pair] : seq1 + off1[pair];
    const uint8_t* t = swap ? seq1 + off1[pair] : seq2 + off2[pair];
    const int lq = swap ? l2 : l1, lt = swap ? l1 : l2;
    const bool is_q = wi < q_stride;
    const uint8_t* src = is_q ? q : t;
    const int len = is_q ? lq : lt;
    const long long w = is_q ? wi : wi - q_stride;
    uint64_t out = 0;
    const long long base = w * 8;
    for (int k = 0; k < 8 && base + k < len; ++k) out |= (uint64_t)src[base + k] << (8 * k);
    if (is_q) q_words[pair * q_stride + w] = out; else t_words[pair * t_stride + w] = out;
    if (wi == 0) { q_len[pair] = lq; t_len[pair] = lt; }
  }
}

void launch_pack_bytes(const uint8_t* seq1, const long long* off1, const int* len1, const uint8_t* seq2,
                       const long long* off2, const int* len2, long long npairs, long long q_stride, long long t_stride,
                       uint64_t* q_words, uint64_t* t_words, int* q_len, int* t_len, int blocks, cudaStream_t s) {
  pack_bytes_kernel<<<blocks, 256, 0, s>>>(seq1, off1, len1, seq2, off2, len2, npairs, q_stride, t_stride, q_words, t_words,
                                           q_len, t_len);
}

}  // namespace swb
