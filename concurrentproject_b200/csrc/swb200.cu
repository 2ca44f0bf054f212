// swb200.cu -- C ABI of libswb200.so (see include/swb200.h, include/algoGPU.h).
//
// Host side of the hot path: what the reference's host functions do around their kernels
// (simpleGPU.cu:109-163, cudaLazy.cu:58-99, cudaSmithM.cu:128-189: cudaMalloc x5, H2D x2, 2N-1
// launches, D2H of the whole H matrix, host max, cudaFree x5) becomes: persistent context, two
// H2D copies, two encode kernels, ONE cooperative launch of the wavefront engine, a 16-byte D2H.
// There is no CPU fallback: every score comes from the engine kernels or the call fails.
#include "../../include/swb200.h"
#include "../../include/algoGPU.h"
#include "swb_kernels.cuh"
#include "swb_traceback.cuh"
#include "swb_chain.cuh"
#include "swb_batch.cuh"
#include "swb_banded.cuh"
#include "swb_align_batch.cuh"
#include "swb_align_banded.cuh"
#include "swb_align_long.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <climits>
#include <memory>
#include <mutex>
#include <thread>
#include <string>
#include <vector>
#include <algorithm>
#include <functional>

namespace {

thread_local std::string g_err;

// Debugging / measurement switches.  Read from the environment ONCE (first use), changed afterwards only through
// swb200_configure(); the scoring calls themselves never touch getenv.
struct Settings {
  long long spin_limit = 40LL * 1000 * 1000;   // SWB200_SPIN_LIMIT: polls before a waiting warp gives up
  int dbg = 0;                                  // SWB200_DBG: timing experiments (1 = no boundary stores, 2 = no polls)
  bool debug = false;                           // SWB200_DEBUG: print the post-mortem of a timed-out hand-off
  std::string prof_path;                        // SWB200_PROF: per-warp cycle counters ("1" = stderr summary, else a file)
  std::string dump_final_path;                  // SWB200_DUMP_FINAL: the two middle rows of a two-sided sweep
  long long batch_chunk_bytes = 0;              // SWB200_BATCH_CHUNK_BYTES: tests force many small chunks
  long long ring_min_cells = 200LL * 1000 * 1000 * 1000;   // SWB200_RING_MIN_CELLS: pairs at least this large use all devices
  int chain = 1;                                // SWB200_CHAIN: 0 = the planner never picks the CTA-chained engine (launch config 7) by itself
  long long align_block_rows = 0;               // SWB200_ALIGN_BLOCK_ROWS: swb200_align's traceback in blocks of this many rows (0 = when needed)
};
std::mutex g_settings_mu;
Settings& settings_locked() {       // caller holds g_settings_mu
  static Settings st;
  static bool init = false;
  if (!init) {
    init = true;
    if (const char* e = getenv("SWB200_SPIN_LIMIT")) st.spin_limit = atoll(e);
    if (const char* e = getenv("SWB200_DBG")) st.dbg = atoi(e);
    st.debug = getenv("SWB200_DEBUG") != nullptr;
    if (const char* e = getenv("SWB200_PROF")) st.prof_path = e;
    if (const char* e = getenv("SWB200_DUMP_FINAL")) st.dump_final_path = e;
    if (const char* e = getenv("SWB200_BATCH_CHUNK_BYTES")) st.batch_chunk_bytes = std::max(1LL, atoll(e));
    if (const char* e = getenv("SWB200_RING_MIN_CELLS")) st.ring_min_cells = std::max(1LL, atoll(e));
    if (const char* e = getenv("SWB200_CHAIN")) st.chain = atoi(e);
    if (const char* e = getenv("SWB200_ALIGN_BLOCK_ROWS")) st.align_block_rows = atoll(e);   // checked by swb200_align
  }
  return st;
}
Settings settings() {               // a copy: cheap, and the caller needs no lock afterwards
  std::lock_guard<std::mutex> lk(g_settings_mu);
  return settings_locked();
}

int fail(int code, const std::string& msg) { g_err = msg; return code; }

#define SWB_CUDA(call)                                                                      \
  do {                                                                                      \
    cudaError_t e_ = (call);                                                                \
    if (e_ != cudaSuccess)                                                                  \
      return fail(SWB200_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));    \
  } while (0)

// Every entry point switches to its context's device; the caller's current device is restored on every return path
// (a host program or a torch process working on device A must not be left on device B).
struct DeviceGuard {
  int prev = -1;
  DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// ---------------------------------------------------------------------------------------------
//  encode kernels: raw bytes -> 2-bit codes
// ---------------------------------------------------------------------------------------------
// Fast path: A,C,G,T -> (c >> 1) & 3 = 0,1,3,2 (injective on ACGT; equality scoring only needs an
// injective recoding).  Any other byte sets STATUS_BAD_SYMBOL and the host re-encodes through a
// 256-entry table built from the symbols actually present (covers the reference's own
// known-answer tests over {A,B,D}, main.cpp:99-100).
__device__ __forceinline__ uint32_t code_of(uint32_t c, const uint8_t* lut, int& bad) {
  if (lut) {
    const uint32_t v = lut[c];
    bad |= v > 3;
    return v & 3;
  }
  const uint32_t v = (c >> 1) & 3;
  bad |= (c != ((0x47544341u >> (8 * v)) & 0xFFu));   // "ACTG"[v]
  return v;
}

// Q side: one code byte per symbol (read once per band by the owning thread).
__global__ void encode_q_kernel(const uint8_t* __restrict__ src, long long n, uint8_t* __restrict__ dst,
                                const uint8_t* __restrict__ lut, int* status) {
  int bad = 0;
  const long long stride = (long long)gridDim.x * blockDim.x * 16;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 16; i < n; i += stride) {
    if (i + 16 <= n && ((reinterpret_cast<uintptr_t>(src + i) & 15) == 0)) {
      const uint4 v = *reinterpret_cast<const uint4*>(src + i);        // coalesced 128-bit read
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
      uint32_t o[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        o[k] = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) o[k] |= code_of((w[k] >> (8 * b)) & 0xFF, lut, bad) << (8 * b);
      }
      *reinterpret_cast<uint4*>(dst + i) = make_uint4(o[0], o[1], o[2], o[3]);
    } else {
      for (long long k = i; k < n && k < i + 16; ++k) dst[k] = (uint8_t)code_of(src[k], lut, bad);
    }
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(status + 1, swb::STATUS_BAD_SYMBOL);
}

// T side: 32 symbols per 64-bit word, symbol p at bits 2*(p%32).
__global__ void encode_t_kernel(const uint8_t* __restrict__ src, long long n, uint64_t* __restrict__ dst,
                                const uint8_t* __restrict__ lut, int* status) {
  int bad = 0;
  const long long nwords = (n + 31) / 32;
  for (long long wi = (long long)blockIdx.x * blockDim.x + threadIdx.x; wi < nwords;
       wi += (long long)gridDim.x * blockDim.x) {
    const long long base = wi * 32;
    uint64_t out = 0;
    if (base + 32 <= n && ((reinterpret_cast<uintptr_t>(src + base) & 15) == 0)) {
      const uint4 a = *reinterpret_cast<const uint4*>(src + base);
      const uint4 b = *reinterpret_cast<const uint4*>(src + base + 16);
      const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
      for (int k = 0; k < 8; ++k)
#pragma unroll
        for (int q = 0; q < 4; ++q)
          out |= (uint64_t)code_of((w[k] >> (8 * q)) & 0xFF, lut, bad) << (2 * (4 * k + q));
    } else {
      for (int k = 0; k < 32 && base + k < n; ++k) out |= (uint64_t)code_of(src[base + k], lut, bad) << (2 * k);
    }
    dst[wi] = out;
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(status + 1, swb::STATUS_BAD_SYMBOL);
}

// Two-sided sweep, second half: Q' = pad rows + reverse(seq[mid..n)), one code byte per symbol.
__global__ void encode_q_rev_kernel(const uint8_t* __restrict__ src, long long n, long long mid, long long pad,
                                    uint8_t* __restrict__ dst, const uint8_t* __restrict__ lut, int* status) {
  int bad = 0;
  const long long total = pad + (n - mid);
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x)
    dst[k] = k < pad ? (uint8_t)4 : (uint8_t)code_of(src[n - 1 - (k - pad)], lut, bad);
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(status + 1, swb::STATUS_BAD_SYMBOL);
}

// Two-sided sweep, second half: T' = reverse(seq), 2-bit packed.
__global__ void encode_t_rev_kernel(const uint8_t* __restrict__ src, long long n, uint64_t* __restrict__ dst,
                                    const uint8_t* __restrict__ lut, int* status) {
  int bad = 0;
  const long long nwords = (n + 31) / 32;
  for (long long wi = (long long)blockIdx.x * blockDim.x + threadIdx.x; wi < nwords; wi += (long long)gridDim.x * blockDim.x) {
    uint64_t out = 0;
    for (int k = 0; k < 32 && wi * 32 + k < n; ++k) out |= (uint64_t)code_of(src[n - 1 - (wi * 32 + k)], lut, bad) << (2 * k);
    dst[wi] = out;
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(status + 1, swb::STATUS_BAD_SYMBOL);
}

// Two-sided sweep: alignments that cross the middle row.  f0[p + skew] = bottom boundary (H-open, F) of the forward
// half at T position p; f1[p' + skew] = the same of the reversed half at reversed position p'.  A crossing path
// passes lattice point (mid, x): best score ending there (forward) + best score starting there (reversed); a
// vertical gap that straddles the row was opened twice, hence the + gap_init - gap_ext variant (Myers-Miller).
// Re-based lanes: the entries are relative to the base their warp published for the 256-step block (b0 / b1, null
// for plain 16-bit lanes).
__global__ void combine_two_sided_kernel(const uint2* __restrict__ f0, const uint2* __restrict__ f1, long long LT, int skew,
                                         int linear, int gap_init, int gap_ext, const uint2* __restrict__ b0,
                                         const uint2* __restrict__ b1, int* result) {
  int best = 0;
  for (long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x; x <= LT; x += (long long)gridDim.x * blockDim.x) {
    int Hf = 0, Ff = -1000000, Hb = 0, Fb = -1000000;
    if (x >= 1) {
      const long long j = x - 1 + skew;
      const uint32_t e = f0[j].x;
      const int base = b0 ? (int)b0[j >> 8].x : 0;
      if (linear) Hf = (int)(short)(e >> 16) + gap_init + base;
      else { Hf = (int)(short)(e & 0xFFFFu) + gap_init + base; Ff = (int)(short)(e >> 16) + base; }
    }
    if (x <= LT - 1) {
      const long long j = (LT - 1 - x) + skew;
      const uint32_t e = f1[j].x;
      const int base = b1 ? (int)b1[j >> 8].x : 0;
      if (linear) Hb = (int)(short)(e >> 16) + gap_init + base;
      else { Hb = (int)(short)(e & 0xFFFFu) + gap_init + base; Fb = (int)(short)(e >> 16) + base; }
    }
    int v = Hf + Hb;
    if (!linear) v = max(v, Ff + Fb + gap_init - gap_ext);
    best = max(best, v);
  }
  best = __reduce_max_sync(0xffffffffu, best);
  if ((threadIdx.x & 31) == 0 && best > 0) atomicMax(result, best);
}

// dst[k] = src[n-1-k]: the reversed prefixes for the anchored start-cell pass.
__global__ void reverse_bytes_kernel(const uint8_t* __restrict__ src, long long n, uint8_t* __restrict__ dst) {
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x)
    dst[k] = src[n - 1 - k];
}

// 256-bit presence map of the byte values in a buffer.
__global__ void presence_kernel(const uint8_t* __restrict__ src, long long n, uint32_t* bitmap) {
  __shared__ uint32_t local[8];
  if (threadIdx.x < 8) local[threadIdx.x] = 0;
  __syncthreads();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t c = src[i];
    atomicOr(&local[c >> 5], 1u << (c & 31));
  }
  __syncthreads();
  if (threadIdx.x < 8 && local[threadIdx.x]) atomicOr(&bitmap[threadIdx.x], local[threadIdx.x]);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
//  context
// ---------------------------------------------------------------------------------------------
struct swb200_ctx {
  int device = 0;
  int sms = 0;
  std::mutex mu;
  cudaStream_t own_stream = nullptr;
  cudaStream_t aux_stream = nullptr;        // host batch calls: kernels run here while own_stream copies the next chunk
  std::vector<cudaEvent_t> chunk_events;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // grow-only device buffers
  uint8_t* d_ascii = nullptr; size_t ascii_cap = 0;
  uint8_t* d_q = nullptr; size_t q_cap = 0;
  uint64_t* d_t = nullptr; size_t t_cap = 0;     // words
  uint8_t* d_q2 = nullptr; size_t q2_cap = 0;    // two-sided sweep: reversed second half
  uint64_t* d_t2 = nullptr; size_t t2_cap = 0;
  uint2* d_final = nullptr; size_t final_cap = 0; // two-sided sweep: the two middle boundary rows
  uint2* d_links = nullptr; size_t links_cap = 0;  // entries
  uint2* d_chain = nullptr; size_t chain_cap = 0;  // CTA-chained engine (launch config 7): one full-length link per CTA
  uint2* d_ext = nullptr; size_t ext_cap = 0;      // entries
  unsigned long long* d_progress = nullptr; size_t progress_cap = 0;
  int* d_cand = nullptr; size_t cand_cap = 0;     // end-cell tracking: {H, T position, Q row} per band
  uint32_t* d_dirs = nullptr; size_t dirs_cap = 0;   // traceback directions (swb200_align): 4 bits per cell of the span rectangle
  unsigned long long* d_ops = nullptr; size_t ops_cap = 0;   // the walk's state (8 words), then its run-length operations, last first
  uint2* d_ckpt = nullptr; size_t ckpt_cap = 0;   // blocked traceback (swb200_align): the bottom row of every block but the last
  uint8_t* d_rev = nullptr; size_t rev_cap = 0;   // start-cell pass: the two reversed prefixes
  int* d_result = nullptr;        // [0] score [1] status, [2..9] presence bitmap
  uint8_t* d_lut = nullptr;       // 256 bytes
  int* h_result = nullptr;        // pinned
  unsigned epoch = 0;
  long long last_nsteps = 0; int last_skew_per_lane = 0;     // geometry of the last engine run (the traceback walk needs it)
  swb200_run_info info{};
  long long* d_prof = nullptr; size_t prof_cap = 0;   // SWB200_PROF counters (grow-only, owned by the context)
  // grow-only staging of the host batch entry points (no cudaMalloc/cudaFree per call)
  uint8_t* hb_seq1 = nullptr; size_t hb_seq1_cap = 0;
  uint8_t* hb_seq2 = nullptr; size_t hb_seq2_cap = 0;
  long long* hb_off1 = nullptr; size_t hb_off1_cap = 0;
  long long* hb_off2 = nullptr; size_t hb_off2_cap = 0;
  int* hb_len1 = nullptr; size_t hb_len1_cap = 0;
  int* hb_len2 = nullptr; size_t hb_len2_cap = 0;
  int* hb_scores = nullptr; size_t hb_scores_cap = 0;
  uint64_t* hb_qw = nullptr; size_t hb_qw_cap = 0;
  uint64_t* hb_tw = nullptr; size_t hb_tw_cap = 0;
  int* hb_ql = nullptr; size_t hb_ql_cap = 0;
  int* hb_tl = nullptr; size_t hb_tl_cap = 0;
  // batch alignment (swb200_align_batch / swb200_batch_align), grow-only
  int2* ab_col = nullptr; size_t ab_col_cap = 0;          // per-thread column buffers
  uint64_t* ab_slot = nullptr; size_t ab_slot_cap = 0;    // per-thread direction slots
  uint64_t* ab_pool = nullptr; size_t ab_pool_cap = 0;    // shared direction pool (allocated only when a rectangle needs it)
  int* ab_list = nullptr; size_t ab_list_cap = 0;         // two pending lists
  unsigned long long* ab_misc = nullptr; size_t ab_misc_cap = 0;   // [0] err | npending << 32, [1] pool words used, [2] cells
  int* hb_spans = nullptr; size_t hb_spans_cap = 0;       // host batch alignment: outputs before the copy back
  uint32_t* hb_ops = nullptr; size_t hb_ops_cap = 0;
  int* hb_opsn = nullptr; size_t hb_opsn_cap = 0;
  // multi-band batch scoring (swb200_score_long_batch / swb200_batch_score_long), grow-only
  uint32_t* lb_bnd = nullptr; size_t lb_bnd_cap = 0;                  // one boundary row per launched warp
  unsigned long long* lb_next = nullptr; size_t lb_next_cap = 0;      // the launch's pair counter
};

namespace swb {
void launch_pack_batch(const uint8_t* seq1, const long long* off1, const int* len1, const uint8_t* seq2,
                       const long long* off2, const int* len2, long long npairs, long long q_stride, long long t_stride,
                       uint64_t* q_words, uint64_t* t_words, int* q_len, int* t_len, int keep_order, int* status,
                       int blocks, cudaStream_t s);
void launch_pack_bytes(const uint8_t* seq1, const long long* off1, const int* len1, const uint8_t* seq2,
                       const long long* off2, const int* len2, long long npairs, long long q_stride, long long t_stride,
                       uint64_t* q_words, uint64_t* t_words, int* q_len, int* t_len, int blocks, cudaStream_t s);
}

// A packed batch resident in HBM (2-bit codes, or bytes, fixed word strides, shorter sequence of each pair first).
struct swb200_batch {
  swb200_ctx* ctx = nullptr;
  long long npairs = 0, q_stride = 0, t_stride = 0;
  int max_short = 0, max_long = 0;
  int keep_order = 0;          // 1: q = seq1, t = seq2 exactly as given (banded scoring needs j-i)
  int bytes = 0;               // 1: raw bytes, 8 per word (swb200_batch_pack_device_bytes; the byte kernels only)
  uint64_t* q_words = nullptr;
  uint64_t* t_words = nullptr;
  int* q_len = nullptr;
  int* t_len = nullptr;
  int* len1 = nullptr;         // keep_order = 0: the caller's seq1 lengths (which pairs were swapped; swb200_batch_align)
  long long cells = 0;
};

// What the root rank needs to combine the two halves of a two-sided sweep over the ring once every rank is done.
struct RingCombine {
  bool pending = false;
  long long LT = 0, ext_len = 0, NB0 = 0, NB1 = 0;
  int skew = 0, linear = 0, rebased = 0, gap_init = 0, gap_ext = 0;
};

// One rank's region: [0, 2*len) boundary stream of the forward ring (entries + bases), [2*len, 4*len) the same for the
// reversed ring of a two-sided sweep, [4*len, 6*len) / [6*len, 8*len) the two middle boundary rows (only the ROOT
// rank's copy is written: the ranks that own the two last bands store there through NVLink).
struct swb200_ring {
  swb200_ctx* ctx = nullptr;
  int rank = 0, world = 1;
  uint2* inbound = nullptr;
  size_t len = 0;              // entries per half-region unit (a power of two)
  size_t entries = 0;          // 8 * len
  uint2* next = nullptr;
  bool next_is_ipc = false;
  uint2* root = nullptr;       // rank 0's region (== inbound on rank 0); null: two-sided sweeps are off for this ring
  bool root_is_ipc = false;
  unsigned calls = 0;
  RingCombine combine;
};

namespace {

// owners for objects under construction: an early SWB_CUDA return frees everything allocated so far
struct CtxDeleter { void operator()(swb200_ctx* c) const { swb200_ctx_destroy(c); } };
struct RingDeleter { void operator()(swb200_ring* r) const { swb200_ring_destroy(r); } };
struct BatchDeleter { void operator()(swb200_batch* b) const { swb200_batch_free(b); } };

template <typename T>
int grow(T*& p, size_t& cap, size_t need, bool zero, cudaStream_t s) {
  if (need <= cap) return SWB200_OK;
  if (p) SWB_CUDA(cudaFree(p));
  p = nullptr; cap = 0;
  const size_t want = need + need / 4 + 1024;
  cudaError_t e = cudaMalloc(&p, want * sizeof(T));
  if (e != cudaSuccess) return fail(SWB200_ERR_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
  cap = want;
  if (zero) SWB_CUDA(cudaMemsetAsync(p, 0, want * sizeof(T), s));
  return SWB200_OK;
}

int check_params(const swb200_params& p) {
  if (p.match < 0 || p.match > 100 || p.mismatch > 0 || p.mismatch < -100 || p.gap_init < 0 || p.gap_init > 100 ||
      p.gap_ext < 0 || p.gap_ext > 100 || p.match + p.gap_init > 127)
    return fail(SWB200_ERR_ARG, "scoring parameters outside the documented limits");
  return SWB200_OK;
}

// NULL parameters / options: MATCH, MISMATCH, GAP_INIT, GAP_EXT of main.cpp:20-23, and every option at its default
swb200_params params_or_default(const swb200_params* p) { return p ? *p : swb200_params{1, -1, 1, 1}; }
swb200_options options_or_default(const swb200_options* o) { return o ? *o : swb200_options{}; }

// Re-based 16-bit lanes are exact as long as the values one warp holds at one time, plus what they can drift
// between two re-base decisions, stay far inside 16 bits: neighbouring cells differ by at most match + gap per
// step, a warp spans 64*R rows and ~100 columns, decisions come every 256 steps, the trigger is +-8000.
bool rebase_is_safe(const swb200_params& p, int R) {
  const long long step = (long long)p.match + std::max(p.gap_init, p.gap_ext);
  return step * (64LL * R + 96 + swb::kRebaseBlock + 64) <= 10000;
}

// End-cell tracking: reduce the per-band candidates {H, T position, Q row} to the best H, then the smallest
// T position, then the smallest Q row (the rule every warp already applied inside its band).  One block.
__global__ void reduce_end_kernel(const int* cand, int nb, int* out3) {
  __shared__ int sh[256], sp[256], sr[256];
  int h = 0, p = 0x7fffffff, r = 0x7fffffff;
  for (int b = (int)threadIdx.x; b < nb; b += 256) {
    const int ch = cand[3 * b], cp = cand[3 * b + 1], cr = cand[3 * b + 2];
    if (ch > h || (ch == h && (cp < p || (cp == p && cr < r)))) { h = ch; p = cp; r = cr; }
  }
  sh[threadIdx.x] = h; sp[threadIdx.x] = p; sr[threadIdx.x] = r;
  __syncthreads();
  for (int d = 128; d > 0; d >>= 1) {
    if ((int)threadIdx.x < d) {
      const int oh = sh[threadIdx.x + d], op = sp[threadIdx.x + d], orr = sr[threadIdx.x + d];
      const int mh = sh[threadIdx.x], mp = sp[threadIdx.x], mr = sr[threadIdx.x];
      if (oh > mh || (oh == mh && (op < mp || (op == mp && orr < mr)))) { sh[threadIdx.x] = oh; sp[threadIdx.x] = op; sr[threadIdx.x] = orr; }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { out3[0] = sh[0]; out3[1] = sp[0]; out3[2] = sr[0]; }
}

// Traceback walk (swb200_align): one thread follows the directions of one launch back (walk_block, swb_traceback.cuh), a
// chain of dependent loads, at most rows + cols of them.  The walk's state stays in *st between the blocks of a blocked
// traceback; first: start at the last cell (rows, cols) of the span.
__global__ void walk_traceback_kernel(const uint32_t* __restrict__ dirs, long long nsteps, int sk, long long row0, bool first,
                                      long long rows, long long cols, swb::WalkState* st, unsigned long long* ops, long long ops_cap) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  swb::WalkState ws = first ? swb::walk_start(rows, cols) : *st;
  swb::walk_block(dirs, nsteps, sk, row0, ws, ops, ops_cap);
  *st = ws;
}

// Blocked traceback: checkpoint row -> the ext_in stream of the next launch, under that launch's tag (swb_traceback.cuh).
__global__ void retag_checkpoint_kernel(const uint2* __restrict__ ckpt, uint2* ext, long long s0, long long s1, uint32_t tag) {
  for (long long s = s0 + (long long)blockIdx.x * blockDim.x + threadIdx.x; s < s1; s += (long long)gridDim.x * blockDim.x)
    swb::retag_slot(ckpt, ext, s, tag);
}

struct Plan {
  int mode;      // 0 s16 affine, 1 s16 linear, 2 s32 affine, 3/4 = 0/1 with re-based lanes, 5 s32 bytes, 6/7 = 2/5 + end cell
  int R, config, ctas;
  bool swap;     // Q = seq2 instead of seq1
  bool two_sided;  // forward sweep over the top half of the rows + reversed sweep over the bottom half
};

// Estimated cycles for one (R, config) choice.  Model and constants fitted to B200 sweeps
// (profiles/r01_sweep_*.jsonl): a warp-step costs per_row*R + 30 cycles (39 in config 2).  With one warp per scheduler
// (configs 1, 3: short-chain row loop, step loops unrolled 8x) per_row = 13.2 / 7.5 / 12 / 15.6 / 9.8 / 14 cycles for s16 affine /
// s16 linear / s32 / re-based affine / re-based linear / byte-compare s32; with two warps per scheduler
// (config 2: fewest-instructions row loop) 14 / 10 / 12.5 / 15 / 11 / 14.5, times 1.5 per warp.  A band starts
// `lag` steps after the band above it (lane skew + 48 steps of poll look-ahead + ~60 steps of L2 visibility);
// the pair is done when the last band is.  The estimate only steers the choice of kernel, never the result.
double estimate(long long LQ, long long LT, int mode, int R, int config, int sms, bool two_sided = false) {
  const int rpb = swb::rows_per_band(R, mode);
  const long long NB = (LQ + rpb - 1) / rpb;
  const int wpc = swb::config_wpc(config), slack = swb::config_slack(config);
  const long long W = (long long)sms * wpc;
  const int skew = swb::config_skew(config, mode);
  static const double kPerRowShort[10] = {13.2, 7.0, 12.0, 15.6, 9.8, 14.0, 14.0, 16.0, 14.5, 16.5};
  static const double kPerRowLong[10] = {14.0, 10.0, 12.5, 15.0, 11.0, 14.5, 14.5, 16.5, 15.0, 17.0};
  const double per_row = (config == 2 ? kPerRowLong : kPerRowShort)[mode];
  double cyc_step = per_row * R + (config == 2 ? 39.0 : 31.0);
  if (config != 2) cyc_step = std::max(cyc_step, 48.0);      // latency floor of a step with one warp per scheduler (r02_diag: R=2 -> 48.7)
  if (config == 2) cyc_step *= 1.5;
  if (config == 3) cyc_step += std::max(0.0, 30.0 - ((mode == 1 || mode == 4) ? 4.0 : 6.0) * R);   // exposed SHFL latency
  const double lag = skew + 48 + 26;        // 32 steps of poll granularity + 16 of speculative look-ahead + visibility
                                            // (measured with %globaltimer stamps per band: 168 steps at skew 94, profiles/r02_diag_baseline.txt)
  if (two_sided) {            // each half has half the bands and half the warps
    const long long NBh = (NB + 1) / 2, Wh = std::max<long long>(W / 2, 1);
    const long long b = NBh - 1, w = b % Wh, r = b / Wh;
    const double start = std::max((double)w * lag + (double)r * (double)(LT + skew), (double)b * lag);
    return (start + (double)(LT + skew)) * cyc_step + 30000.0;      // + the combination kernel
  }
  const long long b = NB - 1, w = b % W, r = b / W;
  const double start = std::max((double)w * lag + (double)r * (double)(LT + skew), (double)b * lag);
  return (start + (double)(LT + skew)) * cyc_step;
}

struct Plan;
const void* kernel_for(const Plan& pl);

// The CTA-chained engine (launch config 7): one band per warp, four consecutive bands per CTA.  Same model as
// estimate(): a band starts `lag` steps after the band above it, but three of four hand-offs stay in shared memory
// and the compute warps carry no chunk prologue.  1e300: this shape does not fit (the caller keeps the other engine).
double estimate_chain(long long LQ, long long LT, int mode, int R, int sms, bool two_sided) {
  if ((mode != 0 && mode != 1) || !swb::chain_kernel(mode, R)) return 1e300;
  const int rpb = swb::rows_per_band(R, mode);
  const long long NB = (LQ + rpb - 1) / rpb;
  const long long NB0 = two_sided ? NB / 2 : NB, NB1 = two_sided ? NB - NB0 : 0;
  if (two_sided && NB0 < 4) return 1e300;
  if ((NB0 + 3) / 4 + (NB1 + 3) / 4 > sms) return 1e300;
  // fitted on one-sided sweeps of a 100 000-row Q against T of 25 000 ... 400 000 (bench/chain_fit.py, profiles/r02_chain_fit.txt):
  // groups of 32 steps: 44.0 cycles per step at R = 3 linear, a band starts 150 steps after the band above it;
  // groups of 16 steps: 67.9 cycles per step at R = 3 affine, 125 steps.  With the helper warps placed as they are now
  // (swb_chain.cuh, SWB_CHAIN_HELPER_WARP): 42.8 and 65.7 on cfg2.
  const bool g32 = swb::chain_group(mode, R) == 32;
  // Linear kernels, from profiles/r02_plancheck.txt (end of round 2): R = 2 / 3 in groups of 32: 40.1 / 42.8; R = 4 / 6 / 8 in
  // groups of 16: 60.4 / 75.1 / 88.5 = 7 R + 32.5.  (The earlier 7 R + 23 made R = 2 look 4 % cheaper than R = 3 below
  // 100 000 rows; measured it is 6-7 % dearer.)  The groups-of-16 term is entered as 7 R + 29.5: the pair engine's own
  // estimate is 4-5 % optimistic at 200 000 - 250 000 rows, where the chained engine measures 3-4 % faster.
  const double cyc_step = mode == 1 ? (g32 ? (R >= 3 ? 42.8 : (R == 2 ? 40.1 : 39.0)) : 7.0 * R + 29.5) : 13.2 * R + 26.1;
  const double lag = g32 ? 150.0 : 125.0;
  const double bands = (double)std::max(NB0, NB1);
  return ((bands - 1.0) * lag + (double)(LT + swb::kChainSkew)) * cyc_step + (two_sided ? 30000.0 : 0.0);
}

Plan make_plan(long long n, long long m, const swb200_params& p, const swb200_options& o, int lanes, int sms,
               bool allow_two_sided = false, bool allow_chain = false) {
  Plan pl{};
  pl.swap = o.orient ? o.orient == 2 : m > n;   // default: stripe the longer sequence across lanes
  const long long LQ = pl.swap ? m : n, LT = pl.swap ? n : m;
  // lanes: 16 = packed s16, 17 = packed s16 re-based, 32 = s32
  pl.mode = lanes == 32 ? 2 : ((p.gap_init == p.gap_ext && !o.no_linear) ? 1 : 0);
  if (lanes == 17) pl.mode += 3;
  if (lanes == 33) pl.mode = 5;          // 32-bit lanes, any byte alphabet
  if (lanes == 34) pl.mode = 6;          // 32-bit lanes + position of the maximum
  if (lanes == 35) pl.mode = 7;          // the same for any byte alphabet
  if (lanes == 36) pl.mode = 8;          // anchored recurrence + position of the maximum (start-cell pass)
  if (lanes == 37) pl.mode = 9;
  if (lanes == 38) pl.mode = 10;         // anchored recurrence + traceback directions (swb200_align)
  if (lanes == 39) pl.mode = 11;
  if (pl.mode >= 10) {                   // one kernel shape: 8 rows per lane (one direction word per step)
    pl.R = 8; pl.config = o.config == 3 ? 3 : 1; pl.two_sided = false; pl.ctas = o.ctas;
    return pl;
  }
  double best = 1e300;
  for (int ci = 1; ci <= swb::kNumConfigs; ++ci) {
    if (o.config && o.config != ci) continue;
    if (ci > 3 && (swb::mode_is_s32(pl.mode) || !o.config)) continue;      // configs 4-6: 16-bit lanes, and only on request
    { Plan probe = pl; probe.R = 1; probe.config = ci; if (!kernel_for(probe)) continue; }
    for (int ri = 0; ri < swb::kNumRowChoices; ++ri) {
      const int R = swb::kRowChoices[ri];
      if (o.rows && o.rows != R) continue;
      const double e = estimate(LQ, LT, pl.mode, R, ci, sms);
      if (e < best && !(o.two_sided > 0 && pl.two_sided)) { best = e; pl.R = R; pl.config = ci; pl.two_sided = false; }
      // two-sided: packed 16-bit lanes (plain or re-based), at least 4 bands per half
      if (allow_two_sided && (pl.mode <= 1 || pl.mode == 3 || pl.mode == 4) && o.two_sided >= 0 &&
          LQ >= 8LL * swb::rows_per_band(R, pl.mode)) {
        const double e2 = estimate(LQ, LT, pl.mode, R, ci, sms, true);
        // a two-sided plan must beat a one-sided one by 3 % (it costs four more small launches); among two-sided plans
        // the cheaper one wins
        const bool better = pl.two_sided ? e2 < best : (e2 < 0.97 * best || o.two_sided > 0);
        if (better) { best = std::min(best, e2); pl.R = R; pl.config = ci; pl.two_sided = true; }
      }
    }
  }
  // the CTA-chained engine: on request (config 7), or by itself when its estimate beats the best plan above
  if (allow_chain && (o.config == swb::kChainConfig || (o.config == 0 && settings().chain > 0))) {
    for (int ri = 0; ri < swb::kNumRowChoices; ++ri) {
      const int R = swb::kRowChoices[ri];
      if (o.rows && o.rows != R) continue;
      for (int t2 = 0; t2 < 2; ++t2) {
        if (t2 ? (!allow_two_sided || o.two_sided < 0 || LQ < 8LL * swb::rows_per_band(R, pl.mode)) : o.two_sided > 0) continue;
        const double e = estimate_chain(LQ, LT, pl.mode, R, sms, t2 != 0);
        if (e < best) { best = e; pl.R = R; pl.config = swb::kChainConfig; pl.two_sided = t2 != 0; }
      }
    }
  }
  if (best == 1e300) { pl.R = o.rows ? o.rows : 4; pl.config = (o.config && o.config != swb::kChainConfig) ? o.config : 1; }
  pl.ctas = o.ctas;
  return pl;
}

const void* kernel_for(const Plan& pl) {
  switch (pl.mode) {
    case 0: return swb::engine_kernel_mode0(pl.R, pl.config);
    case 1: return swb::engine_kernel_mode1(pl.R, pl.config);
    case 2: return swb::engine_kernel_mode2(pl.R, pl.config);
    case 3: return swb::engine_kernel_mode3(pl.R, pl.config);
    case 4: return swb::engine_kernel_mode4(pl.R, pl.config);
    case 6: return swb::engine_kernel_mode6(pl.R, pl.config);
    case 7: return swb::engine_kernel_mode7(pl.R, pl.config);
    case 8: return swb::engine_kernel_mode8(pl.R, pl.config);
    case 9: return swb::engine_kernel_mode9(pl.R, pl.config);
    case 10: return swb::engine_kernel_mode10(pl.R, pl.config);
    case 11: return swb::engine_kernel_mode11(pl.R, pl.config);
    default: return swb::engine_kernel_mode5(pl.R, pl.config);
  }
}

int log2_ceil(long long v) { int s = 0; while ((1LL << s) < v) ++s; return s; }

// Present when the pair is spread over a ring of GPUs (one swb200_ring per rank).
struct RingCfg {
  int rank, world;
  uint2* inbound;        // this rank's region (consumed by local warp 0 of each half)
  uint2* next_inbound;   // the next rank's region, mapped into this process (peer stores over NVLink)
  size_t len;            // region unit (see swb200_ring)
  unsigned call_epoch;   // 1..16383, identical on all ranks for one collective call
  uint2* root;           // rank 0's region, or null (then the plan is one-sided)
  RingCombine* combine;  // filled in when the run was two-sided: the root combines after every rank has finished
};

// One launch of a blocked traceback (swb200_align): the direction kernel runs only the bands [band0, band1) of the span.
struct DirBlock {
  long long band0, band1;
  const uint2* top;      // checkpoint row above band0 (null: band0 == 0, the anchored row-0 border)
  uint2* bottom;         // where band1 - 1 leaves its bottom row (null: not wanted)
  int lanes;             // in/out: the lane width the first launch settled on (0: not yet), and the symbol table it needed
  const uint8_t* lut;
};

// Encode + one engine run at a fixed lane width.  d_seq1/d_seq2 are device pointers.
int run_once(swb200_ctx* c, const uint8_t* d_seq1, long long n, const uint8_t* d_seq2, long long m,
             const swb200_params& p, const swb200_options& o, int lanes, const uint8_t* d_lut, cudaStream_t s,
             int* score, int* status, const RingCfg* ring = nullptr, int* end3 = nullptr, const DirBlock* blk = nullptr) {
  const int world = ring ? ring->world : 1;
  const Plan pl = make_plan(n, m, p, o, lanes, c->sms * world, /*allow_two_sided=*/ring == nullptr || ring->root != nullptr,
                            /*allow_chain=*/ring == nullptr);
  const bool chain = pl.config == swb::kChainConfig;        // CTA-chained engine: plain 16-bit lanes, one band per warp, one GPU
  const void* kern = chain ? swb::chain_kernel(pl.mode, pl.R) : kernel_for(pl);
  if (!kern) return fail(SWB200_ERR_ARG, "no kernel for rows=" + std::to_string(pl.R));
  const uint8_t* dq = pl.swap ? d_seq2 : d_seq1;
  const uint8_t* dt = pl.swap ? d_seq1 : d_seq2;
  const long long LQ = pl.swap ? m : n, LT = pl.swap ? n : m;
  const int wpc = swb::config_wpc(pl.config), slack = swb::config_slack(pl.config);
  const int rpb = swb::rows_per_band(pl.R, pl.mode);
  const long long NB = (LQ + rpb - 1) / rpb;
  if ((pl.mode == 3 || pl.mode == 4) && !rebase_is_safe(p, pl.R))
    return fail(SWB200_ERR_ARG, "re-based lanes are not safe for these scoring parameters / row count");
  if (NB >= (1 << 18)) return fail(SWB200_ERR_ARG, "sequence too long for this row count (bands >= 2^18)");
  if (LT >= (1LL << 30)) return fail(SWB200_ERR_ARG, "streamed sequence too long (>= 2^30)");       // 32-bit step arithmetic
  if (ring && NB > 1 && ring->call_epoch == 0) return fail(SWB200_ERR_ARG, "ring epoch exhausted; create a new ring");
  // two-sided sweep: rows [0, mid) forward, rows [mid, LQ) reversed (with pad rows in front so that the reversed
  // half also ends exactly on a band boundary); mid is a multiple of the band height
  const bool ts = pl.two_sided;
  const long long NB0 = ts ? NB / 2 : NB;
  const long long mid = NB0 * rpb;
  const long long LQ1 = ts ? LQ - mid : 0, NB1 = ts ? (LQ1 + rpb - 1) / rpb : 0, pad1 = NB1 * rpb - LQ1;

  int per_sm = 0;
  SWB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, chain ? swb::kChainThreads : wpc * 32, 0));
  if (per_sm < 1) return fail(SWB200_ERR_CUDA, "engine kernel does not fit on an SM");
  if (blk && (pl.mode < 10 || ts || ring || blk->band0 < 0 || blk->band1 > NB || blk->band0 >= blk->band1))
    return fail(SWB200_ERR_ARG, "internal: bad traceback block");
  const long long want_warps = blk ? blk->band1 - blk->band0 : (ts ? 2 * std::max(NB0, NB1) : NB);
  long long ctas = std::min<long long>((want_warps + wpc - 1) / wpc, (long long)c->sms);   // one CTA per SM
  if (pl.ctas > 0) ctas = std::min<long long>(ctas, pl.ctas);
  ctas = std::max<long long>(ctas, ts ? 2 : 1);
  if (ring) ctas = pl.ctas > 0 ? std::min<long long>(pl.ctas, c->sms) : c->sms;   // every rank launches the same shape
  const long long chain_ctas0 = (NB0 + 3) / 4, chain_ctas1 = (NB1 + 3) / 4;         // a chained CTA owns four consecutive bands
  if (chain) {
    if (ring || chain_ctas0 + chain_ctas1 > (long long)c->sms)
      return fail(SWB200_ERR_ARG, "launch config 7 needs one band per warp on one GPU (more rows per sub-lane, or another config)");
    ctas = chain_ctas0 + chain_ctas1;
  }
  const int warps = (int)ctas * wpc;
  const int split = ts ? warps / 2 : 0;

  const int skew = swb::config_skew(pl.config, pl.mode);
  const int align = swb::mode_is_s32(pl.mode) ? swb::kChunk : swb::kBlock;     // steps per band: whole chunks / whole blocks
  const long long nsteps = ((LT + skew + align - 1) / align) * align;
  const int ext_shift = std::max(4, log2_ceil(nsteps + swb::kChunk));
  const long long ext_len = 1LL << ext_shift;
  // inner rings: at most 256 laps (8-bit lap tag), at least 4096 entries
  int link_shift = std::max(12, log2_ceil((nsteps + 255) / 256));
  const long long link_len = 1LL << link_shift;

  int rc;
  if ((rc = grow(c->d_q, c->q_cap, (size_t)LQ + 64, false, s))) return rc;
  if ((rc = grow(c->d_t, c->t_cap, (size_t)(LT / 32 + 8), false, s))) return rc;
  if (ts) {
    if ((rc = grow(c->d_q2, c->q2_cap, (size_t)(NB1 * rpb) + 64, false, s))) return rc;
    if ((rc = grow(c->d_t2, c->t2_cap, (size_t)(LT / 32 + 8), false, s))) return rc;
    if (!ring && (rc = grow(c->d_final, c->final_cap, 4 * (size_t)ext_len, false, s))) return rc;
  }
  const size_t links_need = (size_t)std::max(warps, 1) * 2 * (size_t)link_len;
  const size_t ext_need = (ts ? 4 : 2) * (size_t)ext_len;
  if ((rc = grow(c->d_links, c->links_cap, links_need, true, s))) return rc;
  const long long chain_stride = nsteps + 64;
  if (chain && (rc = grow(c->d_chain, c->chain_cap, (size_t)ctas * (size_t)chain_stride, true, s))) return rc;
  if (ring) {
    if ((size_t)ext_len > ring->len)
      return fail(SWB200_ERR_ARG, "ring was created for a shorter streamed sequence (max_len too small)");
  } else if ((rc = grow(c->d_ext, c->ext_cap, ext_need, true, s))) return rc;
  if ((rc = grow(c->d_progress, c->progress_cap, (size_t)warps + 4, false, s))) return rc;
  const bool dirs = pl.mode >= 10;
  if (dirs) {
    if (ring || !blk) return fail(SWB200_ERR_ARG, "traceback runs on one GPU through swb200_align");
    const size_t words = (size_t)(blk->band1 - blk->band0) * (size_t)nsteps * 32;   // swb200_align chose the block to fit
    if ((rc = grow(c->d_dirs, c->dirs_cap, words, false, s))) return rc;
  }
  const bool track = pl.mode >= 6 && pl.mode <= 9;
  if (track && (ring || !end3)) return fail(SWB200_ERR_ARG, "end-cell tracking runs on one GPU through swb200_score_end");
  if (track && (rc = grow(c->d_cand, c->cand_cap, 3 * (size_t)NB + 3, false, s))) return rc;

  // tags carry a 6-bit epoch; when it wraps, forget every old tag
  c->epoch += 1;
  if (c->epoch > 63) {
    c->epoch = 1;
    SWB_CUDA(cudaMemsetAsync(c->d_links, 0, c->links_cap * sizeof(uint2), s));
    if (c->d_chain) SWB_CUDA(cudaMemsetAsync(c->d_chain, 0, c->chain_cap * sizeof(uint2), s));
    if (c->d_ext) SWB_CUDA(cudaMemsetAsync(c->d_ext, 0, c->ext_cap * sizeof(uint2), s));
  }
  SWB_CUDA(cudaMemsetAsync(c->d_progress, 0, ((size_t)warps + 4) * sizeof(unsigned long long), s));
  SWB_CUDA(cudaMemsetAsync(c->d_result, 0, 12 * sizeof(int), s));    // [0] score, [1] status, [3..8] timeout post-mortem, [11] protocol-checker mismatches
  if (blk && blk->top) {        // the block's first band reads the checkpoint above it (T positions [0, LT): slots [skew, skew + LT))
    const long long sk0 = swb::config_skew(pl.config, pl.mode);
    const int rb = (int)std::min<long long>((LT + 255) / 256, 4LL * c->sms);
    retag_checkpoint_kernel<<<rb, 256, 0, s>>>(blk->top, c->d_ext, sk0, sk0 + LT, (c->epoch << 26) | ((uint32_t)blk->band0 << 8));
    c->info.aux_launches += 1;
  }

  const bool generic = pl.mode == 5 || pl.mode == 7 || pl.mode == 9 || pl.mode == 11;       // raw bytes straight from the caller's buffers, nothing to encode
  const int eb = (int)std::min<long long>(std::max<long long>(LQ / (16 * 256), 1), 4LL * c->sms);
  const int tb = (int)std::min<long long>(std::max<long long>((LT / 32) / 256, 1), 4LL * c->sms);
  if (!generic) {
    encode_q_kernel<<<eb, 256, 0, s>>>(dq, LQ, c->d_q, d_lut, c->d_result);
    encode_t_kernel<<<tb, 256, 0, s>>>(dt, LT, c->d_t, d_lut, c->d_result);
    c->info.aux_launches += 2;
  }
  if (ts) {
    const int eb2 = (int)std::min<long long>(std::max<long long>((NB1 * rpb) / 256, 1), 4LL * c->sms);
    encode_q_rev_kernel<<<eb2, 256, 0, s>>>(dq, LQ, mid, pad1, c->d_q2, d_lut, c->d_result);
    encode_t_rev_kernel<<<tb, 256, 0, s>>>(dt, LT, c->d_t2, d_lut, c->d_result);
    c->info.aux_launches += 2;
  }
  SWB_CUDA(cudaGetLastError());

  const size_t ring_stride = 2 * (size_t)link_len;
  swb::EngineLaunch L{};
  swb::EngineParams& P = L.a;
  P.q_codes = generic ? dq : c->d_q; P.t_packed = c->d_t; P.t_bytes = dt; P.LQ = ts ? mid : LQ; P.LT = LT; P.NB = (int)NB0;
  const int warps0 = ts ? split : warps;
  P.ring_total = warps0 * world; P.ring_offset = ring ? ring->rank * warps0 : 0; P.warps_local = warps0;
  if (blk) { P.ring_offset = (int)blk->band0; P.NB = (int)blk->band1; }      // a band window on one GPU (swb_engine.cuh, sbase)
  P.links = c->d_links; P.link_mask = (unsigned)(link_len - 1); P.link_shift = link_shift;
  P.progress = c->d_progress;
  P.ext_in = ring ? ring->inbound : c->d_ext; P.ext_out = ring ? ring->next_inbound : c->d_ext;
  P.ext_mask = (unsigned)(ext_len - 1); P.ext_shift = ext_shift;
  P.tag_base = c->epoch << 26; P.result = c->d_result;
  P.ext_tag_base = ring ? (((ring->call_epoch >> 8) & 0x3Fu) << 26) | (ring->call_epoch & 0xFFu) : P.tag_base;
  P.match = p.match; P.mismatch = p.mismatch; P.gap_init = p.gap_init; P.gap_ext = p.gap_ext;
  const Settings cfg = settings();
  P.spin_limit = cfg.spin_limit;
  P.dbg = cfg.dbg;
  long long* d_prof = nullptr;
  if (!cfg.prof_path.empty()) {           // context-owned, grow-only: nothing to leak on an early return
    if ((rc = grow(c->d_prof, c->prof_cap, (size_t)warps * 8, false, s))) return rc;
    d_prof = c->d_prof;
    SWB_CUDA(cudaMemsetAsync(d_prof, 0, (size_t)warps * 8 * sizeof(long long), s));
  }
  P.prof = d_prof;
  P.cand = track ? c->d_cand : nullptr;
  P.dirs = dirs ? c->d_dirs : nullptr;
  L.split = split;
  // the two middle boundary rows of a two-sided sweep: local buffer, or the root rank's region on a ring
  uint2* final_f = ring ? ring->root + 4 * ring->len : c->d_final;
  uint2* final_b = ring ? ring->root + 6 * ring->len : c->d_final + 2 * (size_t)ext_len;
  if (blk && blk->bottom) { P.final_out = blk->bottom; P.final_mask = (unsigned)(ext_len - 1); }
  if (ts) {
    P.final_out = final_f; P.final_mask = (unsigned)(ext_len - 1);
    swb::EngineParams& B = L.b;
    B = P;
    B.q_codes = c->d_q2; B.t_packed = c->d_t2; B.LQ = NB1 * rpb; B.NB = (int)NB1;
    B.warps_local = warps - split; B.ring_total = (warps - split) * world; B.ring_offset = ring ? ring->rank * (warps - split) : 0;
    B.links = c->d_links + (size_t)split * ring_stride;
    B.progress = c->d_progress + split + 2;
    B.ext_in = ring ? ring->inbound + 2 * ring->len : c->d_ext + 2 * (size_t)ext_len;
    B.ext_out = ring ? ring->next_inbound + 2 * ring->len : c->d_ext + 2 * (size_t)ext_len;
    B.final_out = final_b;
    B.prof = d_prof ? d_prof + 8 * (size_t)split : nullptr;
  }
  void* args[] = {&L};
  SWB_CUDA(cudaEventRecord(c->ev0, s));
  if (chain) {
    swb::ChainLaunch CL{};
    swb::ChainParams& A = CL.a;
    A.q_codes = P.q_codes; A.t_packed = P.t_packed; A.LQ = P.LQ; A.LT = (int)LT; A.NB = (int)NB0;
    A.links = c->d_chain; A.link_stride = chain_stride; A.final_out = ts ? final_f : nullptr;
    A.tag = (c->epoch << 26) | 0x5A5A5Au; A.result = c->d_result;
    A.match = p.match; A.mismatch = p.mismatch; A.gap_init = p.gap_init; A.gap_ext = p.gap_ext;
    A.spin_limit = cfg.spin_limit;
    CL.split = (int)chain_ctas0;
    if (ts) {
      swb::ChainParams& B2 = CL.b;
      B2 = A;
      B2.q_codes = c->d_q2; B2.t_packed = c->d_t2; B2.LQ = NB1 * rpb; B2.NB = (int)NB1;
      B2.links = c->d_chain + (size_t)chain_ctas0 * (size_t)chain_stride; B2.final_out = final_b;
    }
    void* cargs[] = {&CL};
    SWB_CUDA(cudaLaunchCooperativeKernel(kern, dim3((unsigned)ctas), dim3((unsigned)swb::kChainThreads), cargs, 0, s));
  } else
  SWB_CUDA(cudaLaunchCooperativeKernel(kern, dim3((unsigned)ctas), dim3((unsigned)(wpc * 32)), args, 0, s));
  if (ts && ring) {
    // the two last bands may live on any rank: the root combines once EVERY rank's kernel has finished
    *ring->combine = RingCombine{true, LT, ext_len, NB0, NB1, skew, pl.mode == 1 || pl.mode == 4, pl.mode == 3 || pl.mode == 4,
                                 p.gap_init, p.gap_ext};
  } else if (ts) {
    // re-based lanes: the final bands' bases sit in the second half of each buffer, region (band & 3) of four
    const bool rb = pl.mode == 3 || pl.mode == 4;
    const uint2* bf = rb ? final_f + (size_t)ext_len + (size_t)((NB0 - 1) & 3) * (size_t)(ext_len / 4) : nullptr;
    const uint2* bb = rb ? final_b + (size_t)ext_len + (size_t)((NB1 - 1) & 3) * (size_t)(ext_len / 4) : nullptr;
    combine_two_sided_kernel<<<2 * c->sms, 256, 0, s>>>(final_f, final_b, LT, skew,
                                                        pl.mode == 1 || pl.mode == 4, p.gap_init, p.gap_ext, bf, bb, c->d_result);
    c->info.aux_launches += 1;
  }
  if (track) {
    reduce_end_kernel<<<1, 256, 0, s>>>(c->d_cand, (int)NB, c->d_result + 24);
    c->info.aux_launches += 1;
  }
  SWB_CUDA(cudaEventRecord(c->ev1, s));
  SWB_CUDA(cudaMemcpyAsync(c->h_result, c->d_result, 12 * sizeof(int), cudaMemcpyDeviceToHost, s));
  if (track) SWB_CUDA(cudaMemcpyAsync(c->h_result + 24, c->d_result + 24, 3 * sizeof(int), cudaMemcpyDeviceToHost, s));
  SWB_CUDA(cudaStreamSynchronize(s));
  if (track) { end3[0] = c->h_result[24]; end3[1] = c->h_result[25]; end3[2] = c->h_result[26]; }
  float ms = 0;
  SWB_CUDA(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  *score = c->h_result[0];
  *status = c->h_result[1];
  if (c->h_result[10] != 0)        // only a -DSWB_CHAIN_CHECK build of swb_chain.cu counts here (bench/chain_check.sh)
    fprintf(stderr, "chaincheck: %d x 1024 steps checked (32 table reads + 1 inbox read each), %d mismatches, score %d\n", c->h_result[10], c->h_result[11], c->h_result[0]);
  if (ts && !ring && !cfg.dump_final_path.empty()) {          // debugging aid: the two middle boundary rows as the kernels wrote them
    std::vector<uint2> h(4 * (size_t)ext_len);
    cudaMemcpy(h.data(), c->d_final, h.size() * sizeof(uint2), cudaMemcpyDeviceToHost);
    FILE* f = fopen(cfg.dump_final_path.c_str(), "wb");
    if (f) {
      long long hdr[6] = {LT, skew, ext_len, mid, pad1, (long long)pl.swap};
      fwrite(hdr, sizeof hdr, 1, f); fwrite(h.data(), sizeof(uint2), h.size(), f); fclose(f);
    }
  }
  if (d_prof) {
    std::vector<long long> hp((size_t)warps * 8);
    cudaMemcpy(hp.data(), d_prof, hp.size() * sizeof(long long), cudaMemcpyDeviceToHost);
    if (cfg.prof_path == "1") {
      for (int wv = 0; wv < warps && wv < 12; ++wv)
        fprintf(stderr, "prof warp %d: prologue %.0f cyc/chunk, steps %.0f cyc/chunk, failed polls %.2f/chunk, chunks %lld\n", wv,
                hp[8 * wv + 3] ? (double)hp[8 * wv] / hp[8 * wv + 3] : 0.0, hp[8 * wv + 3] ? (double)hp[8 * wv + 1] / hp[8 * wv + 3] : 0.0,
                hp[8 * wv + 3] ? (double)hp[8 * wv + 2] / hp[8 * wv + 3] : 0.0, hp[8 * wv + 3]);
    } else if (FILE* f = fopen(cfg.prof_path.c_str(), "a")) {
      // one JSON line per launch: per warp [prologue cycles, step cycles, failed polls, chunks, t_start ns, t_end ns, SM]
      fprintf(f, "{\"mode\": %d, \"R\": %d, \"config\": %d, \"ctas\": %lld, \"NB\": %lld, \"LT\": %lld, \"two_sided\": %d, \"split\": %d, \"ms\": %.4f, \"warps\": [",
              pl.mode, pl.R, pl.config, ctas, NB, LT, (int)ts, split, ms);
      for (int wv = 0; wv < warps; ++wv)
        fprintf(f, "%s[%lld,%lld,%lld,%lld,%lld,%lld,%lld]", wv ? "," : "", hp[8 * wv], hp[8 * wv + 1], hp[8 * wv + 2], hp[8 * wv + 3],
                hp[8 * wv + 4], hp[8 * wv + 5], hp[8 * wv + 6]);
      fprintf(f, "]}\n");
      fclose(f);
    }
  }
  if ((*status & swb::STATUS_SPIN_TIMEOUT) && cfg.debug)
    fprintf(stderr, "libswb200: timeout kind=%d a=%d(0x%x) b=%d(0x%x) c=%d d=%d thread=%d  [mode=%d R=%d config=%d ctas=%lld NB=%lld LT=%lld link_len=%lld ext_len=%lld epoch=%u ts=%d]\n",
            c->h_result[3], c->h_result[4], c->h_result[4], c->h_result[5], c->h_result[5], c->h_result[6], c->h_result[7],
            c->h_result[8], pl.mode, pl.R, pl.config, ctas, NB, LT, link_len, ext_len, c->epoch, (int)ts);
  c->info.lanes = swb::mode_is_s32(pl.mode) ? 32 : 16; c->info.rebased = pl.mode == 3 || pl.mode == 4;
  c->info.linear = pl.mode == 1 || pl.mode == 4;
  c->info.two_sided = ts;
  c->info.rows = pl.R; c->info.config = pl.config;
  c->info.ctas = (int)ctas; c->info.warps = warps; c->info.bands = (int)NB; c->info.engine_launches += 1;
  c->info.engine_ms = ms;
  c->last_nsteps = nsteps; c->last_skew_per_lane = swb::mode_is_s32(pl.mode) ? 1 + slack : 0;
  return SWB200_OK;
}

// Full policy for one pair whose bytes are in device memory.
// end_out != nullptr: also report the end cell {i_end (1-based position in seq2), j_end (in seq1)} of the best local
// alignment -- among cells with the maximal score the one with the smallest j, then the smallest i; {0, 0} for
// score 0.  Runs the 32-bit tracking kernel with seq2 striped and seq1 streamed, whatever the options say.
int score_device_locked(swb200_ctx* c, const uint8_t* d_seq1, long long n, const uint8_t* d_seq2, long long m,
                        const swb200_params* pp, const swb200_options* oo, cudaStream_t s, int* score_out,
                        long long* end_out = nullptr, bool anchored = false, bool record_dirs = false,
                        DirBlock* blk = nullptr) {
  const swb200_params p = params_or_default(pp);
  swb200_options o = options_or_default(oo);
  if (end_out || record_dirs) { o.orient = 2; o.lanes = 0; o.two_sided = -1; o.rebase = -1; if (o.rows > 16) o.rows = 16; }
  int rc;
  if ((rc = check_params(p))) return rc;
  if (n < 0 || m < 0 || !score_out) return fail(SWB200_ERR_ARG, "negative length or null output");
  if (o.lanes != 0 && o.lanes != 16 && o.lanes != 32) return fail(SWB200_ERR_ARG, "lanes must be 0, 16 or 32");
  c->info = swb200_run_info{};
  c->info.cells = n * m;
  if (end_out) { end_out[0] = 0; end_out[1] = 0; }
  if (n == 0 || m == 0) { *score_out = 0; return SWB200_OK; }   // both reference oracles return 0 here
  if (end_out && ((long long)p.match * std::min(n, m) >= (1LL << 20) || std::max(n, m) >= (1LL << 30)))
    return fail(SWB200_ERR_RANGE, "end-cell tracking needs match*min(n,m) < 2^20");
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));

  const uint8_t* lut = nullptr;
  // Lane width policy.  A score is at most match*min(n,m).  If that fits, plain 16-bit lanes.  Otherwise random
  // DNA still scores only ~0.11*N, so up to 8x the range we try plain 16-bit first (the kernel reports leaving
  // the range; the re-based kernel is ~10% slower) and beyond that go straight to re-based 16-bit lanes;
  // 32-bit lanes are the last resort.
  const long long bound = (long long)p.match * std::min(n, m);
  const bool rb_ok = o.rebase >= 0 && o.lanes != 32 && rebase_is_safe(p, o.rows ? o.rows : 16);
  int lanes = o.lanes == 32 ? 32 : 16;
  if (o.lanes != 32 && rb_ok && (o.rebase > 0 || bound > 8LL * 32767)) lanes = 17;
  if (end_out) lanes = anchored ? 36 : 34;
  if (record_dirs) lanes = 38;           // anchored + traceback directions; seq2 striped, seq1 streamed (o.orient = 2 from the caller)
  if (blk && blk->lanes) { lanes = blk->lanes; lut = blk->lut; }   // later launches of a blocked traceback: as the first one settled
  int end3[3] = {0, 0, 0};
  // a score can never exceed match*min(n,m): skip the 16-bit attempt when it cannot fit anyway?  No:
  // random DNA scores ~0.11*N, so 16-bit lanes are right far beyond N = 32767; the engine reports
  // leaving the range and we repeat in 32 bits (bit-exact either way).
  for (int attempt = 0; attempt < 4; ++attempt) {
    int score = 0, status = 0;
    if ((rc = run_once(c, d_seq1, n, d_seq2, m, p, o, lanes, lut, s, &score, &status, nullptr, end_out ? end3 : nullptr, blk))) return rc;
    if (status & swb::STATUS_SPIN_TIMEOUT) return fail(SWB200_ERR_TIMEOUT, "boundary hand-off timed out");
    if ((status & swb::STATUS_BAD_SYMBOL) && lanes != 33 && lanes != 35 && lanes != 37 && lanes != 39) {
      if (lut) return fail(SWB200_ERR_ALPHABET, "internal: remapped symbols still out of range");
      // bytes other than A,C,G,T: remap the (at most 4) distinct values that occur
      SWB_CUDA(cudaMemsetAsync(c->d_result + 16, 0, 8 * sizeof(int), s));
      presence_kernel<<<2 * c->sms, 256, 0, s>>>(d_seq1, n, reinterpret_cast<uint32_t*>(c->d_result + 16));
      presence_kernel<<<2 * c->sms, 256, 0, s>>>(d_seq2, m, reinterpret_cast<uint32_t*>(c->d_result + 16));
      c->info.aux_launches += 2;
      SWB_CUDA(cudaMemcpyAsync(c->h_result + 16, c->d_result + 16, 8 * sizeof(int), cudaMemcpyDeviceToHost, s));
      SWB_CUDA(cudaStreamSynchronize(s));
      uint8_t table[256];
      memset(table, 4, sizeof table);
      int distinct = 0;
      for (int v = 0; v < 256; ++v)
        if ((reinterpret_cast<uint32_t*>(c->h_result + 16)[v >> 5] >> (v & 31)) & 1u) {
          if (distinct < 4) table[v] = (uint8_t)distinct;
          ++distinct;
        }
      if (distinct > 4) {
        // the reference compares raw bytes (main.cpp:28-33): score such pairs with the byte-compare kernel
        lanes = record_dirs ? 39 : (end_out ? (anchored ? 37 : 35) : 33);
        continue;
      }
      SWB_CUDA(cudaMemcpyAsync(c->d_lut, table, 256, cudaMemcpyHostToDevice, s));
      SWB_CUDA(cudaStreamSynchronize(s));
      lut = c->d_lut;
      continue;
    }
    if (status & swb::STATUS_REBASE_RANGE) {
      lanes = 32;                   // never observed; the 32-bit kernel has no such limit
      continue;
    }
    if (status & swb::STATUS_S16_OVERFLOW) {
      if (o.lanes == 16 && o.rebase < 0) return fail(SWB200_ERR_RANGE, "score leaves the 16-bit lane range");
      lanes = rb_ok ? 17 : 32;
      if (o.lanes == 16 && !rb_ok) return fail(SWB200_ERR_RANGE, "score leaves the 16-bit lane range");
      continue;
    }
    *score_out = score;
    if (blk) { blk->lanes = lanes; blk->lut = lut; }
    if (end_out && score > 0) {
      if (end3[0] != score) return fail(SWB200_ERR_CUDA, "internal: tracked maximum differs from the score");
      end_out[0] = (long long)end3[2] + 1;      // Q row -> position in seq2
      end_out[1] = (long long)end3[1] + 1;      // T position -> position in seq1
    }
    return SWB200_OK;
  }
  return fail(SWB200_ERR_CUDA, "internal: retry budget exhausted");
}

std::mutex g_default_mu;
swb200_ctx* g_default_ctx = nullptr;

int default_ctx(swb200_ctx** out) {
  std::lock_guard<std::mutex> lk(g_default_mu);
  if (!g_default_ctx) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
    int rc = swb200_ctx_create(dev, &g_default_ctx);
    if (rc) return rc;
  }
  *out = g_default_ctx;
  return SWB200_OK;
}

int legacy(const unsigned char* a, const unsigned char* b, int n, int m, const char* who) {
  int score = 0;
  const int rc = swb200_score(a, n, b, m, nullptr, &score);
  if (rc != SWB200_OK) {
    // The reference signature has no error channel (SURVEY.md 8b): never return a made-up score.
    fprintf(stderr, "libswb200: %s failed (%d): %s\n", who, rc, swb200_last_error());
    abort();
  }
  return score;
}

}  // namespace

static bool pool_last_run(swb200_run_info* info);
// host pair call: 1 = not a case for the device pool (score it on one GPU), otherwise the call's return code
static int score_pair_on_pool(const unsigned char* seq1, long long n, const unsigned char* seq2, long long m,
                              const swb200_params* p, const swb200_options* opt, int* score_out);

// ---------------------------------------------------------------------------------------------
//  exported C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

const char* swb200_last_error(void) { return g_err.c_str(); }

int swb200_configure(const char* key, const char* value) {
  if (!key || !value) return fail(SWB200_ERR_ARG, "null key or value");
  std::lock_guard<std::mutex> lk(g_settings_mu);
  Settings& st = settings_locked();
  const std::string k = key;
  if (k == "spin_limit") st.spin_limit = atoll(value);
  else if (k == "dbg") st.dbg = atoi(value);
  else if (k == "debug") st.debug = atoi(value) != 0;
  else if (k == "prof") st.prof_path = value;
  else if (k == "dump_final") st.dump_final_path = value;
  else if (k == "batch_chunk_bytes") st.batch_chunk_bytes = std::max(0LL, atoll(value));
  else if (k == "ring_min_cells") st.ring_min_cells = std::max(1LL, atoll(value));
  else if (k == "chain") st.chain = atoi(value);
  else if (k == "align_block_rows") {
    char* end = nullptr;
    const long long v = strtoll(value, &end, 10);
    if (end == value || *end || v < 0 || v % swb::kDirBandRows)
      return fail(SWB200_ERR_ARG, "align_block_rows must be 0 or a positive multiple of 256");
    st.align_block_rows = v;
  }
  else return fail(SWB200_ERR_ARG, "unknown setting: " + k);
  return SWB200_OK;
}

// Diagnostic: what the planner would run for a pair (no GPU needed): out = {mode, rows, config, two_sided}, *est_cycles
// = its cost estimate.  lanes: 16 packed, 17 packed re-based, 32; sms: SMs of ALL GPUs taking part.
int swb200_plan(long long n, long long m, const swb200_params* pp, const swb200_options* oo, int lanes, int sms,
                int allow_two_sided, int out[4], double* est_cycles) {
  if (!out || n < 1 || m < 1 || sms < 1) return fail(SWB200_ERR_ARG, "bad plan arguments");
  const swb200_params p = params_or_default(pp);
  const swb200_options o = options_or_default(oo);
  const Plan pl = make_plan(n, m, p, o, lanes, sms, allow_two_sided != 0, /*allow_chain=*/allow_two_sided != 0);
  out[0] = pl.mode; out[1] = pl.R; out[2] = pl.config; out[3] = pl.two_sided ? 1 : 0;
  if (est_cycles) {
    const long long LQ = pl.swap ? m : n, LT = pl.swap ? n : m;
    *est_cycles = pl.config == swb::kChainConfig ? estimate_chain(LQ, LT, pl.mode, pl.R, sms, pl.two_sided)
                                                 : estimate(LQ, LT, pl.mode, pl.R, pl.config, sms, pl.two_sided);
  }
  return SWB200_OK;
}

int swb200_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int swb200_ctx_create(int device, swb200_ctx** ctx_out) {
  if (!ctx_out) return fail(SWB200_ERR_ARG, "null ctx_out");
  *ctx_out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(SWB200_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e));
  if (device < 0 || device >= count) return fail(SWB200_ERR_ARG, "device index out of range");
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SWB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(SWB200_ERR_CUDA, std::string("libswb200 is built for sm_100a (B200) only; found ") + prop.name);
  int coop = 0;
  SWB_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
  if (!coop) return fail(SWB200_ERR_CUDA, "device lacks cooperative launch");
  std::unique_ptr<swb200_ctx, CtxDeleter> c(new swb200_ctx());
  c->device = device;
  c->sms = prop.multiProcessorCount;
  SWB_CUDA(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
  SWB_CUDA(cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking));
  SWB_CUDA(cudaEventCreate(&c->ev0));
  SWB_CUDA(cudaEventCreate(&c->ev1));
  SWB_CUDA(cudaMalloc(&c->d_result, 32 * sizeof(int)));
  SWB_CUDA(cudaMalloc(&c->d_lut, 256));
  SWB_CUDA(cudaMallocHost(&c->h_result, 32 * sizeof(int)));
  *ctx_out = c.release();
  return SWB200_OK;
}

void swb200_ctx_destroy(swb200_ctx* c) {
  if (!c) return;
  DeviceGuard guard;
  cudaSetDevice(c->device);
  cudaFree(c->d_ascii); cudaFree(c->d_q); cudaFree(c->d_t); cudaFree(c->d_q2); cudaFree(c->d_t2); cudaFree(c->d_final); cudaFree(c->d_links); cudaFree(c->d_chain); cudaFree(c->d_ext);
  cudaFree(c->d_dirs); cudaFree(c->d_ops); cudaFree(c->d_ckpt); cudaFree(c->d_prof); cudaFree(c->d_progress); cudaFree(c->d_cand); cudaFree(c->d_rev); cudaFree(c->d_result); cudaFree(c->d_lut);
  cudaFree(c->hb_seq1); cudaFree(c->hb_seq2); cudaFree(c->hb_off1); cudaFree(c->hb_off2); cudaFree(c->hb_len1); cudaFree(c->hb_len2);
  cudaFree(c->hb_scores); cudaFree(c->hb_qw); cudaFree(c->hb_tw); cudaFree(c->hb_ql); cudaFree(c->hb_tl);
  cudaFree(c->ab_col); cudaFree(c->ab_slot); cudaFree(c->ab_pool); cudaFree(c->ab_list); cudaFree(c->ab_misc);
  cudaFree(c->lb_bnd); cudaFree(c->lb_next);
  cudaFree(c->hb_spans); cudaFree(c->hb_ops); cudaFree(c->hb_opsn);
  if (c->h_result) cudaFreeHost(c->h_result);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
  for (cudaEvent_t e : c->chunk_events) cudaEventDestroy(e);
  delete c;
}

int swb200_score_device(swb200_ctx* c, const unsigned char* d_seq1, long long n, const unsigned char* d_seq2,
                        long long m, const swb200_params* p, const swb200_options* opt, void* stream,
                        int* score_out) {
  if (!c) return fail(SWB200_ERR_ARG, "null context");
  std::lock_guard<std::mutex> lk(c->mu);
  return score_device_locked(c, d_seq1, n, d_seq2, m, p, opt, (cudaStream_t)stream, score_out);
}

int swb200_score_ex(const unsigned char* seq1, long long n, const unsigned char* seq2, long long m,
                    const swb200_params* p, const swb200_options* opt, int* score_out) {
  if (n < 0 || m < 0 || !score_out || (n > 0 && !seq1) || (m > 0 && !seq2))
    return fail(SWB200_ERR_ARG, "bad sequence arguments");
  if (n == 0 || m == 0) {
    if (p) { int rc = check_params(*p); if (rc) return rc; }
    *score_out = 0;
    return SWB200_OK;
  }
  if (const int prc = score_pair_on_pool(seq1, n, seq2, m, p, opt, score_out); prc != 1) return prc;
  swb200_ctx* c = nullptr;
  int rc = default_ctx(&c);
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = c->own_stream;
  // both sequences into one staging buffer, 256-byte aligned so the encoders can use 128-bit reads
  const size_t off2 = ((size_t)n + 255) & ~(size_t)255;
  if ((rc = grow(c->d_ascii, c->ascii_cap, off2 + (size_t)m + 256, false, s))) return rc;
  SWB_CUDA(cudaMemcpyAsync(c->d_ascii, seq1, (size_t)n, cudaMemcpyHostToDevice, s));
  SWB_CUDA(cudaMemcpyAsync(c->d_ascii + off2, seq2, (size_t)m, cudaMemcpyHostToDevice, s));
  return score_device_locked(c, c->d_ascii, n, c->d_ascii + off2, m, p, opt, s, score_out);
}

int swb200_score_end_device(swb200_ctx* c, const unsigned char* d_seq1, long long n, const unsigned char* d_seq2,
                            long long m, const swb200_params* p, void* stream, int* score_out, long long* i_end,
                            long long* j_end) {
  if (!c || !i_end || !j_end) return fail(SWB200_ERR_ARG, "null context or output");
  std::lock_guard<std::mutex> lk(c->mu);
  long long e[2] = {0, 0};
  const int rc = score_device_locked(c, d_seq1, n, d_seq2, m, p, nullptr, (cudaStream_t)stream, score_out, e);
  *i_end = e[0]; *j_end = e[1];
  return rc;
}

int swb200_score_end(const unsigned char* seq1, long long n, const unsigned char* seq2, long long m,
                     const swb200_params* p, int* score_out, long long* i_end, long long* j_end) {
  if (n < 0 || m < 0 || !score_out || !i_end || !j_end || (n > 0 && !seq1) || (m > 0 && !seq2))
    return fail(SWB200_ERR_ARG, "bad sequence arguments");
  *i_end = 0; *j_end = 0;
  if (n == 0 || m == 0) {
    if (p) { int rc = check_params(*p); if (rc) return rc; }
    *score_out = 0;
    return SWB200_OK;
  }
  swb200_ctx* c = nullptr;
  int rc = default_ctx(&c);
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = c->own_stream;
  const size_t off2 = ((size_t)n + 255) & ~(size_t)255;
  if ((rc = grow(c->d_ascii, c->ascii_cap, off2 + (size_t)m + 256, false, s))) return rc;
  SWB_CUDA(cudaMemcpyAsync(c->d_ascii, seq1, (size_t)n, cudaMemcpyHostToDevice, s));
  SWB_CUDA(cudaMemcpyAsync(c->d_ascii + off2, seq2, (size_t)m, cudaMemcpyHostToDevice, s));
  long long e[2] = {0, 0};
  rc = score_device_locked(c, c->d_ascii, n, c->d_ascii + off2, m, p, nullptr, s, score_out, e);
  *i_end = e[0]; *j_end = e[1];
  return rc;
}

// Score, start cell and end cell.  Pass 1: end cell (tracking kernel).  Pass 2: the anchored recurrence over the
// reversed prefixes seq1[0..j_end), seq2[0..i_end): its maximum equals the score and sits at the start cell.
static int score_span_locked(swb200_ctx* c, const uint8_t* d_seq1, long long n, const uint8_t* d_seq2, long long m,
                             const swb200_params* p, cudaStream_t s, int* score_out, long long* span4) {
  span4[0] = span4[1] = span4[2] = span4[3] = 0;
  long long e[2] = {0, 0};
  int rc = score_device_locked(c, d_seq1, n, d_seq2, m, p, nullptr, s, score_out, e);
  if (rc || *score_out <= 0) return rc;
  const long long ie = e[0], je = e[1];
  const size_t off2 = ((size_t)je + 255) & ~(size_t)255;
  if ((rc = grow(c->d_rev, c->rev_cap, off2 + (size_t)ie + 256, false, s))) return rc;
  const int b1 = (int)std::min<long long>((je + 255) / 256, 8LL * c->sms), b2 = (int)std::min<long long>((ie + 255) / 256, 8LL * c->sms);
  reverse_bytes_kernel<<<b1, 256, 0, s>>>(d_seq1, je, c->d_rev);
  reverse_bytes_kernel<<<b2, 256, 0, s>>>(d_seq2, ie, c->d_rev + off2);
  SWB_CUDA(cudaGetLastError());
  const swb200_run_info first = c->info;
  int score2 = 0;
  long long r[2] = {0, 0};
  if ((rc = score_device_locked(c, c->d_rev, je, c->d_rev + off2, ie, p, nullptr, s, &score2, r, /*anchored=*/true))) return rc;
  if (score2 != *score_out) return fail(SWB200_ERR_CUDA, "internal: anchored pass does not reproduce the score");
  c->info.engine_launches += first.engine_launches; c->info.aux_launches += first.aux_launches + 2;
  c->info.engine_ms += first.engine_ms; c->info.cells += first.cells;
  span4[0] = ie - r[0] + 1; span4[1] = je - r[1] + 1; span4[2] = ie; span4[3] = je;
  return SWB200_OK;
}

int swb200_score_span_device(swb200_ctx* c, const unsigned char* d_seq1, long long n, const unsigned char* d_seq2,
                             long long m, const swb200_params* p, void* stream, int* score_out, long long span_out[4]) {
  if (!c || !span_out || !score_out) return fail(SWB200_ERR_ARG, "null context or output");
  std::lock_guard<std::mutex> lk(c->mu);
  return score_span_locked(c, d_seq1, n, d_seq2, m, p, (cudaStream_t)stream, score_out, span_out);
}

int swb200_score_span(const unsigned char* seq1, long long n, const unsigned char* seq2, long long m,
                      const swb200_params* p, int* score_out, long long span_out[4]) {
  if (n < 0 || m < 0 || !score_out || !span_out || (n > 0 && !seq1) || (m > 0 && !seq2))
    return fail(SWB200_ERR_ARG, "bad sequence arguments");
  span_out[0] = span_out[1] = span_out[2] = span_out[3] = 0;
  if (n == 0 || m == 0) {
    if (p) { int rc = check_params(*p); if (rc) return rc; }
    *score_out = 0;
    return SWB200_OK;
  }
  swb200_ctx* c = nullptr;
  int rc = default_ctx(&c);
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = c->own_stream;
  const size_t off2 = ((size_t)n + 255) & ~(size_t)255;
  if ((rc = grow(c->d_ascii, c->ascii_cap, off2 + (size_t)m + 256, false, s))) return rc;
  SWB_CUDA(cudaMemcpyAsync(c->d_ascii, seq1, (size_t)n, cudaMemcpyHostToDevice, s));
  SWB_CUDA(cudaMemcpyAsync(c->d_ascii + off2, seq2, (size_t)m, cudaMemcpyHostToDevice, s));
  return score_span_locked(c, c->d_ascii, n, c->d_ascii + off2, m, p, s, score_out, span_out);
}

// Score, span and the alignment itself.  Pass 1 + 2: swb200_score_span (end cell, start cell).  Pass 3: the anchored
// recurrence over the span rectangle with direction recording (modes 10/11), whose maximum must be the score again; then
// the walk.  When the directions of the whole rectangle do not fit in device memory (or "align_block_rows" asks for it),
// pass 3 runs in blocks of rows (swb_traceback.cuh): a forward sweep that keeps one checkpoint row per block, then the
// walk, block by block from the bottom, each block but the last recomputed from its checkpoint over the columns left
// of the walk.  The operations are those of the one-block walk.  The CIGAR is checked by re-scoring it with the costs of
// main.cpp:28-33,57-58 before it is returned.
static int align_locked(swb200_ctx* c, const uint8_t* d_seq1, long long n, const uint8_t* d_seq2, long long m,
                        const swb200_params* pp, cudaStream_t s, int* score_out, long long* span4, std::string* cigar) {
  cigar->clear();
  const long long block_rows = settings().align_block_rows;
  if (block_rows < 0 || block_rows % swb::kDirBandRows)
    return fail(SWB200_ERR_ARG, "align_block_rows must be 0 or a positive multiple of 256");
  int rc = score_span_locked(c, d_seq1, n, d_seq2, m, pp, s, score_out, span4);
  if (rc || *score_out <= 0) return rc;
  const swb200_params p = params_or_default(pp);
  const long long is = span4[0], js = span4[1], ie = span4[2], je = span4[3];
  const long long rows = ie - is + 1, cols = je - js + 1;
  const swb200_run_info before = c->info;
  // pass 3 geometry (make_plan for modes 10/11: launch config 1, 8 rows per lane): seq2's span striped in 256-row
  // bands, seq1's span streamed over nsteps steps
  const int skew = swb::config_skew(1, 10);
  const long long NB = (rows + swb::kDirBandRows - 1) / swb::kDirBandRows;
  const long long nsteps = ((cols + skew + swb::kChunk - 1) / swb::kChunk) * swb::kChunk;
  const long long ext_len = 1LL << std::max(4, log2_ceil(nsteps + swb::kChunk));   // run_once's boundary stream length
  const size_t band_bytes = (size_t)nsteps * 32 * sizeof(uint32_t);
  long long kb = block_rows / swb::kDirBandRows;                   // bands per block; 0: the whole span in one launch
  if (kb == 0) {
    size_t free_b = 0, total_b = 0;
    {
      DeviceGuard guard;
      SWB_CUDA(cudaSetDevice(c->device));
      SWB_CUDA(cudaMemGetInfo(&free_b, &total_b));
    }
    // today's rule for the whole rectangle (run_once); otherwise the tallest block whose directions, with the
    // checkpoints, fit (grow() allocates a quarter more than it is asked for), at most one band per launched warp
    const double have = (double)free_b + (double)c->dirs_cap * 4 + (double)c->ckpt_cap * 8 - (double)(1ull << 30);
    if ((size_t)NB * band_bytes / 4 > c->dirs_cap && (double)NB * band_bytes + (double)(1ull << 30) > (double)free_b + (double)c->dirs_cap * 4) {
      for (long long k = std::min<long long>(NB - 1, 4LL * c->sms); k >= 1 && kb == 0; --k) {
        const long long B = (NB + k - 1) / k;
        const double need = 1.25 * ((double)k * band_bytes + (double)(B - 1) * 2 * ext_len * sizeof(uint2));
        if (need <= have) kb = k;
      }
      if (kb == 0)
        return fail(SWB200_ERR_NOMEM, "the traceback of this alignment does not fit in device memory even in blocks of 256 rows (" +
                                      std::to_string(band_bytes >> 20) + " MiB of directions per block)");
    }
  }
  const long long bands = kb > 0 ? kb : NB, B = (NB + bands - 1) / bands;   // bands per block, blocks
  const size_t cap = (size_t)(rows + cols + 4);
  if ((rc = grow(c->d_ops, c->ops_cap, cap + 8, false, s))) return rc;
  swb::WalkState* d_walk = reinterpret_cast<swb::WalkState*>(c->d_ops);
  unsigned long long* d_opsv = c->d_ops + 8;
  static_assert(sizeof(swb::WalkState) <= 8 * sizeof(unsigned long long), "the walk's state sits in front of its operations");
  swb200_run_info tot = before;
  auto add_info = [&](long long cells) {
    tot.engine_launches += c->info.engine_launches; tot.aux_launches += c->info.aux_launches;
    tot.engine_ms += c->info.engine_ms; tot.cells += cells;
  };
  int score3 = 0;
  swb::WalkState ws{};
  if (B > 1 && (rc = grow(c->d_ckpt, c->ckpt_cap, (size_t)(B - 1) * 2 * (size_t)ext_len, false, s))) return rc;
  DirBlock blk{};
  // one launch over the bands of block b and the columns [0, ncols); forward: keep its bottom row (all blocks but the last).
  // One block is today's whole-rectangle launch.
  auto block = [&](long long b, long long ncols, bool forward, int* best) -> int {
    blk.band0 = b * bands; blk.band1 = std::min(NB, (b + 1) * bands);
    blk.top = b > 0 ? c->d_ckpt + (size_t)(b - 1) * 2 * (size_t)ext_len : nullptr;
    blk.bottom = forward && b + 1 < B ? c->d_ckpt + (size_t)b * 2 * (size_t)ext_len : nullptr;
    int sc = 0;
    const int r = score_device_locked(c, d_seq1 + (js - 1), ncols, d_seq2 + (is - 1), rows, pp, nullptr, s, &sc, nullptr, true, true, &blk);
    if (r) return r;
    add_info((std::min(rows, blk.band1 * swb::kDirBandRows) - blk.band0 * swb::kDirBandRows) * ncols);
    *best = std::max(*best, sc);
    return SWB200_OK;
  };
  for (long long b = 0; b < B; ++b)                        // forward sweep, top to bottom
    if ((rc = block(b, cols, true, &score3))) return rc;
  if (score3 != *score_out) return fail(SWB200_ERR_CUDA, "internal: the traceback pass does not reproduce the score");
  // the walk starts in the last block, whose directions the forward sweep left in place
  for (long long b = B - 1; b >= 0; --b) {
    if (b < B - 1) {
      int unused = 0;
      if ((rc = block(b, ws.j, false, &unused))) return rc;
    }
    walk_traceback_kernel<<<1, 32, 0, s>>>(c->d_dirs, c->last_nsteps, c->last_skew_per_lane, blk.band0 * swb::kDirBandRows,
                                           b == B - 1, rows, cols, d_walk, d_opsv, (long long)cap);
    SWB_CUDA(cudaGetLastError());
    tot.aux_launches += 1;
    SWB_CUDA(cudaMemcpyAsync(&ws, d_walk, sizeof ws, cudaMemcpyDeviceToHost, s));
    SWB_CUDA(cudaStreamSynchronize(s));
    if (ws.done) break;
  }
  const long long nops = ws.nops;
  if (!ws.done || nops < 0 || (size_t)nops > cap) return fail(SWB200_ERR_CUDA, "internal: traceback walk overflowed its buffer");
  std::vector<unsigned long long> ops((size_t)nops);
  std::vector<uint8_t> a((size_t)cols), b((size_t)rows);
  if (nops) SWB_CUDA(cudaMemcpyAsync(ops.data(), d_opsv, (size_t)nops * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
  SWB_CUDA(cudaMemcpyAsync(a.data(), d_seq1 + (js - 1), (size_t)cols, cudaMemcpyDeviceToHost, s));
  SWB_CUDA(cudaMemcpyAsync(b.data(), d_seq2 + (is - 1), (size_t)rows, cudaMemcpyDeviceToHost, s));
  SWB_CUDA(cudaStreamSynchronize(s));
  // forward order, 'M' split into '=' / 'X', re-scored on the way
  long long i = 0, j = 0, total = 0;
  char last = 0; long long run = 0;
  auto put = [&](char op) {
    if (op == last) { ++run; return; }
    if (run) { *cigar += std::to_string(run); *cigar += last; }
    last = op; run = 1;
  };
  for (long long k = nops - 1; k >= 0; --k) {
    const char op = (char)(ops[(size_t)k] >> 56);
    const long long cnt = (long long)(ops[(size_t)k] & 0x00FFFFFFFFFFFFFFull);
    if (op == 'M') {
      for (long long t = 0; t < cnt; ++t, ++i, ++j) {
        if (i >= rows || j >= cols) return fail(SWB200_ERR_CUDA, "internal: traceback leaves the span");
        const bool eq = a[(size_t)j] == b[(size_t)i];
        total += eq ? p.match : p.mismatch;
        put(eq ? '=' : 'X');
      }
    } else if (op == 'I' || op == 'D') {
      total -= p.gap_init + (cnt - 1) * (long long)p.gap_ext;          // main.cpp:57-58: first gap character costs G_INIT
      for (long long t = 0; t < cnt; ++t) put(op);
      if (op == 'I') j += cnt; else i += cnt;
    } else return fail(SWB200_ERR_CUDA, "internal: unknown traceback operation");
  }
  put(0);
  if (i != rows || j != cols || total != *score_out)
    return fail(SWB200_ERR_CUDA, "internal: the alignment does not re-score to the score (" + std::to_string(total) + " vs " + std::to_string(*score_out) + ")");
  c->info.engine_launches = tot.engine_launches; c->info.aux_launches = tot.aux_launches;
  c->info.engine_ms = tot.engine_ms; c->info.cells = tot.cells;
  return SWB200_OK;
}

static int align_finish(const std::string& cigar, char* cigar_out, long long cigar_cap, long long* cigar_len_out) {
  if (cigar_len_out) *cigar_len_out = (long long)cigar.size();
  if (!cigar_out) return SWB200_OK;                          // length query
  if (cigar_cap < (long long)cigar.size() + 1) return fail(SWB200_ERR_ARG, "cigar buffer too small (see cigar_len_out)");
  memcpy(cigar_out, cigar.c_str(), cigar.size() + 1);
  return SWB200_OK;
}

int swb200_align_device(swb200_ctx* c, const unsigned char* d_seq1, long long n, const unsigned char* d_seq2, long long m,
                        const swb200_params* p, void* stream, int* score_out, long long span_out[4], char* cigar_out,
                        long long cigar_cap, long long* cigar_len_out) {
  if (!c || !span_out || !score_out) return fail(SWB200_ERR_ARG, "null context or output");
  std::lock_guard<std::mutex> lk(c->mu);
  std::string cigar;
  const int rc = align_locked(c, d_seq1, n, d_seq2, m, p, (cudaStream_t)stream, score_out, span_out, &cigar);
  if (rc) return rc;
  return align_finish(cigar, cigar_out, cigar_cap, cigar_len_out);
}

int swb200_align(const unsigned char* seq1, long long n, const unsigned char* seq2, long long m, const swb200_params* p,
                 int* score_out, long long span_out[4], char* cigar_out, long long cigar_cap, long long* cigar_len_out) {
  if (n < 0 || m < 0 || !score_out || !span_out || (n > 0 && !seq1) || (m > 0 && !seq2))
    return fail(SWB200_ERR_ARG, "bad sequence arguments");
  span_out[0] = span_out[1] = span_out[2] = span_out[3] = 0;
  if (cigar_len_out) *cigar_len_out = 0;
  if (cigar_out && cigar_cap > 0) cigar_out[0] = 0;
  if (n == 0 || m == 0) {
    if (p) { int rc = check_params(*p); if (rc) return rc; }
    *score_out = 0;
    return SWB200_OK;
  }
  swb200_ctx* c = nullptr;
  int rc = default_ctx(&c);
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = c->own_stream;
  const size_t off2 = ((size_t)n + 255) & ~(size_t)255;
  if ((rc = grow(c->d_ascii, c->ascii_cap, off2 + (size_t)m + 256, false, s))) return rc;
  SWB_CUDA(cudaMemcpyAsync(c->d_ascii, seq1, (size_t)n, cudaMemcpyHostToDevice, s));
  SWB_CUDA(cudaMemcpyAsync(c->d_ascii + off2, seq2, (size_t)m, cudaMemcpyHostToDevice, s));
  std::string cigar;
  if ((rc = align_locked(c, c->d_ascii, n, c->d_ascii + off2, m, p, s, score_out, span_out, &cigar))) return rc;
  return align_finish(cigar, cigar_out, cigar_cap, cigar_len_out);
}

int swb200_score(const unsigned char* seq1, int n, const unsigned char* seq2, int m, const swb200_params* p,
                 int* score_out) {
  return swb200_score_ex(seq1, n, seq2, m, p, nullptr, score_out);
}

int swb200_last_run(swb200_ctx* c, swb200_run_info* info) {
  if (!info) return fail(SWB200_ERR_ARG, "null info");
  if (!c) {
    if (pool_last_run(info)) return SWB200_OK;       // the last host-buffer call ran on the device pool
    int rc = default_ctx(&c);
    if (rc) return rc;
  }
  std::lock_guard<std::mutex> lk(c->mu);
  *info = c->info;
  return SWB200_OK;
}

// ---- batches of independent pairs --------------------------------------------------------------------
// Word strides of the resident 2-bit layout (32 symbols per 64-bit word) for sequences of up to max_q / max_t symbols: at
// least one word; +2 on the T side because the kernels prefetch one word past the end; +2 on the Q side of a batch kept
// in caller order (keep_order: the banded kernel streams both sequences).
struct Strides { long long q, t; };
static Strides batch_strides_for(int max_q, int max_t, bool keep_order) {
  return Strides{std::max(1, (max_q + 31) / 32) + (keep_order ? 2 : 0), std::max(1, (max_t + 31) / 32) + 2};
}
static bool fits_strides(int q, int t, const Strides& s, bool keep_order) {
  const Strides need = batch_strides_for(q, t, keep_order);
  return q >= 0 && t >= 0 && need.q <= s.q && need.t <= s.t;
}
// Word strides of the byte layout (8 bytes per 64-bit word, shorter sequence first): at least one word; the byte kernels
// read no word past a sequence's end.
static Strides byte_strides_for(int max_q, int max_t) {
  return Strides{std::max(1, (max_q + 7) / 8), std::max(1, (max_t + 7) / 8)};
}
// The packer of either layout: bytes = raw bytes (byte_strides_for, never keep_order), else 2-bit codes.
static void launch_pack(bool bytes, const uint8_t* seq1, const long long* off1, const int* len1, const uint8_t* seq2,
                        const long long* off2, const int* len2, long long npairs, const Strides& st, uint64_t* q_words,
                        uint64_t* t_words, int* q_len, int* t_len, int keep_order, int* status, int blocks, cudaStream_t s) {
  if (bytes)
    swb::launch_pack_bytes(seq1, off1, len1, seq2, off2, len2, npairs, st.q, st.t, q_words, t_words, q_len, t_len, blocks, s);
  else
    swb::launch_pack_batch(seq1, off1, len1, seq2, off2, len2, npairs, st.q, st.t, q_words, t_words, q_len, t_len, keep_order,
                           status, blocks, s);
}

static int batch_pack_device(swb200_ctx* c, const unsigned char* d_seq1, const long long* d_off1, const int* d_len1,
                             const unsigned char* d_seq2, const long long* d_off2, const int* d_len2, long long npairs,
                             int max_short, int max_long, long long total_cells, int keep_order, bool bytes, void* stream,
                             swb200_batch** out) {
  if (!c || !out || npairs < 0 || max_short < 0 || max_long < 0 || (!keep_order && max_long < max_short))
    return fail(SWB200_ERR_ARG, "bad batch arguments");
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  std::unique_ptr<swb200_batch, BatchDeleter> b(new swb200_batch());   // freed on every early return
  b->ctx = c; b->npairs = npairs; b->max_short = max_short; b->max_long = max_long; b->cells = total_cells;
  b->keep_order = keep_order ? 1 : 0;
  b->bytes = bytes ? 1 : 0;
  const Strides st = bytes ? byte_strides_for(max_short, max_long) : batch_strides_for(max_short, max_long, keep_order);
  b->q_stride = st.q; b->t_stride = st.t;
  const size_t np = (size_t)std::max<long long>(npairs, 1);
  SWB_CUDA(cudaMalloc(&b->q_words, np * b->q_stride * sizeof(uint64_t)));
  SWB_CUDA(cudaMalloc(&b->t_words, np * b->t_stride * sizeof(uint64_t)));
  SWB_CUDA(cudaMalloc(&b->q_len, np * sizeof(int)));
  SWB_CUDA(cudaMalloc(&b->t_len, np * sizeof(int)));
  if (!keep_order) SWB_CUDA(cudaMalloc(&b->len1, np * sizeof(int)));
  SWB_CUDA(cudaMemsetAsync(c->d_result, 0, 12 * sizeof(int), s));    // [0] score, [1] status, [3..8] timeout post-mortem, [11] protocol-checker mismatches
  if (npairs > 0) {
    const long long total = npairs * (b->q_stride + b->t_stride);
    const int blocks = (int)std::min<long long>((total + 255) / 256, 64LL * c->sms);
    launch_pack(bytes, d_seq1, d_off1, d_len1, d_seq2, d_off2, d_len2, npairs, st, b->q_words, b->t_words, b->q_len, b->t_len,
                b->keep_order, c->d_result, blocks, s);
    SWB_CUDA(cudaGetLastError());
    if (b->len1) SWB_CUDA(cudaMemcpyAsync(b->len1, d_len1, (size_t)npairs * sizeof(int), cudaMemcpyDeviceToDevice, s));
  }
  SWB_CUDA(cudaMemcpyAsync(c->h_result, c->d_result, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
  SWB_CUDA(cudaStreamSynchronize(s));
  if (c->h_result[1] & swb::STATUS_BAD_SYMBOL)
    return fail(SWB200_ERR_ALPHABET, "batch input contains bytes other than A,C,G,T");
  *out = b.release();
  return SWB200_OK;
}

int swb200_batch_pack_device(swb200_ctx* c, const unsigned char* d_seq1, const long long* d_off1, const int* d_len1,
                             const unsigned char* d_seq2, const long long* d_off2, const int* d_len2, long long npairs,
                             int max_short, int max_long, long long total_cells, int keep_order, void* stream,
                             swb200_batch** out) {
  return batch_pack_device(c, d_seq1, d_off1, d_len1, d_seq2, d_off2, d_len2, npairs, max_short, max_long, total_cells,
                           keep_order, false, stream, out);
}

int swb200_batch_pack_device_bytes(swb200_ctx* c, const unsigned char* d_seq1, const long long* d_off1, const int* d_len1,
                                   const unsigned char* d_seq2, const long long* d_off2, const int* d_len2, long long npairs,
                                   int max_short, int max_long, long long total_cells, void* stream, swb200_batch** out) {
  return batch_pack_device(c, d_seq1, d_off1, d_len1, d_seq2, d_off2, d_len2, npairs, max_short, max_long, total_cells, 0,
                           true, stream, out);
}

// A contiguous range of pairs of a packed batch (all pointers already offset to its first pair).
struct BatchView {
  const uint64_t* q_words; const uint64_t* t_words; const int* q_len; const int* t_len;
  long long q_stride, t_stride, npairs;
  int max_short, max_long;      // of the WHOLE batch: every range of one batch runs the same kernel
  bool bytes = false;           // the byte layout (byte_strides_for): only the byte kernels read it
};

// The calls that have no byte kernel refuse a byte batch.
static int refuse_bytes(const swb200_batch* b) {
  return b->bytes ? fail(SWB200_ERR_ARG, "batch was packed as bytes; only swb200_batch_score and swb200_batch_align take it")
                  : SWB200_OK;
}

static int check_batch_score(const swb200_params& p, int keep_order, int max_short) {
  if (keep_order) return fail(SWB200_ERR_ARG, "batch was packed in caller order (banded); re-pack with keep_order=0");
  if (max_short > 1024)
    return fail(SWB200_ERR_ARG, "batch kernel needs min(len1,len2) <= 1024 per pair; use swb200_score for long pairs");
  if ((long long)p.match * max_short > 32767 - p.match - 1)
    return fail(SWB200_ERR_RANGE, "match * min(len) does not fit the 16-bit lanes of the batch kernel");
  return SWB200_OK;
}

// Launches the batch kernel for one range; no synchronisation, no events.
static int launch_batch_score(swb200_ctx* c, const BatchView& v, const swb200_params& p, const swb200_options& o,
                              cudaStream_t s, int* d_scores, swb200_run_info* info) {
  if (v.npairs == 0) return SWB200_OK;
  int G = 8, per = 16;
  if (v.max_short > 16 * 16) { G = 16; per = 32; }
  if (v.max_short > 32 * 16) { G = 32; per = 64; }
  int R = 16;
  for (int k = swb::kNumBatchRowChoices - 1; k >= 0; --k)
    if (swb::kBatchRowChoices[k] * per >= v.max_short) R = swb::kBatchRowChoices[k];
  if (o.rows) R = o.rows;
  if (R * per < v.max_short) return fail(SWB200_ERR_ARG, "rows too small for the longest short sequence");
  const int mode = (p.gap_init == p.gap_ext && !o.no_linear) ? 1 : 0;
  const void* kern = swb::batch_kernel(R, mode, G);
  if (!kern) return fail(SWB200_ERR_ARG, "no batch kernel for rows=" + std::to_string(R));
  swb::BatchParams P{};
  P.q_words = v.q_words; P.t_words = v.t_words; P.q_len = v.q_len; P.t_len = v.t_len;
  P.q_stride = v.q_stride; P.t_stride = v.t_stride; P.npairs = v.npairs; P.scores = d_scores;
  P.match = p.match; P.mismatch = p.mismatch; P.gap_init = p.gap_init; P.gap_ext = p.gap_ext;
  int per_sm = 0;
  SWB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, 0));
  per_sm = std::max(per_sm, 1);
  const long long groups = (v.npairs + (32 / G) - 1) / (32 / G);
  const long long ctas = std::max<long long>(1, std::min<long long>((groups + 7) / 8, (long long)c->sms * per_sm));
  void* args[] = {&P};
  SWB_CUDA(cudaLaunchKernel(kern, dim3((unsigned)ctas), dim3(256), args, 0, s));
  info->lanes = 16; info->linear = mode == 1; info->rows = R; info->config = 100 + G; info->ctas = (int)ctas;
  info->warps = (int)ctas * 8; info->bands = 0; info->engine_launches += 1;
  return SWB200_OK;
}

// The byte score kernel (swb_bytes_batch.cu): one thread per pair, as many threads as are resident at once.
static long long bytes_score_threads(swb200_ctx* c) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, swb::bytes_score_kernel_ptr(), 256, 0) != cudaSuccess || per_sm < 1)
    per_sm = 1;
  return 256LL * c->sms * per_sm;
}

// Launches the byte score kernel for one range of a byte batch; no synchronisation, no events.  The column buffer is
// ab_col, shared by the ranges of one call (they run one after another on stream s).
static int launch_bytes_score(swb200_ctx* c, const BatchView& v, const swb200_params& p, cudaStream_t s, int* d_scores,
                              swb200_run_info* info) {
  if (v.npairs == 0) return SWB200_OK;
  const long long blocks = std::max(1LL, std::min<long long>((v.npairs + 255) / 256, bytes_score_threads(c) / 256));
  const long long nt = blocks * 256;
  if (int rc = grow(c->ab_col, c->ab_col_cap, (size_t)(v.max_short + 1) * nt, false, s)) return rc;
  swb::AlignBatchParams P{};
  P.q_words = v.q_words; P.t_words = v.t_words; P.q_len = v.q_len; P.t_len = v.t_len;
  P.q_stride = v.q_stride; P.t_stride = v.t_stride; P.npairs = v.npairs;
  P.match = p.match; P.mismatch = p.mismatch; P.gap_init = p.gap_init; P.gap_ext = p.gap_ext;
  P.scores = d_scores; P.col = c->ab_col; P.nthreads = nt;
  swb::launch_bytes_score(P, (int)blocks, s);
  SWB_CUDA(cudaGetLastError());
  info->lanes = 32; info->linear = 0; info->rows = swb::kAlignStrip; info->config = 101; info->ctas = (int)blocks;
  info->warps = (int)blocks * 8; info->bands = 0; info->engine_launches += 1;
  return SWB200_OK;
}

// The multi-band batch kernel (swb_batch.cuh, LONG): one pair per warp, Q cut into bands of 64*R rows, so the shorter
// side has no cap beyond the 16-bit range.
static int check_long_score(const swb200_params& p, const swb200_options& o, int keep_order, int max_short) {
  if (keep_order) return fail(SWB200_ERR_ARG, "batch was packed in caller order (banded); re-pack with keep_order=0");
  bool known = o.rows == 0;
  for (int k = 0; k < swb::kNumBatchRowChoices; ++k) known |= o.rows == swb::kBatchRowChoices[k];
  if (!known) return fail(SWB200_ERR_ARG, "rows must be 0 or one of 2,4,6,8,10,12,16");
  if ((long long)p.match * max_short > 32767 - p.match - 1)
    return fail(SWB200_ERR_RANGE, "match * min(len) does not fit the 16-bit lanes of the batch kernel");
  return SWB200_OK;
}

// R of the multi-band kernel: options.rows, else the smallest choice whose band of 64*R rows holds the tallest pair, else 16
static int long_rows(const swb200_options& o, int max_short) {
  if (o.rows) return o.rows;
  for (int k = 0; k < swb::kNumBatchRowChoices; ++k)
    if (64 * swb::kBatchRowChoices[k] >= max_short) return swb::kBatchRowChoices[k];
  return 16;
}

// warps of the multi-band kernel resident at once (one pair each): a host chunk is a whole number of them
static long long long_wave_pairs(swb200_ctx* c, const swb200_params& p, const swb200_options& o, int max_short) {
  const int mode = (p.gap_init == p.gap_ext && !o.no_linear) ? 1 : 0;
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, swb::long_batch_kernel(long_rows(o, max_short), mode), 256, 0) !=
          cudaSuccess || per_sm < 1) per_sm = 1;
  return 8LL * c->sms * per_sm;
}

static int launch_long_score(swb200_ctx* c, const BatchView& v, const swb200_params& p, const swb200_options& o,
                             cudaStream_t s, int* d_scores, swb200_run_info* info) {
  if (v.npairs == 0) return SWB200_OK;
  const int R = long_rows(o, v.max_short);
  const int mode = (p.gap_init == p.gap_ext && !o.no_linear) ? 1 : 0;
  const void* kern = swb::long_batch_kernel(R, mode);
  if (!kern) return fail(SWB200_ERR_ARG, "no batch kernel for rows=" + std::to_string(R));
  swb::BatchParams P{};
  P.q_words = v.q_words; P.t_words = v.t_words; P.q_len = v.q_len; P.t_len = v.t_len;
  P.q_stride = v.q_stride; P.t_stride = v.t_stride; P.npairs = v.npairs; P.scores = d_scores;
  P.match = p.match; P.mismatch = p.mismatch; P.gap_init = p.gap_init; P.gap_ext = p.gap_ext;
  int per_sm = 0;
  SWB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, 0));
  per_sm = std::max(per_sm, 1);
  const long long ctas = std::max<long long>(1, std::min<long long>((v.npairs + 7) / 8, (long long)c->sms * per_sm));
  // one boundary row of the longest T per launched warp, 128-byte lines
  long long stride = ((long long)std::max(v.max_long, 1) + 31) / 32 * 32;
  int rc;
  if ((rc = grow(c->lb_bnd, c->lb_bnd_cap, (size_t)(ctas * 8) * (size_t)stride, false, s)) ||
      (rc = grow(c->lb_next, c->lb_next_cap, 1, false, s))) return rc;
  SWB_CUDA(cudaMemsetAsync(c->lb_next, 0, sizeof(unsigned long long), s));
  uint32_t* bnd = c->lb_bnd;
  unsigned long long* next = c->lb_next;
  void* args[] = {&P, &bnd, &stride, &next};
  SWB_CUDA(cudaLaunchKernel(kern, dim3((unsigned)ctas), dim3(256), args, 0, s));
  const int band_rows = 64 * R;
  info->lanes = 16; info->linear = mode == 1; info->rows = R; info->config = 332; info->ctas = (int)ctas;
  info->warps = (int)ctas * 8; info->bands = std::max(1, (v.max_short + band_rows - 1) / band_rows);
  info->engine_launches += 1;
  return SWB200_OK;
}

// The band widths the banded kernels have: W = band_hi - band_lo + 1 in {64, 128, 256, 512}.  Every banded call checks
// here first.
static int check_band_width(int band_lo, int band_hi) {
  const long long w = (long long)band_hi - band_lo + 1;
  if (w != 64 && w != 128 && w != 256 && w != 512)
    return fail(SWB200_ERR_ARG, "the banded kernels handle bands of 64, 128, 256 or 512 diagonals");
  return SWB200_OK;
}

static int check_banded_score(const swb200_params& p, int keep_order, int band_lo, int band_hi, int max1, int max2) {
  if (!keep_order) return fail(SWB200_ERR_ARG, "banded scoring needs a batch packed with keep_order=1");
  if (int rc = check_band_width(band_lo, band_hi)) return rc;
  if ((long long)p.match * std::min(max1, max2) > 32767 - p.match - 1)
    return fail(SWB200_ERR_RANGE, "match * min(len) does not fit the 16-bit lanes of the banded kernel");
  return SWB200_OK;
}

// Kernel, threads per CTA, pairs per CTA and run-info config code of the banded layout for a band of band_w diagonals
// and the options.  64 diagonals: four layouts, 4 threads per pair with eight register sets each (the default), 8 threads
// with four (options.config = 8), 16 threads with two (16) and 2 threads with sixteen (2), the last three kept for
// comparison; 16 pairs per CTA in each.  128, 256, 512 diagonals: band_w / 16 threads per pair with eight register sets,
// two warps and 1024 / band_w pairs per CTA, config 2128 / 2256 / 2512 whatever options.config says.
struct BandedLayout {
  const void* kern;
  int threads, pairs_per_cta, config, mode;
};
static BandedLayout banded_layout(const swb200_params& p, const swb200_options& o, int band_w) {
  const int mode = (p.gap_init == p.gap_ext && !o.no_linear) ? 1 : 0;
  if (band_w != swb::kBandWidth) return BandedLayout{swb::banded_wide_kernel(mode, band_w), 64, 1024 / band_w, 2000 + band_w, mode};
  const bool wide = o.config == 16, mid = o.config == 8, two = o.config == 2;
  const void* kern = wide ? swb::banded_kernel(mode) : (mid ? swb::banded8_kernel(mode) : (two ? swb::banded2_kernel(mode) : swb::banded4_kernel(mode)));
  return BandedLayout{kern, wide ? 256 : (mid ? 128 : (two ? 32 : 64)), 16, wide ? 216 : (mid ? 208 : (two ? 202 : 204)), mode};
}

// pairs one full wave of resident CTAs scores
static long long banded_wave_pairs(swb200_ctx* c, const swb200_params& p, const swb200_options& o, int band_w) {
  const BandedLayout L = banded_layout(p, o, band_w);
  cudaFuncSetAttribute(L.kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, L.kern, L.threads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
  return (long long)L.pairs_per_cta * c->sms * per_sm;
}

static int launch_banded_score(swb200_ctx* c, const BatchView& v, int band_lo, int band_w, const swb200_params& p,
                               const swb200_options& o, cudaStream_t s, int* d_scores, swb200_run_info* info) {
  if (v.npairs == 0) return SWB200_OK;
  const BandedLayout L = banded_layout(p, o, band_w);
  const void* kern = L.kern;
  const int threads = L.threads, mode = L.mode, pairs_per_cta = L.pairs_per_cta;
  // several CTAs of 34-35 KB static shared memory per SM: ask for the large shared-memory carve-out
  cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  swb::BandedParams P{};
  P.a_words = v.q_words; P.b_words = v.t_words; P.a_len = v.q_len; P.b_len = v.t_len;
  P.a_stride = v.q_stride; P.b_stride = v.t_stride; P.npairs = v.npairs; P.band_lo = band_lo; P.scores = d_scores;
  P.match = p.match; P.mismatch = p.mismatch; P.gap_init = p.gap_init; P.gap_ext = p.gap_ext;
  int per_sm = 0;
  SWB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, 0));
  per_sm = std::max(per_sm, 1);
  const long long ctas = std::max<long long>(1, std::min<long long>((v.npairs + pairs_per_cta - 1) / pairs_per_cta, (long long)c->sms * per_sm));
  void* args[] = {&P};
  SWB_CUDA(cudaLaunchKernel(kern, dim3((unsigned)ctas), dim3((unsigned)threads), args, 0, s));
  info->lanes = 16; info->linear = mode == 1; info->rows = 0; info->config = L.config; info->ctas = (int)ctas;
  info->warps = (int)ctas * (threads / 32); info->bands = band_w; info->engine_launches += 1;
  return SWB200_OK;
}

static BatchView whole_batch(const swb200_batch* b) {
  return BatchView{b->q_words, b->t_words, b->q_len, b->t_len, b->q_stride, b->t_stride, b->npairs, b->max_short, b->max_long,
                   b->bytes != 0};
}

// The device-batch calls after their argument checks: b's context locked and its device current, the run info reset to
// `cells`, nothing more for an empty batch, else work(c, s) between the two timing events on the caller's stream.
static int run_device_batch(swb200_batch* b, long long cells, void* stream,
                            const std::function<int(swb200_ctx*, cudaStream_t)>& work) {
  swb200_ctx* c = b->ctx;
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  const cudaStream_t s = (cudaStream_t)stream;
  c->info = swb200_run_info{};
  c->info.cells = cells;
  if (b->npairs == 0) return SWB200_OK;
  SWB_CUDA(cudaEventRecord(c->ev0, s));
  int rc;
  if ((rc = work(c, s))) return rc;
  SWB_CUDA(cudaEventRecord(c->ev1, s));
  SWB_CUDA(cudaStreamSynchronize(s));
  float ms = 0;
  SWB_CUDA(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  c->info.engine_ms = ms;
  return SWB200_OK;
}

int swb200_batch_score(swb200_batch* b, const swb200_params* pp, const swb200_options* oo, void* stream,
                       int* d_scores) {
  if (!b || !d_scores) return fail(SWB200_ERR_ARG, "bad batch arguments");
  const swb200_params p = params_or_default(pp);
  const swb200_options o = options_or_default(oo);
  int rc;
  if ((rc = check_params(p)) || (rc = check_batch_score(p, b->keep_order, b->max_short))) return rc;
  return run_device_batch(b, b->cells, stream, [&](swb200_ctx* c, cudaStream_t s) {
    return b->bytes ? launch_bytes_score(c, whole_batch(b), p, s, d_scores, &c->info)
                    : launch_batch_score(c, whole_batch(b), p, o, s, d_scores, &c->info);
  });
}

int swb200_batch_score_long(swb200_batch* b, const swb200_params* pp, const swb200_options* oo, void* stream, int* d_scores) {
  if (!b || !d_scores) return fail(SWB200_ERR_ARG, "bad batch arguments");
  const swb200_params p = params_or_default(pp);
  const swb200_options o = options_or_default(oo);
  int rc;
  if ((rc = refuse_bytes(b)) || (rc = check_params(p)) || (rc = check_long_score(p, o, b->keep_order, b->max_short))) return rc;
  return run_device_batch(b, b->cells, stream, [&](swb200_ctx* c, cudaStream_t s) {
    return launch_long_score(c, whole_batch(b), p, o, s, d_scores, &c->info);
  });
}

int swb200_batch_score_banded(swb200_batch* b, int band_lo, int band_hi, const swb200_params* pp, const swb200_options* oo,
                              void* stream, int* d_scores) {
  if (!b || !d_scores) return fail(SWB200_ERR_ARG, "bad batch arguments");
  const swb200_params p = params_or_default(pp);
  const swb200_options o = options_or_default(oo);
  int rc;
  if ((rc = refuse_bytes(b)) || (rc = check_params(p)) ||
      (rc = check_banded_score(p, b->keep_order, band_lo, band_hi, b->max_short, b->max_long))) return rc;
  return run_device_batch(b, b->cells, stream, [&](swb200_ctx* c, cudaStream_t s) {
    return launch_banded_score(c, whole_batch(b), band_lo, band_hi - band_lo + 1, p, o, s, d_scores, &c->info);
  });
}

void swb200_batch_free(swb200_batch* b) {
  if (!b) return;
  DeviceGuard guard;
  cudaSetDevice(b->ctx->device);
  cudaFree(b->q_words); cudaFree(b->t_words); cudaFree(b->q_len); cudaFree(b->t_len); cudaFree(b->len1);
  delete b;
}

// An ASCII host batch, or a contiguous range of one: pointers at its first pair, offsets absolute.
struct HostPairs {
  const unsigned char* seq1; const long long* off1; const int* len1;
  const unsigned char* seq2; const long long* off2; const int* len2;
  HostPairs from(long long k0) const { return HostPairs{seq1, off1 + k0, len1 + k0, seq2, off2 + k0, len2 + k0}; }
};

// What the host calls learn from pairs [k0, k1) of an ASCII batch before they touch a device.
struct PairScan {
  long long neg = 0;                                            // sign bit set iff a length or an offset is negative
  int max1 = 0, max2 = 0, max_min = 0;                          // longest seq1, longest seq2, longest shorter sequence
  long long cells = 0;
  long long lo1 = LLONG_MAX, hi1 = 0, lo2 = LLONG_MAX, hi2 = 0;   // lowest offset and highest end on each side
  // the batch shape: a banded batch (keep_order) keeps seq1 / seq2 in place, the others put the shorter sequence first
  int max_short(bool keep_order) const { return keep_order ? max1 : max_min; }
  int max_long(bool keep_order) const { return keep_order ? max2 : std::max(max1, max2); }
  void merge(const PairScan& o) {
    neg |= o.neg; max1 = std::max(max1, o.max1); max2 = std::max(max2, o.max2); max_min = std::max(max_min, o.max_min);
    cells += o.cells;
    lo1 = std::min(lo1, o.lo1); hi1 = std::max(hi1, o.hi1); lo2 = std::min(lo2, o.lo2); hi2 = std::max(hi2, o.hi2);
  }
};

// Branch-free (this pass runs before the first copy can start: 1 ns per pair instead of 2-3).
static PairScan scan_pairs(const HostPairs& h, long long k0, long long k1) {
  long long neg = 0, cells = 0, lo1 = LLONG_MAX, hi1 = 0, lo2 = LLONG_MAX, hi2 = 0;
  int mx1 = 0, mx2 = 0, mxmin = 0;
  for (long long k = k0; k < k1; ++k) {
    const int a = h.len1[k], b = h.len2[k];
    const long long o1 = h.off1[k], o2 = h.off2[k];
    neg |= (long long)(a | b) | o1 | o2;
    hi1 = std::max(hi1, o1 + a);
    hi2 = std::max(hi2, o2 + b);
    lo1 = std::min(lo1, o1);
    lo2 = std::min(lo2, o2);
    mx1 = std::max(mx1, a); mx2 = std::max(mx2, b); mxmin = std::max(mxmin, std::min(a, b));
    cells += (long long)a * b;
  }
  return PairScan{neg, mx1, mx2, mxmin, cells, lo1, hi1, lo2, hi2};
}

// which kernel a host ASCII score batch runs (bytes: the byte layout and its score kernel, the limits of batch)
enum class ScoreKind { batch, banded, long_pairs, bytes };

static int check_score_pairs(const PairScan& s, const swb200_params& p, const swb200_options& o, ScoreKind kind, int band_lo,
                             int band_hi) {
  if (s.neg < 0) return fail(SWB200_ERR_ARG, "negative length or offset");
  int rc;
  if ((rc = check_params(p))) return rc;
  switch (kind) {
    case ScoreKind::banded: return check_banded_score(p, 1, band_lo, band_hi, s.max1, s.max2);
    case ScoreKind::long_pairs: return check_long_score(p, o, 0, s.max_min);
    default: return check_batch_score(p, 0, s.max_min);
  }
}

// chunk_events of the host pipelines, grow-only: one per chunk of a call
static int chunk_events_at_least(swb200_ctx* c, size_t n) {
  while (c->chunk_events.size() < n) {
    cudaEvent_t e;
    SWB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    c->chunk_events.push_back(e);
  }
  return SWB200_OK;
}

// Copy/pack pipeline of the ASCII host calls for one context's range h of npairs pairs (c locked, its device current;
// part: the range's scan, whole: the whole batch's).  The pairs are cut into chunks of ~48 MB of sequence; own_stream
// copies chunk k+1 from the host while aux_stream packs chunk k and runs each_chunk (if any) on it.  The staging pool is
// sized for the whole range, so chunks need no double buffering: every byte keeps its position relative to the range's
// lowest offset.  With pinned host buffers the call runs at PCIe speed.  ev0 is recorded at the first pack; *staged is
// the packed range.  wave > 0: every chunk but the last holds a whole multiple of wave pairs.  bytes: the byte layout.
static int stage_and_pack_locked(swb200_ctx* c, const HostPairs& h, long long npairs, const PairScan& part,
                                 const PairScan& whole, bool keep_order, bool bytes, BatchView* staged,
                                 const std::function<int(const BatchView& chunk, long long k0)>& each_chunk,
                                 long long wave = 0) {
  cudaStream_t sc = c->own_stream, sk = c->aux_stream;
  const size_t np = (size_t)npairs;
  const long long base1 = part.lo1 & ~15LL, base2 = part.lo2 & ~15LL;
  const int max_short = whole.max_short(keep_order), max_long = whole.max_long(keep_order);
  const Strides st = bytes ? byte_strides_for(max_short, max_long) : batch_strides_for(max_short, max_long, keep_order);
  int rc;
  if ((rc = grow(c->hb_seq1, c->hb_seq1_cap, (size_t)(part.hi1 - base1) + 16, false, sc)) ||
      (rc = grow(c->hb_seq2, c->hb_seq2_cap, (size_t)(part.hi2 - base2) + 16, false, sc)) ||
      (rc = grow(c->hb_off1, c->hb_off1_cap, np, false, sc)) || (rc = grow(c->hb_off2, c->hb_off2_cap, np, false, sc)) ||
      (rc = grow(c->hb_len1, c->hb_len1_cap, np, false, sc)) || (rc = grow(c->hb_len2, c->hb_len2_cap, np, false, sc)) ||
      (rc = grow(c->hb_scores, c->hb_scores_cap, np, false, sc)) ||
      (rc = grow(c->hb_qw, c->hb_qw_cap, np * st.q, false, sc)) || (rc = grow(c->hb_tw, c->hb_tw_cap, np * st.t, false, sc)) ||
      (rc = grow(c->hb_ql, c->hb_ql_cap, np, false, sc)) || (rc = grow(c->hb_tl, c->hb_tl_cap, np, false, sc))) return rc;
  *staged = BatchView{c->hb_qw, c->hb_tw, c->hb_ql, c->hb_tl, st.q, st.t, npairs, max_short, max_long, bytes};
  SWB_CUDA(cudaMemsetAsync(c->d_result, 0, 10 * sizeof(int), sc));
  SWB_CUDA(cudaMemcpyAsync(c->hb_off1, h.off1, np * sizeof(long long), cudaMemcpyHostToDevice, sc));
  SWB_CUDA(cudaMemcpyAsync(c->hb_off2, h.off2, np * sizeof(long long), cudaMemcpyHostToDevice, sc));
  SWB_CUDA(cudaMemcpyAsync(c->hb_len1, h.len1, np * sizeof(int), cudaMemcpyHostToDevice, sc));
  SWB_CUDA(cudaMemcpyAsync(c->hb_len2, h.len2, np * sizeof(int), cudaMemcpyHostToDevice, sc));
  size_t ci = 0;
  long long k0 = 0, acc = 0, lo1 = LLONG_MAX, hi1 = 0, lo2 = LLONG_MAX, hi2 = 0;
  auto issue = [&](long long k1) -> int {
    int r;
    if ((r = chunk_events_at_least(c, ci + 1))) return r;
    if (hi1 > lo1) SWB_CUDA(cudaMemcpyAsync(c->hb_seq1 + (lo1 - base1), h.seq1 + lo1, (size_t)(hi1 - lo1), cudaMemcpyHostToDevice, sc));
    if (hi2 > lo2) SWB_CUDA(cudaMemcpyAsync(c->hb_seq2 + (lo2 - base2), h.seq2 + lo2, (size_t)(hi2 - lo2), cudaMemcpyHostToDevice, sc));
    SWB_CUDA(cudaEventRecord(c->chunk_events[ci], sc));
    SWB_CUDA(cudaStreamWaitEvent(sk, c->chunk_events[ci], 0));
    if (ci++ == 0) SWB_CUDA(cudaEventRecord(c->ev0, sk));
    const long long nk = k1 - k0;
    const int blocks = (int)std::min<long long>((nk * (st.q + st.t) + 255) / 256, 64LL * c->sms);
    // the pack kernel adds the absolute offsets: hand it the staging pointers shifted back by the range's base
    launch_pack(bytes, c->hb_seq1 - base1, c->hb_off1 + k0, c->hb_len1 + k0, c->hb_seq2 - base2, c->hb_off2 + k0,
                c->hb_len2 + k0, nk, st, c->hb_qw + k0 * st.q, c->hb_tw + k0 * st.t, c->hb_ql + k0, c->hb_tl + k0,
                keep_order ? 1 : 0, c->d_result, blocks, sk);
    SWB_CUDA(cudaGetLastError());
    c->info.aux_launches += 1;
    if (!each_chunk) return SWB200_OK;
    return each_chunk(BatchView{c->hb_qw + k0 * st.q, c->hb_tw + k0 * st.t, c->hb_ql + k0, c->hb_tl + k0, st.q, st.t, nk,
                                max_short, max_long, bytes}, k0);
  };
  // a chunk is issued the moment the scan over the pairs has found its end, so the GPU works while the host is still
  // cutting the later chunks
  const long long forced = settings().batch_chunk_bytes;           // tests: force many small chunks
  const long long target = forced > 0 ? forced : 48LL << 20, min_pairs = forced > 0 ? 1 : 1024;
  for (long long k = 0; k < npairs; ++k) {
    lo1 = std::min(lo1, h.off1[k]); hi1 = std::max(hi1, h.off1[k] + h.len1[k]);
    lo2 = std::min(lo2, h.off2[k]); hi2 = std::max(hi2, h.off2[k] + h.len2[k]);
    acc += (long long)h.len1[k] + h.len2[k];
    const bool whole_waves = forced > 0 || wave <= 0 || (k + 1 - k0) % wave == 0;
    if (!((acc >= target && k + 1 - k0 >= min_pairs && whole_waves) || k + 1 == npairs)) continue;
    if ((rc = issue(k + 1))) { cudaStreamSynchronize(sc); cudaStreamSynchronize(sk); return rc; }
    k0 = k + 1; acc = 0; lo1 = LLONG_MAX; hi1 = 0; lo2 = LLONG_MAX; hi2 = 0;
  }
  return SWB200_OK;
}

// One context's share of a host ASCII score batch (arguments checked by the caller): every chunk is scored as soon as it
// is packed, while the next one is copied.
static int score_ascii_ctx(swb200_ctx* c, const HostPairs& h, long long npairs, const PairScan& part, const PairScan& whole,
                           const swb200_params& p, const swb200_options& o, ScoreKind kind, int band_lo, int band_w,
                           int* scores_out) {
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  cudaStream_t sc = c->own_stream, sk = c->aux_stream;
  c->info = swb200_run_info{};
  c->info.cells = part.cells;
  BatchView staged;
  // a multi-band launch runs as long as its longest pairs however few they are: its chunks are whole waves of warps; a
  // byte launch runs one pair per thread: its chunks are whole waves of resident threads
  const bool banded = kind == ScoreKind::banded, bytes = kind == ScoreKind::bytes;
  const long long wave = kind == ScoreKind::long_pairs ? long_wave_pairs(c, p, o, whole.max_min) : (bytes ? bytes_score_threads(c) : 0);
  int rc = stage_and_pack_locked(c, h, npairs, part, whole, banded, bytes, &staged, [&](const BatchView& v, long long k0) {
    switch (kind) {
      case ScoreKind::banded: return launch_banded_score(c, v, band_lo, band_w, p, o, sk, c->hb_scores + k0, &c->info);
      case ScoreKind::long_pairs: return launch_long_score(c, v, p, o, sk, c->hb_scores + k0, &c->info);
      case ScoreKind::bytes: return launch_bytes_score(c, v, p, sk, c->hb_scores + k0, &c->info);
      default: return launch_batch_score(c, v, p, o, sk, c->hb_scores + k0, &c->info);
    }
  }, wave);
  if (rc) return rc;
  SWB_CUDA(cudaEventRecord(c->ev1, sk));
  SWB_CUDA(cudaMemcpyAsync(scores_out, c->hb_scores, npairs * sizeof(int), cudaMemcpyDeviceToHost, sk));
  SWB_CUDA(cudaMemcpyAsync(c->h_result, c->d_result, 2 * sizeof(int), cudaMemcpyDeviceToHost, sk));
  SWB_CUDA(cudaStreamSynchronize(sk));
  SWB_CUDA(cudaStreamSynchronize(sc));
  float ms = 0;
  SWB_CUDA(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  c->info.engine_ms = ms;          // first pack to last kernel, copies of later chunks overlapped
  if (c->h_result[1] & swb::STATUS_BAD_SYMBOL) return fail(SWB200_ERR_ALPHABET, "batch input contains bytes other than A,C,G,T");
  return SWB200_OK;
}

int swb200_score_banded(const unsigned char* seq1, int n, const unsigned char* seq2, int m, int band_lo, int band_hi,
                        const swb200_params* p, int* score_out) {
  if (n < 0 || m < 0 || !score_out || (n > 0 && !seq1) || (m > 0 && !seq2)) return fail(SWB200_ERR_ARG, "bad sequence arguments");
  if (int rc = check_band_width(band_lo, band_hi)) return rc;
  *score_out = 0;
  if (n == 0 || m == 0) { if (p) { int rc = check_params(*p); if (rc) return rc; } return SWB200_OK; }
  const long long off = 0;
  const HostPairs in{seq1, &off, &n, seq2, &off, &m};
  const PairScan s = scan_pairs(in, 0, 1);
  const swb200_params pv = params_or_default(p);
  swb200_ctx* c = nullptr;
  int rc;
  if ((rc = check_score_pairs(s, pv, swb200_options{}, ScoreKind::banded, band_lo, band_hi)) || (rc = default_ctx(&c))) return rc;
  return score_ascii_ctx(c, in, 1, s, s, pv, swb200_options{}, ScoreKind::banded, band_lo, band_hi - band_lo + 1, score_out);
}

// ---- one pair over a ring of GPUs (one swb200_ring per GPU / per process) -------------------------
int swb200_ring_create(swb200_ctx* c, int rank, int world, long long max_stream_len, swb200_ring** ring_out,
                       unsigned char handle_out[64]) {
  if (!c || !ring_out || !handle_out || world < 1 || rank < 0 || rank >= world || max_stream_len < 1)
    return fail(SWB200_ERR_ARG, "bad ring arguments");
  *ring_out = nullptr;
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  std::unique_ptr<swb200_ring, RingDeleter> r(new swb200_ring());
  r->ctx = c; r->rank = rank; r->world = world;
  r->len = (size_t)1 << log2_ceil(max_stream_len + 4 * 96 + 2 * swb::kRebaseBlock);
  r->entries = 8 * r->len;
  SWB_CUDA(cudaMalloc(&r->inbound, r->entries * sizeof(uint2)));
  SWB_CUDA(cudaMemset(r->inbound, 0, r->entries * sizeof(uint2)));
  cudaIpcMemHandle_t h;
  SWB_CUDA(cudaIpcGetMemHandle(&h, r->inbound));
  static_assert(sizeof(h) == 64, "CUDA IPC handle size");
  memcpy(handle_out, &h, 64);
  if (world == 1) { r->next = r->inbound; r->root = r->inbound; }
  *ring_out = r.release();
  return SWB200_OK;
}

static int ring_open_ipc(swb200_ring* r, const unsigned char handle[64], uint2** out) {
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  void* p = nullptr;
  SWB_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  *out = reinterpret_cast<uint2*>(p);
  return SWB200_OK;
}

int swb200_ring_connect(swb200_ring* r, const unsigned char next_handle[64]) {
  if (!r || !next_handle) return fail(SWB200_ERR_ARG, "bad ring arguments");
  std::lock_guard<std::mutex> lk(r->ctx->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(r->ctx->device));
  if (r->world == 1) return SWB200_OK;
  int rc = ring_open_ipc(r, next_handle, &r->next);
  if (rc) return rc;
  r->next_is_ipc = true;
  return SWB200_OK;
}

int swb200_ring_connect_root(swb200_ring* r, const unsigned char root_handle[64]) {
  if (!r || !root_handle) return fail(SWB200_ERR_ARG, "bad ring arguments");
  std::lock_guard<std::mutex> lk(r->ctx->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(r->ctx->device));
  if (r->world == 1 || r->rank == 0) { r->root = r->inbound; return SWB200_OK; }
  if (r->rank == r->world - 1 && r->next) { r->root = r->next; return SWB200_OK; }   // already mapped: the next rank IS the root
  int rc = ring_open_ipc(r, root_handle, &r->root);
  if (rc) return rc;
  r->root_is_ipc = true;
  return SWB200_OK;
}

static int ring_enable_peer(swb200_ring* r, swb200_ring* other) {
  if (other->ctx->device == r->ctx->device) return SWB200_OK;
  SWB_CUDA(cudaSetDevice(r->ctx->device));
  int can = 0;
  SWB_CUDA(cudaDeviceCanAccessPeer(&can, r->ctx->device, other->ctx->device));
  if (!can) return fail(SWB200_ERR_CUDA, "no peer access between the ring's devices");
  cudaError_t e = cudaDeviceEnablePeerAccess(other->ctx->device, 0);
  if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
    return fail(SWB200_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
  cudaGetLastError();
  return SWB200_OK;
}

int swb200_ring_connect_local(swb200_ring* r, swb200_ring* next) {
  if (!r || !next) return fail(SWB200_ERR_ARG, "bad ring arguments");
  if (next->entries != r->entries) return fail(SWB200_ERR_ARG, "rings of different capacity");
  DeviceGuard guard;
  int rc = ring_enable_peer(r, next);
  if (rc) return rc;
  r->next = next->inbound;
  return SWB200_OK;
}

int swb200_ring_connect_root_local(swb200_ring* r, swb200_ring* root) {
  if (!r || !root) return fail(SWB200_ERR_ARG, "bad ring arguments");
  if (root->entries != r->entries || root->rank != 0) return fail(SWB200_ERR_ARG, "not the root ring of this ring");
  DeviceGuard guard;
  int rc = ring_enable_peer(r, root);
  if (rc) return rc;
  r->root = root->inbound;
  return SWB200_OK;
}

int swb200_ring_score_device(swb200_ring* r, const unsigned char* d_seq1, long long n, const unsigned char* d_seq2,
                             long long m, const swb200_params* pp, const swb200_options* oo, void* stream,
                             int* partial_score_out, int* status_out) {
  if (!r || !partial_score_out || !status_out) return fail(SWB200_ERR_ARG, "bad ring arguments");
  if (!r->next) return fail(SWB200_ERR_ARG, "ring is not connected");
  swb200_ctx* c = r->ctx;
  std::lock_guard<std::mutex> lk(c->mu);
  const swb200_params p = params_or_default(pp);
  swb200_options o = options_or_default(oo);
  int rc;
  if ((rc = check_params(p))) return rc;
  if (n < 1 || m < 1) return fail(SWB200_ERR_ARG, "ring scoring needs non-empty sequences");
  if (o.lanes != 16 && o.lanes != 32) return fail(SWB200_ERR_ARG, "ring scoring needs an explicit lane width (16 or 32)");
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  c->info = swb200_run_info{};
  c->info.cells = n * m;
  r->calls += 1;
  r->combine = RingCombine{};
  RingCfg cfg{r->rank, r->world, r->inbound, r->next, r->len, r->calls < 16384 ? r->calls : 0u, r->root, &r->combine};
  const int lanes = (o.lanes == 16 && o.rebase > 0) ? 17 : o.lanes;
  return run_once(c, d_seq1, n, d_seq2, m, p, o, lanes, nullptr, (cudaStream_t)stream, partial_score_out, status_out, &cfg);
}

int swb200_ring_combine_pending(swb200_ring* r) { return r && r->combine.pending ? 1 : 0; }

int swb200_ring_combine(swb200_ring* r, void* stream, int* crossing_score_out) {
  if (!r || !crossing_score_out) return fail(SWB200_ERR_ARG, "bad ring arguments");
  *crossing_score_out = 0;
  swb200_ctx* c = r->ctx;
  std::lock_guard<std::mutex> lk(c->mu);
  const RingCombine cb = r->combine;
  r->combine.pending = false;
  if (!cb.pending || r->rank != 0) return SWB200_OK;      // only the root holds the two middle rows
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  const uint2* ff = r->inbound + 4 * r->len;
  const uint2* fb = r->inbound + 6 * r->len;
  const uint2* bf = cb.rebased ? ff + (size_t)cb.ext_len + (size_t)((cb.NB0 - 1) & 3) * (size_t)(cb.ext_len / 4) : nullptr;
  const uint2* bb = cb.rebased ? fb + (size_t)cb.ext_len + (size_t)((cb.NB1 - 1) & 3) * (size_t)(cb.ext_len / 4) : nullptr;
  SWB_CUDA(cudaMemsetAsync(c->d_result + 28, 0, sizeof(int), s));
  combine_two_sided_kernel<<<2 * c->sms, 256, 0, s>>>(ff, fb, cb.LT, cb.skew, cb.linear, cb.gap_init, cb.gap_ext, bf, bb,
                                                      c->d_result + 28);
  SWB_CUDA(cudaGetLastError());
  SWB_CUDA(cudaMemcpyAsync(c->h_result + 28, c->d_result + 28, sizeof(int), cudaMemcpyDeviceToHost, s));
  SWB_CUDA(cudaStreamSynchronize(s));
  c->info.aux_launches += 1;
  *crossing_score_out = c->h_result[28];
  return SWB200_OK;
}

void swb200_ring_destroy(swb200_ring* r) {
  if (!r) return;
  DeviceGuard guard;
  cudaSetDevice(r->ctx->device);
  if (r->root_is_ipc && r->root) cudaIpcCloseMemHandle(r->root);
  if (r->next_is_ipc && r->next) cudaIpcCloseMemHandle(r->next);
  cudaFree(r->inbound);
  delete r;
}

}  // extern "C"

// ---- several GPUs driven from ONE host process (the reference's caller is a single-threaded C++ loop,
//      TestFileWithGPU.cpp:57-94): swb200_set_devices(G) makes the host-buffer entry points use G GPUs --
//      a long pair is spread over an in-process ring (one host thread per GPU for the duration of the call, peer
//      access instead of IPC handles), a batch is cut into G contiguous ranges of pairs, one copy/compute pipeline
//      per GPU, no communication.
namespace {

struct Pool {
  std::mutex mu;                       // one pool call at a time
  std::vector<swb200_ctx*> ctx;        // device g = ctx[g]
  std::vector<swb200_ring*> ring;
  long long ring_stream_len = 0;
  swb200_run_info info{};              // what the last pool call ran (swb200_last_run(NULL, ..))
  bool info_valid = false;
};
Pool g_pool;

// fn(g) on one host thread per device; the first failure wins and its message is carried over to the caller's thread
template <class F>
int pool_parallel(int n, F fn) {
  std::vector<int> rc((size_t)n, 0);
  std::vector<std::string> err((size_t)n);
  std::vector<std::thread> th;
  th.reserve((size_t)n);
  for (int g = 0; g < n; ++g)
    th.emplace_back([&rc, &err, &fn, g] {
      rc[(size_t)g] = fn(g);
      if (rc[(size_t)g]) err[(size_t)g] = g_err;
    });
  for (auto& t : th) t.join();
  for (int g = 0; g < n; ++g)
    if (rc[(size_t)g]) return fail(rc[(size_t)g], "device " + std::to_string(g) + ": " + err[(size_t)g]);
  return SWB200_OK;
}

void pool_clear_locked() {
  for (swb200_ring* r : g_pool.ring) swb200_ring_destroy(r);
  g_pool.ring.clear();
  g_pool.ring_stream_len = 0;
  for (swb200_ctx* c : g_pool.ctx) swb200_ctx_destroy(c);
  g_pool.ctx.clear();
  g_pool.info_valid = false;
}

int pool_rings_locked(long long stream_len) {
  const int G = (int)g_pool.ctx.size();
  if ((int)g_pool.ring.size() == G && g_pool.ring_stream_len >= stream_len) return SWB200_OK;
  for (swb200_ring* r : g_pool.ring) swb200_ring_destroy(r);
  g_pool.ring.clear();
  g_pool.ring_stream_len = 0;
  const long long want = std::max<long long>(stream_len, 1 << 16);
  int rc;
  for (int g = 0; g < G; ++g) {
    swb200_ring* r = nullptr;
    unsigned char handle[64];
    if ((rc = swb200_ring_create(g_pool.ctx[(size_t)g], g, G, want, &r, handle))) return rc;
    g_pool.ring.push_back(r);
  }
  for (int g = 0; g < G; ++g) {
    if ((rc = swb200_ring_connect_local(g_pool.ring[(size_t)g], g_pool.ring[(size_t)((g + 1) % G)]))) return rc;
    if ((rc = swb200_ring_connect_root_local(g_pool.ring[(size_t)g], g_pool.ring[0]))) return rc;
  }
  g_pool.ring_stream_len = want;
  return SWB200_OK;
}

// One long host pair over the pool's ring.  *handled = false: not a case for the ring (bytes other than A,C,G,T),
// the caller scores it on one GPU.
int pool_score_pair(const unsigned char* seq1, long long n, const unsigned char* seq2, long long m, const swb200_params* pp,
                    const swb200_options* oo, int* score_out, bool* handled) {
  *handled = true;
  const int G = (int)g_pool.ctx.size();
  const swb200_params p = params_or_default(pp);
  const swb200_options o = options_or_default(oo);
  int rc;
  if ((rc = check_params(p))) return rc;
  const bool stream_is_shorter = o.orient == 0;
  if ((rc = pool_rings_locked(stream_is_shorter ? std::min(n, m) : std::max(n, m)))) return rc;
  // every GPU gets both sequences (G uploads in parallel, one per PCIe link)
  const size_t off2 = ((size_t)n + 255) & ~(size_t)255;
  rc = pool_parallel(G, [&](int g) -> int {
    swb200_ctx* c = g_pool.ctx[(size_t)g];
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard guard;
    SWB_CUDA(cudaSetDevice(c->device));
    int r;
    if ((r = grow(c->d_ascii, c->ascii_cap, off2 + (size_t)m + 256, false, c->own_stream))) return r;
    SWB_CUDA(cudaMemcpyAsync(c->d_ascii, seq1, (size_t)n, cudaMemcpyHostToDevice, c->own_stream));
    SWB_CUDA(cudaMemcpyAsync(c->d_ascii + off2, seq2, (size_t)m, cudaMemcpyHostToDevice, c->own_stream));
    return SWB200_OK;
  });
  if (rc) return rc;
  // lane-width policy of swb200_score (score_device_locked), decided once for all ranks
  struct Attempt { int lanes, rebase; };
  std::vector<Attempt> attempts;
  const long long bound = (long long)p.match * std::min(n, m);
  const bool rb_ok = o.rebase >= 0 && rebase_is_safe(p, o.rows ? o.rows : 16);
  if (o.lanes == 32) attempts.push_back({32, -1});
  else if (o.lanes == 16) attempts.push_back({16, o.rebase});
  else {
    if (bound <= 8LL * 32767 && o.rebase <= 0) attempts.push_back({16, -1});
    if (rb_ok) attempts.push_back({16, 1});
    attempts.push_back({32, -1});
  }
  for (const Attempt& at : attempts) {
    std::vector<int> part((size_t)G, 0), status((size_t)G, 0);
    swb200_options oa = o;
    oa.lanes = at.lanes; oa.rebase = at.rebase;
    rc = pool_parallel(G, [&](int g) -> int {
      swb200_ctx* c = g_pool.ctx[(size_t)g];
      return swb200_ring_score_device(g_pool.ring[(size_t)g], c->d_ascii, n, c->d_ascii + off2, m, &p, &oa, c->own_stream,
                                      &part[(size_t)g], &status[(size_t)g]);
    });
    if (rc) return rc;
    int best = 0, st = 0;
    float ms = 0;
    for (int g = 0; g < G; ++g) {
      best = std::max(best, part[(size_t)g]);
      st |= status[(size_t)g];
      ms = std::max(ms, g_pool.ctx[(size_t)g]->info.engine_ms);
    }
    int crossing = 0;
    const bool two_sided = swb200_ring_combine_pending(g_pool.ring[0]) != 0;
    if ((rc = swb200_ring_combine(g_pool.ring[0], g_pool.ctx[0]->own_stream, &crossing))) return rc;
    for (int g = 1; g < G; ++g) g_pool.ring[(size_t)g]->combine.pending = false;
    best = std::max(best, crossing);
    if (st & swb::STATUS_SPIN_TIMEOUT) return fail(SWB200_ERR_TIMEOUT, "boundary hand-off between GPUs timed out");
    if (st & swb::STATUS_BAD_SYMBOL) { *handled = false; return SWB200_OK; }
    if (st & (swb::STATUS_S16_OVERFLOW | swb::STATUS_REBASE_RANGE)) {
      if (o.lanes == 16) return fail(SWB200_ERR_RANGE, "score leaves the 16-bit lane range");
      continue;
    }
    g_pool.info = g_pool.ctx[0]->info;
    g_pool.info.engine_ms = ms;          // max over the GPUs
    g_pool.info.two_sided = two_sided;
    g_pool.info.ctas *= G; g_pool.info.warps *= G;
    g_pool.info_valid = true;
    *score_out = best;
    return SWB200_OK;
  }
  return fail(SWB200_ERR_RANGE, "no lane width could score this pair");
}

// The host batch calls: the whole batch on one GPU, or contiguous ranges of pairs, one per device chosen with
// swb200_set_devices (SURVEY.md 8e: pair_id / ceil(P / G); no data-path communication).  scan(k0, k1) reads a range's
// host inputs, each range on its own host thread (a serial pass over 10 M pairs costs milliseconds before the first copy
// can start); check(whole) validates the merged scan before any device is touched; run(ctx, k0, k1, part, whole) is one
// context's share, given its range's scan and the whole batch's.
template <class ScanFn, class CheckFn, class RunFn>
int run_host_batch(long long npairs, ScanFn scan, CheckFn check, RunFn run) {
  using Scan = decltype(scan(0LL, 0LL));
  std::unique_lock<std::mutex> pl(g_pool.mu);
  g_pool.info_valid = false;
  int G = (int)g_pool.ctx.size();
  int rc;
  if (G < 2 || npairs < 2LL * G) {
    pl.unlock();
    const Scan whole = scan(0, npairs);
    swb200_ctx* c = nullptr;
    if ((rc = check(whole)) || (rc = default_ctx(&c))) return rc;
    return run(c, 0, npairs, whole, whole);
  }
  const long long per = (npairs + G - 1) / G;
  auto first = [&](int g) { return std::min<long long>(npairs, (long long)g * per); };
  std::vector<Scan> part((size_t)G);
  if ((rc = pool_parallel(G, [&](int g) { part[(size_t)g] = scan(first(g), first(g + 1)); return SWB200_OK; }))) return rc;
  Scan whole = part[0];
  for (int g = 1; g < G; ++g) whole.merge(part[(size_t)g]);
  if ((rc = check(whole))) return rc;
  if ((rc = pool_parallel(G, [&](int g) {
         return first(g) == first(g + 1) ? SWB200_OK : run(g_pool.ctx[(size_t)g], first(g), first(g + 1), part[(size_t)g], whole);
       }))) return rc;
  // what the call ran: cells and launches summed over the GPUs (a device left without pairs ran nothing), the longest
  // device time, everything else as device 0 ran it
  swb200_run_info& info = g_pool.info;
  info = g_pool.ctx[0]->info;
  info.cells = 0; info.engine_launches = 0; info.aux_launches = 0; info.engine_ms = 0;
  for (int g = 0; g < G && first(g) < npairs; ++g) {
    const swb200_run_info& gi = g_pool.ctx[(size_t)g]->info;
    info.cells += gi.cells; info.engine_launches += gi.engine_launches; info.aux_launches += gi.aux_launches;
    info.engine_ms = std::max(info.engine_ms, gi.engine_ms);
  }
  g_pool.info_valid = true;
  return SWB200_OK;
}

}  // namespace

static int score_pair_on_pool(const unsigned char* seq1, long long n, const unsigned char* seq2, long long m,
                              const swb200_params* p, const swb200_options* opt, int* score_out) {
  std::lock_guard<std::mutex> pl(g_pool.mu);
  g_pool.info_valid = false;
  if (g_pool.ctx.size() < 2) return 1;
  const long long min_cells = settings().ring_min_cells;
  if ((double)n * (double)m < (double)min_cells) return 1;
  bool handled = true;
  const int rc = pool_score_pair(seq1, n, seq2, m, p, opt, score_out, &handled);
  if (rc) return rc;
  return handled ? SWB200_OK : 1;
}

// swb200_score_batch / swb200_score_banded_batch / swb200_score_long_batch / swb200_score_batch_bytes
static int score_batch_host(const HostPairs& in, long long npairs, const swb200_params* pp, const swb200_options* oo,
                            ScoreKind kind, int band_lo, int band_hi, int* scores_out) {
  if (npairs < 0 || (npairs > 0 && (!in.seq1 || !in.seq2 || !in.off1 || !in.off2 || !in.len1 || !in.len2 || !scores_out)))
    return fail(SWB200_ERR_ARG, "bad batch arguments");
  if (npairs == 0) return SWB200_OK;
  const swb200_params p = params_or_default(pp);
  const swb200_options o = options_or_default(oo);
  return run_host_batch(
      npairs, [&](long long k0, long long k1) { return scan_pairs(in, k0, k1); },
      [&](const PairScan& whole) { return check_score_pairs(whole, p, o, kind, band_lo, band_hi); },
      [&](swb200_ctx* c, long long k0, long long k1, const PairScan& part, const PairScan& whole) {
        return score_ascii_ctx(c, in.from(k0), k1 - k0, part, whole, p, o, kind, band_lo, band_hi - band_lo + 1, scores_out + k0);
      });
}

// ---- host batches that are ALREADY in the resident 2-bit format: a quarter of the bytes over PCIe, no pack kernel ----
// One branch-free pass over the lengths of a packed host batch (a loop with early returns cost 1-2 ns per pair, 2-4 ms
// per million pairs BEFORE the first copy started): maxima, sum of cells, and whether any pair breaks the rules
// (a negative length; with `ordered`, a q longer than its t).
struct LenScan {
  int max_q = 0, max_t = 0; long long cells = 0; bool bad = false;
  void merge(const LenScan& o) { max_q = std::max(max_q, o.max_q); max_t = std::max(max_t, o.max_t); cells += o.cells; bad |= o.bad; }
};
static LenScan scan_lens(const int* q_len, const int* t_len, long long k0, long long k1, bool ordered) {
  LenScan r;
  int bad = 0;
  for (long long k = k0; k < k1; ++k) {
    const int q = q_len[k], t = t_len[k];
    bad |= (q | t) < 0;
    bad |= ordered & (t < q);
    r.max_q = q > r.max_q ? q : r.max_q;
    r.max_t = t > r.max_t ? t : r.max_t;
    r.cells += (long long)q * t;
  }
  r.bad = bad != 0;
  return r;
}

// One context's share of a packed host batch (arguments checked by the caller): chunks of 24 MB (banded: whole waves of
// ~48 MB) copied on own_stream while aux_stream scores the chunk before.
static int score_batch_packed_ctx(swb200_ctx* c, const unsigned long long* q_words, long long q_stride,
                                  const unsigned long long* t_words, long long t_stride, const int* q_len, const int* t_len,
                                  long long npairs, int max_short, int max_long, long long cells, const swb200_params& pv,
                                  const swb200_options& ov, int banded, int band_lo, int band_w, int* scores_out) {
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  cudaStream_t sc = c->own_stream, sk = c->aux_stream;
  const size_t np = (size_t)npairs;
  int rc;
  if ((rc = grow(c->hb_scores, c->hb_scores_cap, np, false, sc)) || (rc = grow(c->hb_qw, c->hb_qw_cap, np * q_stride, false, sc)) ||
      (rc = grow(c->hb_tw, c->hb_tw_cap, np * t_stride, false, sc)) || (rc = grow(c->hb_ql, c->hb_ql_cap, np, false, sc)) ||
      (rc = grow(c->hb_tl, c->hb_tl_cap, np, false, sc))) return rc;
  const long long forced = settings().batch_chunk_bytes;
  const long long target = forced > 0 ? forced : (banded ? 48LL << 20 : 24LL << 20);   // measured: bench/batch_e2e.py, bench/banded_e2e.py
  const long long per_pair = (q_stride + t_stride) * 8 + 8;
  long long chunk_pairs = std::max<long long>(forced > 0 ? 1 : 1024, target / per_pair);
  if (banded && forced <= 0) {
    // a banded kernel runs as long as its pairs are long however few they are: chunks are whole waves of resident CTAs
    // (10 kb reads: 14 208 pairs = 72 MB; 48 MB chunks left a third of every launch idle: 42.5 -> 30 ms for 250 000 pairs)
    const long long wave = banded_wave_pairs(c, pv, ov, band_w);
    chunk_pairs = wave * std::max<long long>(1, (target + wave * per_pair / 2) / (wave * per_pair));
  }
  const size_t nchunks = (size_t)((npairs + chunk_pairs - 1) / chunk_pairs);
  if ((rc = chunk_events_at_least(c, nchunks + 1))) return rc;
  c->info = swb200_run_info{};
  c->info.cells = cells;
  bool first = true;
  for (size_t ci = 0; ci < nchunks; ++ci) {
    const long long k0 = (long long)ci * chunk_pairs, nk = std::min(chunk_pairs, npairs - k0);
    SWB_CUDA(cudaMemcpyAsync(c->hb_qw + k0 * q_stride, q_words + k0 * q_stride, (size_t)(nk * q_stride) * 8, cudaMemcpyHostToDevice, sc));
    SWB_CUDA(cudaMemcpyAsync(c->hb_tw + k0 * t_stride, t_words + k0 * t_stride, (size_t)(nk * t_stride) * 8, cudaMemcpyHostToDevice, sc));
    SWB_CUDA(cudaMemcpyAsync(c->hb_ql + k0, q_len + k0, (size_t)nk * sizeof(int), cudaMemcpyHostToDevice, sc));
    SWB_CUDA(cudaMemcpyAsync(c->hb_tl + k0, t_len + k0, (size_t)nk * sizeof(int), cudaMemcpyHostToDevice, sc));
    SWB_CUDA(cudaEventRecord(c->chunk_events[ci], sc));
    SWB_CUDA(cudaStreamWaitEvent(sk, c->chunk_events[ci], 0));
    if (first) { SWB_CUDA(cudaEventRecord(c->ev0, sk)); first = false; }
    const BatchView v{c->hb_qw + k0 * q_stride, c->hb_tw + k0 * t_stride, c->hb_ql + k0, c->hb_tl + k0, q_stride, t_stride, nk, max_short, max_long};
    rc = banded ? launch_banded_score(c, v, band_lo, band_w, pv, ov, sk, c->hb_scores + k0, &c->info)
                : launch_batch_score(c, v, pv, ov, sk, c->hb_scores + k0, &c->info);
    if (rc) { cudaStreamSynchronize(sc); cudaStreamSynchronize(sk); return rc; }
  }
  SWB_CUDA(cudaEventRecord(c->ev1, sk));
  SWB_CUDA(cudaMemcpyAsync(scores_out, c->hb_scores, npairs * sizeof(int), cudaMemcpyDeviceToHost, sk));
  SWB_CUDA(cudaStreamSynchronize(sk));
  SWB_CUDA(cudaStreamSynchronize(sc));
  float ms = 0;
  SWB_CUDA(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  c->info.engine_ms = ms;
  return SWB200_OK;
}

// swb200_score_batch_packed / swb200_score_banded_batch_packed (banded: q = seq1 and t = seq2, in caller order)
static int score_packed_host(const unsigned long long* q_words, long long q_stride, const unsigned long long* t_words,
                             long long t_stride, const int* q_len, const int* t_len, long long npairs, int banded, int band_lo,
                             int band_hi, const swb200_params* pp, const swb200_options* oo, int* scores_out) {
  const Strides st{q_stride, t_stride}, least = batch_strides_for(0, 0, banded != 0);
  if (npairs < 0 || q_stride < least.q || t_stride < least.t ||
      (npairs > 0 && (!q_words || !t_words || !q_len || !t_len || !scores_out)))
    return fail(SWB200_ERR_ARG, "bad batch arguments");
  if (npairs == 0) return SWB200_OK;
  const swb200_params p = params_or_default(pp);
  const swb200_options o = options_or_default(oo);
  return run_host_batch(
      npairs, [&](long long k0, long long k1) { return scan_lens(q_len, t_len, k0, k1, !banded); },
      [&](const LenScan& whole) {
        if (whole.bad || !fits_strides(whole.max_q, whole.max_t, st, banded != 0))
          return fail(SWB200_ERR_ARG, banded ? "pair lengths do not fit the strides"
                                             : "pair lengths do not fit the strides (q must be the shorter sequence)");
        int rc;
        if ((rc = check_params(p))) return rc;
        return banded ? check_banded_score(p, 1, band_lo, band_hi, whole.max_q, whole.max_t) : check_batch_score(p, 0, whole.max_q);
      },
      [&](swb200_ctx* c, long long k0, long long k1, const LenScan& part, const LenScan& whole) {
        return score_batch_packed_ctx(c, q_words + k0 * q_stride, q_stride, t_words + k0 * t_stride, t_stride, q_len + k0,
                                      t_len + k0, k1 - k0, whole.max_q, whole.max_t, part.cells, p, o, banded, band_lo,
                                      band_hi - band_lo + 1, scores_out + k0);
      });
}

extern "C" {

int swb200_score_batch(const unsigned char* seq1_all, const long long* off1, const int* len1,
                       const unsigned char* seq2_all, const long long* off2, const int* len2, long long npairs,
                       const swb200_params* p, const swb200_options* opt, int* scores_out) {
  return score_batch_host(HostPairs{seq1_all, off1, len1, seq2_all, off2, len2}, npairs, p, opt, ScoreKind::batch, 0, 0,
                          scores_out);
}

int swb200_score_batch_bytes(const unsigned char* seq1_all, const long long* off1, const int* len1,
                             const unsigned char* seq2_all, const long long* off2, const int* len2, long long npairs,
                             const swb200_params* p, const swb200_options* opt, int* scores_out) {
  return score_batch_host(HostPairs{seq1_all, off1, len1, seq2_all, off2, len2}, npairs, p, opt, ScoreKind::bytes, 0, 0,
                          scores_out);
}

int swb200_score_long_batch(const unsigned char* seq1_all, const long long* off1, const int* len1,
                            const unsigned char* seq2_all, const long long* off2, const int* len2, long long npairs,
                            const swb200_params* p, const swb200_options* opt, int* scores_out) {
  return score_batch_host(HostPairs{seq1_all, off1, len1, seq2_all, off2, len2}, npairs, p, opt, ScoreKind::long_pairs, 0, 0,
                          scores_out);
}

int swb200_score_banded_batch(const unsigned char* seq1_all, const long long* off1, const int* len1,
                              const unsigned char* seq2_all, const long long* off2, const int* len2, long long npairs,
                              int band_lo, int band_hi, const swb200_params* p, const swb200_options* opt,
                              int* scores_out) {
  if (int rc = check_band_width(band_lo, band_hi)) return rc;
  return score_batch_host(HostPairs{seq1_all, off1, len1, seq2_all, off2, len2}, npairs, p, opt, ScoreKind::banded, band_lo,
                          band_hi, scores_out);
}

int swb200_batch_strides(int max_short, int max_long, long long* q_stride, long long* t_stride) {
  if (max_short < 0 || max_long < max_short || !q_stride || !t_stride) return fail(SWB200_ERR_ARG, "bad batch shape");
  const Strides st = batch_strides_for(max_short, max_long, false);
  *q_stride = st.q; *t_stride = st.t;
  return SWB200_OK;
}

// Format conversion on the host (no scoring here): raw A,C,G,T bytes -> the resident 2-bit layout, shorter sequence of
// each pair first.  Same words as the device packer (swb_batch.cu: pack_batch_kernel) produces.
// 2-bit code of a byte, 0xFF for anything but A,C,G,T (the codes of the device packer: (c >> 1) & 3)
struct PackLut {
  unsigned char v[256];
  PackLut() { memset(v, 0xFF, sizeof v); v['A'] = 0; v['C'] = 1; v['G'] = 3; v['T'] = 2; }
};
static const PackLut g_pack_lut;

// pairs [k0, k1): 0 = fine, 1 = a pair does not fit the strides, 2 = a byte other than A,C,G,T
static int pack_host_range(const unsigned char* seq1_all, const long long* off1, const int* len1, const unsigned char* seq2_all,
                           const long long* off2, const int* len2, long long k0, long long k1, long long q_stride, long long t_stride,
                           unsigned long long* q_words, unsigned long long* t_words, int* q_len, int* t_len, bool keep_order) {
  const unsigned char* const lut = g_pack_lut.v;
  unsigned bad = 0;
  for (long long k = k0; k < k1; ++k) {
    const bool swap = !keep_order && len1[k] > len2[k];
    const unsigned char* q = swap ? seq2_all + off2[k] : seq1_all + off1[k];
    const unsigned char* t = swap ? seq1_all + off1[k] : seq2_all + off2[k];
    const int lq = swap ? len2[k] : len1[k], lt = swap ? len1[k] : len2[k];
    if (!fits_strides(lq, lt, Strides{q_stride, t_stride}, keep_order)) return 1;
    for (int side = 0; side < 2; ++side) {
      const unsigned char* src = side ? t : q;
      const int len = side ? lt : lq;
      unsigned long long* dst = side ? t_words + k * t_stride : q_words + k * q_stride;
      const long long stride = side ? t_stride : q_stride;
      const long long full = len / 32;
      for (long long w = 0; w < full; ++w) {                       // whole words: 32 table look-ups, no bounds test
        const unsigned char* s32 = src + w * 32;
        unsigned long long out = 0;
#pragma unroll
        for (int b = 0; b < 32; ++b) {
          const unsigned v = lut[s32[b]];
          bad |= v;
          out |= (unsigned long long)(v & 3u) << (2 * b);
        }
        dst[w] = out;
      }
      for (long long w = full; w < stride; ++w) {
        unsigned long long out = 0;
        for (int b = 0; b < 32 && w * 32 + b < len; ++b) {
          const unsigned v = lut[src[w * 32 + b]];
          bad |= v;
          out |= (unsigned long long)(v & 3u) << (2 * b);
        }
        dst[w] = out;
      }
    }
    q_len[k] = lq; t_len[k] = lt;
  }
  return (bad & 0x80u) ? 2 : 0;
}

// Format conversion on the host, spread over up to 16 threads (5 GB of long reads are seconds of work for one).
static int pack_host_impl(const unsigned char* seq1_all, const long long* off1, const int* len1, const unsigned char* seq2_all,
                          const long long* off2, const int* len2, long long npairs, long long q_stride, long long t_stride,
                          unsigned long long* q_words, unsigned long long* t_words, int* q_len, int* t_len, bool keep_order) {
  if (npairs < 0 || (npairs > 0 && (!seq1_all || !seq2_all || !off1 || !off2 || !len1 || !len2 || !q_words || !t_words || !q_len || !t_len)))
    return fail(SWB200_ERR_ARG, "bad batch arguments");
  long long bytes = 0;
  for (long long k = 0; k < npairs; ++k) bytes += (long long)(len1[k] > 0 ? len1[k] : 0) + (len2[k] > 0 ? len2[k] : 0);
  const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  const int T = (int)std::max<long long>(1, std::min<long long>({16LL, (long long)hw, bytes >> 22, npairs}));   // >= 4 MB per thread
  std::vector<int> rc((size_t)T, 0);
  auto run = [&](int t) {
    const long long k0 = npairs * t / T, k1 = npairs * (t + 1) / T;
    rc[(size_t)t] = pack_host_range(seq1_all, off1, len1, seq2_all, off2, len2, k0, k1, q_stride, t_stride, q_words, t_words, q_len, t_len, keep_order);
  };
  if (T == 1) run(0);
  else {
    std::vector<std::thread> th;
    th.reserve((size_t)T);
    for (int t = 0; t < T; ++t) th.emplace_back(run, t);
    for (auto& x : th) x.join();
  }
  for (int t = 0; t < T; ++t) {
    if (rc[(size_t)t] == 1) return fail(SWB200_ERR_ARG, "pair longer than the strides allow");
    if (rc[(size_t)t] == 2) return fail(SWB200_ERR_ALPHABET, "batch input contains bytes other than A,C,G,T");
  }
  return SWB200_OK;
}

int swb200_pack_batch_host(const unsigned char* seq1_all, const long long* off1, const int* len1, const unsigned char* seq2_all,
                           const long long* off2, const int* len2, long long npairs, long long q_stride, long long t_stride,
                           unsigned long long* q_words, unsigned long long* t_words, int* q_len, int* t_len) {
  return pack_host_impl(seq1_all, off1, len1, seq2_all, off2, len2, npairs, q_stride, t_stride, q_words, t_words, q_len, t_len, false);
}

// ---- banded batches in the resident format: seq1 (columns) and seq2 (rows) keep their roles ----
int swb200_banded_strides(int max_len1, int max_len2, long long* stride1, long long* stride2) {
  if (max_len1 < 0 || max_len2 < 0 || !stride1 || !stride2) return fail(SWB200_ERR_ARG, "bad batch shape");
  const Strides st = batch_strides_for(max_len1, max_len2, true);
  *stride1 = st.q; *stride2 = st.t;
  return SWB200_OK;
}

int swb200_pack_banded_host(const unsigned char* seq1_all, const long long* off1, const int* len1, const unsigned char* seq2_all,
                            const long long* off2, const int* len2, long long npairs, long long stride1, long long stride2,
                            unsigned long long* words1, unsigned long long* words2) {
  if (npairs < 0) return fail(SWB200_ERR_ARG, "bad batch arguments");
  std::vector<int> l1((size_t)std::max<long long>(npairs, 1)), l2((size_t)std::max<long long>(npairs, 1));
  return pack_host_impl(seq1_all, off1, len1, seq2_all, off2, len2, npairs, stride1, stride2, words1, words2, l1.data(), l2.data(), true);
}

int swb200_score_banded_batch_packed(const unsigned long long* words1, long long stride1, const unsigned long long* words2,
                                     long long stride2, const int* len1, const int* len2, long long npairs, int band_lo,
                                     int band_hi, const swb200_params* p, const swb200_options* opt, int* scores_out) {
  return score_packed_host(words1, stride1, words2, stride2, len1, len2, npairs, 1, band_lo, band_hi, p, opt, scores_out);
}

int swb200_score_batch_packed(const unsigned long long* q_words, long long q_stride, const unsigned long long* t_words,
                              long long t_stride, const int* q_len, const int* t_len, long long npairs,
                              const swb200_params* p, const swb200_options* opt, int* scores_out) {
  return score_packed_host(q_words, q_stride, t_words, t_stride, q_len, t_len, npairs, 0, 0, 0, p, opt, scores_out);
}

}  // extern "C"

static bool pool_last_run(swb200_run_info* info) {
  std::lock_guard<std::mutex> pl(g_pool.mu);
  if (!g_pool.info_valid) return false;
  *info = g_pool.info;
  return true;
}

extern "C" {

int swb200_set_devices(int count) {
  std::lock_guard<std::mutex> pl(g_pool.mu);
  if (count < 0) return fail(SWB200_ERR_ARG, "negative device count");
  const int avail = swb200_device_count();
  if (count > 1 && count > avail)
    return fail(SWB200_ERR_ARG, "asked for " + std::to_string(count) + " devices, " + std::to_string(avail) + " present");
  pool_clear_locked();
  if (count <= 1) return SWB200_OK;
  for (int g = 0; g < count; ++g) {
    swb200_ctx* c = nullptr;
    const int rc = swb200_ctx_create(g, &c);
    if (rc) { const std::string msg = g_err; pool_clear_locked(); return fail(rc, msg); }
    g_pool.ctx.push_back(c);
  }
  return SWB200_OK;
}

int swb200_get_devices(void) {
  std::lock_guard<std::mutex> pl(g_pool.mu);
  return std::max<int>(1, (int)g_pool.ctx.size());
}

}  // extern "C"

// ---- batch alignment: score, span and CIGAR for every pair (swb_align_batch.cuh) ----------------------------------
namespace {

constexpr long long kAlignSlotWords = 2048;        // direction slot per thread: 2048 x 16 cells (a 150-base read's span: ~1 500)
constexpr long long kAlignPoolWords = 32LL << 20;  // shared pool for larger rectangles: 256 MB, or the largest rectangle if more

// The limits of swb200_score_batch, checked on the host before any device is touched.
int check_align_batch_limits(const swb200_params& p, int max_short) {
  if (max_short > 1024)
    return fail(SWB200_ERR_ARG, "batch alignment needs min(len1,len2) <= 1024 per pair; use swb200_align for long pairs");
  if ((long long)p.match * max_short > 32767 - p.match - 1)
    return fail(SWB200_ERR_RANGE, "match * min(len) is outside the batch limits; use swb200_align for such pairs");
  return SWB200_OK;
}

// The trace rounds of both batch alignments, after their first trace launch on stream s: one sync per round reads the
// error bits and the pending count; an error fails the call, nothing pending ends it; otherwise the pool gets room for
// pool_need 64-bit words and is emptied, and relaunch(todo, ntodo, pending) runs the pending pairs again.
int align_rounds_locked(swb200_ctx* c, cudaStream_t s, long long npairs, size_t pool_need, swb200_run_info* info,
                        const std::function<void(const int* todo, int ntodo, int* pending)>& relaunch) {
  int rc;
  for (int cur = 0;;) {
    unsigned long long h[3] = {0, 0, 0};
    SWB_CUDA(cudaMemcpyAsync(h, c->ab_misc, sizeof h, cudaMemcpyDeviceToHost, s));
    SWB_CUDA(cudaStreamSynchronize(s));
    const int err = (int)(uint32_t)h[0], npend = (int)(h[0] >> 32);
    if (err & swb::kAlignErrStart) return fail(SWB200_ERR_CUDA, "internal: anchored pass does not reproduce the score");
    if (err & swb::kAlignErrTrace) return fail(SWB200_ERR_CUDA, "internal: the traceback pass does not reproduce the score");
    if (err) return fail(SWB200_ERR_CUDA, "internal: the alignment does not re-score to the score");
    if (npend == 0) {
      info->cells += (long long)h[2];
      return SWB200_OK;
    }
    // the pool's first taker always fits (pool_need covers the largest rectangle)
    if ((rc = grow(c->ab_pool, c->ab_pool_cap, pool_need, false, s))) return rc;
    const int* todo = c->ab_list + (size_t)cur * npairs;
    cur ^= 1;
    SWB_CUDA(cudaMemsetAsync(c->ab_misc, 0, 2 * sizeof(unsigned long long), s));
    relaunch(todo, npend, c->ab_list + (size_t)cur * npairs);
    SWB_CUDA(cudaGetLastError());
    info->engine_launches += 1;
  }
}

// Passes 1-3 and the walk over a packed range (shorter sequence first, len1 = the caller's seq1 lengths), everything on
// stream s of c's device, with the kernels of the range's layout (v.bytes: swb_bytes_batch.cu).  Synchronises once per
// trace round (the pending count decides whether another round runs).
int align_packed_locked(swb200_ctx* c, const BatchView& v, const int* d_len1, const swb200_params& p, cudaStream_t s,
                        int* d_scores, int* d_spans, uint32_t* d_ops, int ops_stride, int* d_ops_count, swb200_run_info* info) {
  if (v.npairs == 0) return SWB200_OK;
  const long long blocks = std::max(1LL, std::min<long long>((v.npairs + 255) / 256, 2LL * c->sms));
  const long long nt = blocks * 256;
  int rc;
  if ((rc = grow(c->ab_col, c->ab_col_cap, (size_t)(v.max_short + 1) * nt, false, s)) ||
      (rc = grow(c->ab_slot, c->ab_slot_cap, (size_t)(kAlignSlotWords * nt), false, s)) ||
      (rc = grow(c->ab_list, c->ab_list_cap, 2 * (size_t)v.npairs, false, s)) ||
      (rc = grow(c->ab_misc, c->ab_misc_cap, 4, false, s))) return rc;
  SWB_CUDA(cudaMemsetAsync(c->ab_misc, 0, 3 * sizeof(unsigned long long), s));
  swb::AlignBatchParams P{};
  P.q_words = v.q_words; P.t_words = v.t_words; P.q_len = v.q_len; P.t_len = v.t_len; P.len1 = d_len1;
  P.q_stride = v.q_stride; P.t_stride = v.t_stride; P.npairs = v.npairs;
  P.match = p.match; P.mismatch = p.mismatch; P.gap_init = p.gap_init; P.gap_ext = p.gap_ext;
  P.scores = d_scores; P.spans = d_spans; P.col = c->ab_col; P.nthreads = nt;
  P.slot = c->ab_slot; P.slot_words = kAlignSlotWords; P.pool = c->ab_pool; P.pool_words = (long long)c->ab_pool_cap;
  P.pool_used = c->ab_misc + 1;
  P.todo = nullptr; P.ntodo = v.npairs;
  P.pending = c->ab_list; P.npending = reinterpret_cast<int*>(c->ab_misc) + 1;
  P.ops = d_ops; P.ops_stride = ops_stride; P.ops_count = d_ops_count;
  P.err = reinterpret_cast<int*>(c->ab_misc); P.cells = c->ab_misc + 2;
  const auto span = v.bytes ? swb::launch_bytes_span : swb::launch_align_span;
  const auto trace = v.bytes ? swb::launch_bytes_trace : swb::launch_align_trace;
  span(P, (int)blocks, s);
  trace(P, (int)blocks, s);
  SWB_CUDA(cudaGetLastError());
  info->engine_launches += 2;
  // rectangles larger than a slot: the pool, emptied for every round; its first taker always fits
  const size_t need = (size_t)std::max(kAlignPoolWords, swb::align_dir_words(v.max_long, v.max_short));
  if ((rc = align_rounds_locked(c, s, v.npairs, need, info, [&](const int* todo, int ntodo, int* pending) {
         P.pool = c->ab_pool; P.pool_words = (long long)c->ab_pool_cap;
         P.todo = todo; P.ntodo = ntodo; P.pending = pending;
         trace(P, (int)std::max(1LL, std::min<long long>(blocks, (ntodo + 255) / 256)), s);
       }))) return rc;
  info->lanes = 32; info->config = v.bytes ? 301 : 300; info->rows = swb::kAlignStrip;
  return SWB200_OK;
}

constexpr long long kBandSlotWords = 32LL * 3072;  // direction slot per warp and K: 384 KB, spans with len1 + len2 < 24 568 (cfg5: ~20 000)
constexpr int kBandCtasPerSm = 8;                  // 32 resident warps per SM: enough to hide the shuffle chain of a step

// Passes 1-3 and the walk over a packed range in caller order (q = seq1, t = seq2), everything on stream s of c's device:
// one warp per pair, the trace rounds of align_rounds_locked.  A band of band_w = 64 K diagonals stores K nibbles per
// lane and anti-diagonal, so the direction slot of a launched warp is K x kBandSlotWords: the same spans fit one slot at
// every width.  The slots of all warps take at most a fifth of the device memory free to this context (free memory plus
// the slots it already holds): if K x kBandSlotWords per warp would take more, fewer warps are launched (at least one
// CTA per SM).  On a 180 GB B200 occupancy allows 8 / 5 / 4 / 3 CTAs per SM at K = 1 / 2 / 4 / 8: 1.8 / 2.3 / 3.7 / 5.6 GB
// of slots, well inside the share.
int align_banded_packed_locked(swb200_ctx* c, const BatchView& v, int band_lo, int band_w, const swb200_params& p, cudaStream_t s,
                               int* d_scores, int* d_spans, uint32_t* d_ops, int ops_stride, int* d_ops_count,
                               swb200_run_info* info) {
  if (v.npairs == 0) return SWB200_OK;
  constexpr int W = swb::kBandAlignWarps;
  const int K = band_w / 64;
  const long long slot_words = kBandSlotWords * K;
  int per_sm = 0;
  SWB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, swb::align_banded_trace_kernel_ptr(K), 32 * W, 0));
  per_sm = std::max(1, std::min(per_sm, kBandCtasPerSm));
  if (K > 1) {
    size_t fr = 0, tot = 0;
    SWB_CUDA(cudaMemGetInfo(&fr, &tot));
    const double share = (double)(fr + c->ab_slot_cap * sizeof(uint64_t)) / 5;
    const long long fit = (long long)(share / ((double)slot_words * sizeof(uint32_t) * W * c->sms));   // CTAs per SM
    per_sm = std::max(1, std::min<int>(per_sm, (int)std::min<long long>(fit, kBandCtasPerSm)));
  }
  const long long blocks = std::max(1LL, std::min<long long>((v.npairs + W - 1) / W, (long long)c->sms * per_sm));
  const long long nw = blocks * W;
  int rc;
  if ((rc = grow(c->ab_slot, c->ab_slot_cap, (size_t)(slot_words * nw + 1) / 2, false, s)) ||
      (rc = grow(c->ab_list, c->ab_list_cap, 2 * (size_t)v.npairs, false, s)) ||
      (rc = grow(c->ab_misc, c->ab_misc_cap, 4, false, s))) return rc;
  SWB_CUDA(cudaMemsetAsync(c->ab_misc, 0, 3 * sizeof(unsigned long long), s));
  swb::AlignBandedParams P{};
  P.a_words = v.q_words; P.b_words = v.t_words; P.a_len = v.q_len; P.b_len = v.t_len;
  P.a_stride = v.q_stride; P.b_stride = v.t_stride; P.npairs = v.npairs; P.band_lo = band_lo;
  P.match = p.match; P.mismatch = p.mismatch; P.gap_init = p.gap_init; P.gap_ext = p.gap_ext;
  P.scores = d_scores; P.spans = d_spans; P.nwarps = nw;
  P.slot = reinterpret_cast<uint32_t*>(c->ab_slot); P.slot_words = slot_words;
  P.pool = reinterpret_cast<uint32_t*>(c->ab_pool); P.pool_words = 2 * (long long)c->ab_pool_cap;
  P.pool_used = c->ab_misc + 1;
  P.todo = nullptr; P.ntodo = v.npairs;
  P.pending = c->ab_list; P.npending = reinterpret_cast<int*>(c->ab_misc) + 1;
  P.ops = d_ops; P.ops_stride = ops_stride; P.ops_count = d_ops_count;
  P.err = reinterpret_cast<int*>(c->ab_misc); P.cells = c->ab_misc + 2;
  swb::launch_align_banded_span(P, K, (int)blocks, s);
  swb::launch_align_banded_trace(P, K, (int)blocks, s);
  SWB_CUDA(cudaGetLastError());
  info->engine_launches += 2;
  // spans larger than a slot: the pool (64-bit words here), sized for the largest span the batch can have
  const size_t need = (size_t)std::max(kAlignPoolWords, (K * swb::band_dir_words(v.max_short, v.max_long) + 1) / 2);
  if ((rc = align_rounds_locked(c, s, v.npairs, need, info, [&](const int* todo, int ntodo, int* pending) {
         P.pool = reinterpret_cast<uint32_t*>(c->ab_pool); P.pool_words = 2 * (long long)c->ab_pool_cap;
         P.todo = todo; P.ntodo = ntodo; P.pending = pending;
         swb::launch_align_banded_trace(P, K, (int)std::max(1LL, std::min<long long>(blocks, (ntodo + W - 1) / W)), s);
       }))) return rc;
  info->lanes = 32; info->config = K == 1 ? 310 : (K == 2 ? 311 : (K == 4 ? 312 : 313)); info->rows = 0; info->bands = band_w;
  info->ctas = (int)blocks; info->warps = (int)nw;
  return SWB200_OK;
}

constexpr int kLongTraceCtasPerSm = 4;    // 16 warps per SM trace (each owns a direction slot); the span kernel runs full

// Direction storage of the long-pair alignment, in 64-bit words: *slot per warp of the trace launch and *pool shared.
// A slot holds the largest span the batch can have (max_long x max_short), capped so that the slots of all nw warps take
// at most a fifth of the device memory free to this context (free memory plus the slots it already holds): with the
// quarter of headroom grow() adds, under a quarter.  The pool, used only when a span exceeds a slot, gets the same
// share, and at least the largest span (its first taker always fits).  On a 180 GB B200 with 2 368 trace warps: 5 kb
// pairs need 12.9 MB a span, 30.5 GB of slots in all, one trace round; 20 kb pairs need 202 MB a span, get 15 MB slots
// and share a ~35 GB pool, about 170 spans a round.
static int long_dir_budget(swb200_ctx* c, const BatchView& v, long long nw, long long* slot, size_t* pool) {
  size_t fr = 0, tot = 0;
  SWB_CUDA(cudaMemGetInfo(&fr, &tot));
  const long long share = (long long)((fr + c->ab_slot_cap * sizeof(uint64_t)) / 5 / sizeof(uint64_t));
  const long long largest = (swb::long_dir_words(v.max_long, v.max_short) + 1) / 2;
  *slot = std::max(1LL, std::min(largest, share / nw));
  *pool = (size_t)std::max(largest, std::max(kAlignPoolWords, share));
  return SWB200_OK;
}

// Passes 1-3 and the walk over a packed range (shorter sequence first, len1 = the caller's seq1 lengths) whose shorter
// side may exceed 1024, everything on stream s of c's device: one warp per pair, warps drawing pairs from a counter,
// the trace rounds of align_rounds_locked.
int align_long_packed_locked(swb200_ctx* c, const BatchView& v, const int* d_len1, const swb200_params& p, cudaStream_t s,
                             int* d_scores, int* d_spans, uint32_t* d_ops, int ops_stride, int* d_ops_count,
                             swb200_run_info* info) {
  if (v.npairs == 0) return SWB200_OK;
  constexpr int W = swb::kLongAlignWarps;
  int span_sm = 0, trace_sm = 0;
  SWB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&span_sm, swb::align_long_span_kernel_ptr(), 32 * W, 0));
  SWB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&trace_sm, swb::align_long_trace_kernel_ptr(), 32 * W, 0));
  const long long want = (v.npairs + W - 1) / W;
  const long long span_blocks = std::max(1LL, std::min<long long>(want, (long long)c->sms * std::max(1, span_sm)));
  const long long blocks = std::max(1LL, std::min<long long>(want, (long long)c->sms * std::max(1, std::min(trace_sm, kLongTraceCtasPerSm))));
  const long long nw = blocks * W;
  const long long row_stride = ((long long)std::max(v.max_long, 1) + 31) / 32 * 32;   // int2 entries, 128-byte lines
  long long slot_words = 0;
  size_t pool_need = 0;
  int rc;
  if ((rc = long_dir_budget(c, v, nw, &slot_words, &pool_need)) ||
      (rc = grow(c->lb_bnd, c->lb_bnd_cap, (size_t)(2 * row_stride * std::max(span_blocks, blocks) * W), false, s)) ||
      (rc = grow(c->ab_slot, c->ab_slot_cap, (size_t)(slot_words * nw), false, s)) ||
      (rc = grow(c->ab_list, c->ab_list_cap, 2 * (size_t)v.npairs, false, s)) ||
      (rc = grow(c->ab_misc, c->ab_misc_cap, 5, false, s))) return rc;
  // [0] err | npending << 32, [1] pool words used, [2] cells, [3] the span kernel's pair counter, [4] the trace kernel's
  SWB_CUDA(cudaMemsetAsync(c->ab_misc, 0, 5 * sizeof(unsigned long long), s));
  swb::AlignBatchParams P{};
  P.q_words = v.q_words; P.t_words = v.t_words; P.q_len = v.q_len; P.t_len = v.t_len; P.len1 = d_len1;
  P.q_stride = v.q_stride; P.t_stride = v.t_stride; P.npairs = v.npairs;
  P.match = p.match; P.mismatch = p.mismatch; P.gap_init = p.gap_init; P.gap_ext = p.gap_ext;
  P.scores = d_scores; P.spans = d_spans;
  P.col = reinterpret_cast<int2*>(c->lb_bnd); P.row_stride = row_stride; P.nthreads = nw * 32;
  P.slot = c->ab_slot; P.slot_words = slot_words; P.pool = c->ab_pool; P.pool_words = (long long)c->ab_pool_cap;
  P.pool_used = c->ab_misc + 1;
  P.todo = nullptr; P.ntodo = v.npairs;
  P.pending = c->ab_list; P.npending = reinterpret_cast<int*>(c->ab_misc) + 1;
  P.ops = d_ops; P.ops_stride = ops_stride; P.ops_count = d_ops_count;
  P.err = reinterpret_cast<int*>(c->ab_misc); P.cells = c->ab_misc + 2;
  P.next = c->ab_misc + 3;
  swb::launch_align_long_span(P, (int)span_blocks, s);
  P.next = c->ab_misc + 4;
  swb::launch_align_long_trace(P, (int)blocks, s);
  SWB_CUDA(cudaGetLastError());
  info->engine_launches += 2;
  // spans larger than a slot: the pool, emptied for every round (the relaunch restarts the trace kernel's counter; a
  // failed memset shows in align_rounds_locked's cudaGetLastError)
  if ((rc = align_rounds_locked(c, s, v.npairs, pool_need, info, [&](const int* todo, int ntodo, int* pending) {
         cudaMemsetAsync(c->ab_misc + 4, 0, sizeof(unsigned long long), s);
         P.pool = c->ab_pool; P.pool_words = (long long)c->ab_pool_cap;
         P.todo = todo; P.ntodo = ntodo; P.pending = pending;
         swb::launch_align_long_trace(P, (int)std::max(1LL, std::min<long long>(blocks, (ntodo + W - 1) / W)), s);
       }))) return rc;
  info->lanes = 32; info->config = 320; info->rows = swb::kLongLaneRows;
  info->bands = std::max(1, (v.max_short + swb::kLongBandRows - 1) / swb::kLongBandRows);
  info->ctas = (int)blocks; info->warps = (int)nw;
  return SWB200_OK;
}

}  // namespace

// which kernels a host batch alignment runs (bytes: the byte layout and kernels, the limits of batch)
enum class AlignKind { batch, banded, long_pairs, bytes };

// One context's share of a host batch alignment (arguments checked by the caller): the copy/pack pipeline of the score
// calls, then the passes over the whole range, then the outputs back.  banded: the pairs stay in caller order and the
// banded passes run with band band_lo .. band_lo + band_w - 1.
static int align_batch_host_ctx(swb200_ctx* c, const HostPairs& h, long long npairs, const PairScan& part, const PairScan& whole,
                                const swb200_params& p, AlignKind kind, int band_lo, int band_w, int* scores_out, int* spans_out,
                                unsigned int* ops_out, int ops_stride, int* ops_count) {
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard guard;
  SWB_CUDA(cudaSetDevice(c->device));
  cudaStream_t sc = c->own_stream, sk = c->aux_stream;
  const size_t np = (size_t)npairs;
  int rc;
  if ((rc = grow(c->hb_spans, c->hb_spans_cap, 4 * np, false, sc)) ||
      (rc = grow(c->hb_ops, c->hb_ops_cap, np * (size_t)ops_stride, false, sc)) || (rc = grow(c->hb_opsn, c->hb_opsn_cap, np, false, sc))) return rc;
  c->info = swb200_run_info{};
  BatchView v;
  if ((rc = stage_and_pack_locked(c, h, npairs, part, whole, kind == AlignKind::banded, kind == AlignKind::bytes, &v, nullptr)))
    return rc;
  SWB_CUDA(cudaMemcpyAsync(c->h_result, c->d_result, 2 * sizeof(int), cudaMemcpyDeviceToHost, sk));
  SWB_CUDA(cudaStreamSynchronize(sk));
  SWB_CUDA(cudaStreamSynchronize(sc));
  if (c->h_result[1] & swb::STATUS_BAD_SYMBOL) return fail(SWB200_ERR_ALPHABET, "batch input contains bytes other than A,C,G,T");
  SWB_CUDA(cudaMemsetAsync(c->hb_ops, 0, np * (size_t)ops_stride * sizeof(uint32_t), sk));   // overflowed pairs come back as zeros
  switch (kind) {
    case AlignKind::banded:
      rc = align_banded_packed_locked(c, v, band_lo, band_w, p, sk, c->hb_scores, c->hb_spans, c->hb_ops, ops_stride, c->hb_opsn,
                                      &c->info);
      break;
    case AlignKind::long_pairs:
      rc = align_long_packed_locked(c, v, c->hb_len1, p, sk, c->hb_scores, c->hb_spans, c->hb_ops, ops_stride, c->hb_opsn, &c->info);
      break;
    default:
      rc = align_packed_locked(c, v, c->hb_len1, p, sk, c->hb_scores, c->hb_spans, c->hb_ops, ops_stride, c->hb_opsn, &c->info);
  }
  if (rc) return rc;
  SWB_CUDA(cudaEventRecord(c->ev1, sk));
  SWB_CUDA(cudaMemcpyAsync(scores_out, c->hb_scores, np * sizeof(int), cudaMemcpyDeviceToHost, sk));
  SWB_CUDA(cudaMemcpyAsync(spans_out, c->hb_spans, 4 * np * sizeof(int), cudaMemcpyDeviceToHost, sk));
  SWB_CUDA(cudaMemcpyAsync(ops_count, c->hb_opsn, np * sizeof(int), cudaMemcpyDeviceToHost, sk));
  SWB_CUDA(cudaMemcpyAsync(ops_out, c->hb_ops, np * (size_t)ops_stride * sizeof(uint32_t), cudaMemcpyDeviceToHost, sk));
  SWB_CUDA(cudaStreamSynchronize(sk));
  float ms = 0;
  SWB_CUDA(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  c->info.engine_ms = ms;          // first pack to the last trace round
  return SWB200_OK;
}

// swb200_align_batch / swb200_align_batch_bytes
static int align_batch_host(const unsigned char* seq1_all, const long long* off1, const int* len1, const unsigned char* seq2_all,
                            const long long* off2, const int* len2, long long npairs, const swb200_params* pp, AlignKind kind,
                            int* scores_out, int* spans_out, unsigned int* ops_out, int ops_stride, int* ops_count) {
  if (npairs < 0 || ops_stride < 1 ||
      (npairs > 0 && (!seq1_all || !seq2_all || !off1 || !off2 || !len1 || !len2 || !scores_out || !spans_out || !ops_out || !ops_count)))
    return fail(SWB200_ERR_ARG, "bad batch arguments");
  const swb200_params p = params_or_default(pp);
  const HostPairs in{seq1_all, off1, len1, seq2_all, off2, len2};
  auto check = [&](const PairScan& whole) {
    if (whole.neg < 0) return fail(SWB200_ERR_ARG, "negative length or offset");
    int rc;
    if ((rc = check_params(p))) return rc;
    return check_align_batch_limits(p, whole.max_min);
  };
  if (npairs == 0) return check(PairScan{});
  return run_host_batch(
      npairs, [&](long long k0, long long k1) { return scan_pairs(in, k0, k1); }, check,
      [&](swb200_ctx* c, long long k0, long long k1, const PairScan& part, const PairScan& whole) {
        return align_batch_host_ctx(c, in.from(k0), k1 - k0, part, whole, p, kind, 0, 0, scores_out + k0, spans_out + 4 * k0,
                                    ops_out + k0 * (long long)ops_stride, ops_stride, ops_count + k0);
      });
}

extern "C" {

int swb200_align_batch(const unsigned char* seq1_all, const long long* off1, const int* len1, const unsigned char* seq2_all,
                       const long long* off2, const int* len2, long long npairs, const swb200_params* pp, const swb200_options* opt,
                       int* scores_out, int* spans_out, unsigned int* ops_out, int ops_stride, int* ops_count) {
  (void)opt;
  return align_batch_host(seq1_all, off1, len1, seq2_all, off2, len2, npairs, pp, AlignKind::batch, scores_out, spans_out, ops_out,
                          ops_stride, ops_count);
}

int swb200_align_batch_bytes(const unsigned char* seq1_all, const long long* off1, const int* len1, const unsigned char* seq2_all,
                             const long long* off2, const int* len2, long long npairs, const swb200_params* pp,
                             const swb200_options* opt, int* scores_out, int* spans_out, unsigned int* ops_out, int ops_stride,
                             int* ops_count) {
  (void)opt;
  return align_batch_host(seq1_all, off1, len1, seq2_all, off2, len2, npairs, pp, AlignKind::bytes, scores_out, spans_out, ops_out,
                          ops_stride, ops_count);
}

int swb200_batch_align(swb200_batch* b, const swb200_params* pp, const swb200_options* opt, void* stream, int* d_scores,
                       int* d_spans, unsigned int* d_ops, int ops_stride, int* d_ops_count) {
  (void)opt;
  if (!b || ops_stride < 1 || (b->npairs > 0 && (!d_scores || !d_spans || !d_ops || !d_ops_count)))
    return fail(SWB200_ERR_ARG, "bad batch arguments");
  if (b->keep_order || !b->len1) return fail(SWB200_ERR_ARG, "batch was packed in caller order (banded); re-pack with keep_order=0");
  const swb200_params p = params_or_default(pp);
  int rc;
  if ((rc = check_params(p)) || (rc = check_align_batch_limits(p, b->max_short))) return rc;
  return run_device_batch(b, 0, stream, [&](swb200_ctx* c, cudaStream_t s) {
    return align_packed_locked(c, whole_batch(b), b->len1, p, s, d_scores, d_spans, d_ops, ops_stride, d_ops_count, &c->info);
  });
}

int swb200_align_banded_batch(const unsigned char* seq1_all, const long long* off1, const int* len1,
                              const unsigned char* seq2_all, const long long* off2, const int* len2, long long npairs,
                              int band_lo, int band_hi, const swb200_params* pp, const swb200_options* opt, int* scores_out,
                              int* spans_out, unsigned int* ops_out, int ops_stride, int* ops_count) {
  (void)opt;
  if (int rc = check_band_width(band_lo, band_hi)) return rc;
  if (npairs < 0 || ops_stride < 1 ||
      (npairs > 0 && (!seq1_all || !seq2_all || !off1 || !off2 || !len1 || !len2 || !scores_out || !spans_out || !ops_out || !ops_count)))
    return fail(SWB200_ERR_ARG, "bad batch arguments");
  const swb200_params p = params_or_default(pp);
  const HostPairs in{seq1_all, off1, len1, seq2_all, off2, len2};
  auto check = [&](const PairScan& whole) { return check_score_pairs(whole, p, swb200_options{}, ScoreKind::banded, band_lo, band_hi); };
  if (npairs == 0) return check(PairScan{});
  return run_host_batch(
      npairs, [&](long long k0, long long k1) { return scan_pairs(in, k0, k1); }, check,
      [&](swb200_ctx* c, long long k0, long long k1, const PairScan& part, const PairScan& whole) {
        return align_batch_host_ctx(c, in.from(k0), k1 - k0, part, whole, p, AlignKind::banded, band_lo, band_hi - band_lo + 1,
                                    scores_out + k0, spans_out + 4 * k0,
                                    ops_out + k0 * (long long)ops_stride, ops_stride, ops_count + k0);
      });
}

int swb200_batch_align_banded(swb200_batch* b, int band_lo, int band_hi, const swb200_params* pp, const swb200_options* opt,
                              void* stream, int* d_scores, int* d_spans, unsigned int* d_ops, int ops_stride, int* d_ops_count) {
  (void)opt;
  if (!b || ops_stride < 1 || (b->npairs > 0 && (!d_scores || !d_spans || !d_ops || !d_ops_count)))
    return fail(SWB200_ERR_ARG, "bad batch arguments");
  const swb200_params p = params_or_default(pp);
  int rc;
  if ((rc = refuse_bytes(b)) || (rc = check_params(p)) ||
      (rc = check_banded_score(p, b->keep_order, band_lo, band_hi, b->max_short, b->max_long))) return rc;
  return run_device_batch(b, 0, stream, [&](swb200_ctx* c, cudaStream_t s) {
    return align_banded_packed_locked(c, whole_batch(b), band_lo, band_hi - band_lo + 1, p, s, d_scores, d_spans, d_ops, ops_stride,
                                      d_ops_count, &c->info);
  });
}

int swb200_align_long_batch(const unsigned char* seq1_all, const long long* off1, const int* len1,
                            const unsigned char* seq2_all, const long long* off2, const int* len2, long long npairs,
                            const swb200_params* pp, const swb200_options* opt, int* scores_out, int* spans_out,
                            unsigned int* ops_out, int ops_stride, int* ops_count) {
  (void)opt;
  if (npairs < 0 || ops_stride < 1 ||
      (npairs > 0 && (!seq1_all || !seq2_all || !off1 || !off2 || !len1 || !len2 || !scores_out || !spans_out || !ops_out || !ops_count)))
    return fail(SWB200_ERR_ARG, "bad batch arguments");
  const swb200_params p = params_or_default(pp);
  const HostPairs in{seq1_all, off1, len1, seq2_all, off2, len2};
  auto check = [&](const PairScan& whole) { return check_score_pairs(whole, p, swb200_options{}, ScoreKind::long_pairs, 0, 0); };
  if (npairs == 0) return check(PairScan{});
  return run_host_batch(
      npairs, [&](long long k0, long long k1) { return scan_pairs(in, k0, k1); }, check,
      [&](swb200_ctx* c, long long k0, long long k1, const PairScan& part, const PairScan& whole) {
        return align_batch_host_ctx(c, in.from(k0), k1 - k0, part, whole, p, AlignKind::long_pairs, 0, 0, scores_out + k0,
                                    spans_out + 4 * k0, ops_out + k0 * (long long)ops_stride, ops_stride, ops_count + k0);
      });
}

int swb200_batch_align_long(swb200_batch* b, const swb200_params* pp, const swb200_options* opt, void* stream, int* d_scores,
                            int* d_spans, unsigned int* d_ops, int ops_stride, int* d_ops_count) {
  (void)opt;
  if (!b || ops_stride < 1 || (b->npairs > 0 && (!d_scores || !d_spans || !d_ops || !d_ops_count)))
    return fail(SWB200_ERR_ARG, "bad batch arguments");
  if (b->keep_order || !b->len1) return fail(SWB200_ERR_ARG, "batch was packed in caller order (banded); re-pack with keep_order=0");
  const swb200_params p = params_or_default(pp);
  int rc;
  if ((rc = refuse_bytes(b)) || (rc = check_params(p)) || (rc = check_long_score(p, swb200_options{}, 0, b->max_short))) return rc;
  return run_device_batch(b, 0, stream, [&](swb200_ctx* c, cudaStream_t s) {
    return align_long_packed_locked(c, whole_batch(b), b->len1, p, s, d_scores, d_spans, d_ops, ops_stride, d_ops_count, &c->info);
  });
}

}  // extern "C"

extern "C" {

// ---- the reference's names (algoGPU.h:5-9, SmithDiagonalGPUrefactored.cu:174) ---------------------
int SequentialSmithWatermanScoreGPU(unsigned char* seq1, unsigned char* seq2, int len1, int len2) {
  return legacy(seq1, seq2, len1, len2, "SequentialSmithWatermanScoreGPU");
}
int SmithWatermanLazyGPU(const unsigned char* seq1, const unsigned char* seq2, int n, int m) {
  return legacy(seq1, seq2, n, m, "SmithWatermanLazyGPU");
}
int SmithWatermanScoreCUDA(const unsigned char* seq1, const unsigned char* seq2, int n, int m) {
  return legacy(seq1, seq2, n, m, "SmithWatermanScoreCUDA");
}
int SmithDiagonalGPU(unsigned char* seq1, unsigned char* seq2, int n, int m) {
  return legacy(seq1, seq2, n, m, "SmithDiagonalGPU");
}

}  // extern "C"
