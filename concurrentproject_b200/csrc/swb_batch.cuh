// swb_batch.cuh -- many independent pairs at once (BASELINE config 4: 150 bp reads vs 1 kb windows).
//
// Same recurrence and the same packed-16-bit striping as the single-pair engine (swb_engine.cuh), but
// a pair is small enough for a GROUP of G lanes (G = 8: sixteen sub-lanes x R rows cover a read of up
// to 16*R bases), so a warp scores 32/G pairs side by side and nothing ever leaves the registers:
// the top boundary of every pair is the zero row of main.cpp:43-52, there is no hand-off, no polling.
// The shorter sequence of a pair is striped (Q), the longer one is streamed (T).
// The reference has no batch entry point; its harness loops over pairs (TestFileWithGPU.cpp:57-94).
#pragma once
#include "swb_engine.cuh"

#ifndef SWB_BATCH_UNROLL
#define SWB_BATCH_UNROLL 4
#endif
namespace swb {
constexpr int kSwbBatchUnroll = SWB_BATCH_UNROLL;   // step-loop unroll factor

constexpr int kBatchRing = 128;   // per-group ring of substitution tables, kept twice

struct BatchParams {
  const uint64_t* q_words;   // striped sequences, 2-bit packed, q_stride words per pair
  const uint64_t* t_words;   // streamed sequences, 2-bit packed, t_stride words per pair
  const int* q_len;          // per pair (after the shorter/longer swap)
  const int* t_len;
  long long q_stride, t_stride;
  long long npairs;
  int* scores;
  int match, mismatch, gap_init, gap_ext;
};

// smem per warp: 32/G groups x 2*kBatchRing words  (sized for G = 8)
struct BatchWarpSmem {
  uint32_t tab[4 * 2 * kBatchRing];
};

// LONG (G = 32, one pair per warp, no cap on the shorter side): Q is cut into bands of 64*R rows and the warp sweeps
// band 0 over the whole of T, then band 1, and so on (DESIGN.md section 4d).  Lane 31's bottom-row word xsend (H - gap_init
// and F as s16x2; the linear mode: H - gap_init only) goes per T column into the warp's boundary row `bnd` (one word per
// column, updated in place); in the next band lane 31 hands that word to lane 0 where band 0 hands it the zero row.  Pairs
// come from the counter *next_pair (zeroed by the host before the launch), so a warp that drew a short pair takes the next
// one while others still sweep long ones.  Nothing waits on another warp.
template <int R, int MODE, int G, bool LONG = false>
SWB_HD void batch_warp(const BatchParams& P, const WarpCtx& w, long long warp_id, long long num_warps, BatchWarpSmem* sm,
                       uint32_t* bnd = nullptr, unsigned long long* next_pair = nullptr) {
  static_assert(!LONG || G == 32, "the multi-band sweep runs one pair per warp");
  constexpr int GROUPS = 32 / G;
  constexpr int SK = 2;                      // lane skew (boundary value consumed in the step after it was made)
  constexpr int SKEW = SK * (G - 1) + 1;
  const int lane = w.lane;
  const int gl = lane % G, grp = lane / G;
  const bool last_in_group = gl == G - 1;
  const int src_lane = grp * G + (gl + G - 1) % G;
  const uint32_t nopen = pack2(-P.gap_init), next = pack2(-P.gap_ext);
  const uint32_t padb = (uint32_t)(P.mismatch + P.gap_init) & 0xFFu;
  const uint32_t padw = padb * 0x01010101u;
  const uint32_t flip = padb ^ ((uint32_t)(P.match + P.gap_init) & 0xFFu);
  uint32_t* tab = sm->tab + grp * 2 * kBatchRing;
  const long long ngroups = (P.npairs + GROUPS - 1) / GROUPS;

  auto take = [&]() -> long long {                 // LONG: the next pair from the launch's counter
    unsigned long long v = 0;
    if (lane == 0) v = atomic_fetch_add_u64(next_pair, 1ull);
    return (long long)(((unsigned long long)w.shfl((uint32_t)(v >> 32), 0) << 32) | w.shfl((uint32_t)v, 0));
  };
  // LONG: the boundary row is staged in the 3/4 of sm->tab the single group leaves free: bin[2][32] holds the words lane
  // 31 hands down in this chunk of 32 steps (and the next), bout[128] collects lane 31's bottom-row words by column
  uint32_t* const bin = sm->tab + 2 * kBatchRing;
  uint32_t* const bout = bin + 2 * kChunk;
  for (long long pg = LONG ? take() : warp_id; pg < ngroups; pg = LONG ? take() : pg + num_warps) {
    const long long pair = pg * GROUPS + grp;
    const bool valid = pair < P.npairs;
    const int LQ = valid ? P.q_len[pair] : 0;
    const int LT = valid ? P.t_len[pair] : 0;
    const uint64_t* qw = P.q_words + (valid ? pair : 0) * P.q_stride;
    const uint64_t* tw = P.t_words + (valid ? pair : 0) * P.t_stride;
    const int maxLT = w.reduce_max(LT);
    const int nsteps = ((maxLT + SKEW + kChunk - 1) / kChunk) * kChunk;
    constexpr int BAND = 2 * G * R;                                   // rows of one band
    const int nbands = LONG ? (LQ + BAND - 1) / BAND : 1;            // LONG, LQ = 0: one band of pad rows, score 0
    uint32_t pair_best0 = 0, pair_best1 = 0;                          // carried across the bands
    int band = 0;
    do {
      const bool carry_out = LONG && band + 1 < nbands;                 // the next band reads this band's bottom row
      uint32_t sel[R];
      {
        const int row_lo = band * BAND + 2 * gl * R;
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const int a = row_lo + r, b = row_lo + R + r;
          const uint32_t ca = a < LQ ? (uint32_t)(qw[a >> 5] >> (2 * (a & 31))) & 3u : 4u;
          const uint32_t cb = b < LQ ? (uint32_t)(qw[b >> 5] >> (2 * (b & 31))) & 3u : 4u;
          sel[r] = mk_sel16(ca, cb);
        }
      }
      uint32_t Ho[R], E[R];
#pragma unroll
      for (int r = 0; r < R; ++r) { Ho[r] = nopen; E[r] = nopen; }
      uint32_t Fbot = nopen, up_prev = nopen, xsend = nopen, Thi = padw;
      uint32_t best0 = pair_best0, best1 = pair_best1;

      // table ring of this group: all pad, then positions [0, 32); each lane converts 32/G symbols
      w.sync();
      for (int k = gl; k < 2 * kBatchRing; k += G) tab[k] = padw;
      w.sync();
      constexpr int PER = kChunk / G;          // symbols per lane per refill
      uint64_t tword = LT > 0 ? tw[0] : 0ull;
#pragma unroll
      for (int u = 0; u < PER; ++u) {
        const int q = gl * PER + u;
        const uint32_t c = q < LT ? (uint32_t)(tword >> (2 * q)) & 3u : 4u;
        const uint32_t t = table_word(c, padw, flip);
        tab[q] = t;
        tab[q + kBatchRing] = t;
      }
      uint64_t twpref = kChunk < LT ? tw[1] : 0ull;
      // boundary words of columns [0, 32): the zero row in band 0 and at columns >= LT (pad cells: they never feed a real one)
      uint32_t bpref = nopen;
      if (LONG && band > 0 && lane < LT) bpref = bnd[lane];

      for (int i0 = 0; i0 < nsteps; i0 += kChunk) {
        // tables for positions [i0+32, i0+64)
#pragma unroll
        for (int u = 0; u < PER; ++u) {
          const int q = i0 + kChunk + gl * PER + u;
          const uint32_t c = q < LT ? (uint32_t)(twpref >> (2 * (q & 31))) & 3u : 4u;
          const uint32_t t = table_word(c, padw, flip);
          tab[q & (kBatchRing - 1)] = t;
          tab[(q & (kBatchRing - 1)) + kBatchRing] = t;
        }
        twpref = (i0 + 2 * kChunk < LT) ? tw[(i0 + 2 * kChunk) >> 5] : 0ull;
        uint32_t* const binp = bin + (i0 & kChunk);
        if (LONG) {
          // One boundary row per warp, updated in place, is safe: lane 0 of this band consumes column c at step c (its word
          // was loaded into bpref a whole chunk earlier), while lane 31 produces column c at step c + SKEW = c + 63 and the
          // warp stores it only after the chunk that completes its 128-byte line.  So this chunk's load covers
          // [i0+32, i0+64) and its store covers [i0-96, i0-64): disjoint, and every column is read before it is written.
          // Load and store of a column are made by the same lane (column % 32), so no other ordering is needed.
          binp[lane] = bpref;
          const int c = i0 + kChunk + lane;
          bpref = (band > 0 && c < LT) ? bnd[c] : nopen;
        }
        w.sync();
        if (carry_out) {
          const int c = i0 - 3 * kChunk + lane;                          // lane 31 wrote its last word at step i0-1
          if (c >= 0 && c < LT) bnd[c] = bout[(c + SKEW) & (4 * kChunk - 1)];
        }
        uint32_t* const boutp = bout + (i0 & (4 * kChunk - 1));          // column i0+k-SKEW at slot (i0+k) % 128
        const uint32_t* tabp = tab + ((i0 - SK * gl) & (kBatchRing - 1));
        uint32_t Tnext = tabp[0];
#pragma unroll (kSwbBatchUnroll)
        for (int k = 0; k < kChunk; ++k) {
          const uint32_t Tlo = Tnext;
          Tnext = tabp[k + 1];
          // lane 0 of a group gets the zero boundary row (LONG: the row above the band)
          const uint32_t xs = last_in_group ? (LONG ? binp[k] : nopen) : xsend;
          const uint32_t yuse = w.shfl(xs, src_lane);
          uint32_t upHo, F;
          if (MODE == 0) {
            upHo = prmt(yuse, Ho[R - 1], 0x5410u);
            F = prmt(yuse, Fbot, 0x5432u);
          } else {
            upHo = prmt(yuse, Ho[R - 1], 0x5432u);
            F = 0;
          }
          uint32_t diag = up_prev, Hup = upHo;
          up_prev = upHo;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const uint32_t s = prmt(Tlo, Thi, sel[r]);
            const uint32_t old = Ho[r];
            uint32_t h;
            if (MODE == 0) {
              const uint32_t d = add16x2(diag, s);
              E[r] = addmax16x2(E[r], next, old);
              F = addmax16x2(F, next, Hup);
              h = max3relu16x2(d, E[r], F);
            } else {
              // the clamp at 0 rides on the fused add-max; the second max is then the plain (full-rate) VIMNMX
              h = max16x2(addmaxrelu16x2(diag, s, old), Hup);
            }
            Ho[r] = add16x2(h, nopen);
            Hup = Ho[r];
            diag = old;
            if (r & 1) best1 = max16x2(best1, h); else best0 = max16x2(best0, h);
          }
          Fbot = F;
          xsend = (MODE == 0) ? prmt(Ho[R - 1], Fbot, 0x7632u) : Ho[R - 1];
          if (carry_out && last_in_group) boutp[k] = xsend;
          Thi = Tlo;
        }
      }
      if (carry_out) {
        // the last two lines: [nsteps-96, nsteps-64) and the one holding column nsteps-64 >= LT-1
        w.sync();
        for (int c = nsteps - 3 * kChunk + lane; c < nsteps - kChunk; c += kChunk)
          if (c >= 0 && c < LT) bnd[c] = bout[(c + SKEW) & (4 * kChunk - 1)];
      }
      pair_best0 = best0; pair_best1 = best1;
    } while (LONG && ++band < nbands);
    // best of the group
    const uint32_t b = max16x2(pair_best0, pair_best1);
    int m = (int)(short)(b & 0xFFFFu), mh = (int)(short)(b >> 16);
    m = m > mh ? m : mh;
#pragma unroll
    for (int d = 1; d < G; d <<= 1) {
      const int o = (int)w.shfl((uint32_t)m, lane ^ d);
      m = m > o ? m : o;
    }
    if (valid && gl == 0) P.scores[pair] = m;
  }
}

#ifdef __CUDACC__
template <int R, int MODE, int G>
__global__ void __launch_bounds__(256, 2) sw_batch_kernel(const __grid_constant__ BatchParams P) {
  __shared__ BatchWarpSmem sm[8];
  WarpCtx w{(int)(threadIdx.x & 31)};
  const int wi = (int)(threadIdx.x >> 5);
  batch_warp<R, MODE, G>(P, w, (long long)blockIdx.x * 8 + wi, (long long)gridDim.x * 8, &sm[wi]);
}

// The multi-band batch kernel: one pair per warp, any shorter side.  bnd: bnd_stride words per launched warp.
template <int R, int MODE>
__global__ void __launch_bounds__(256, 2) sw_long_batch_kernel(const __grid_constant__ BatchParams P, uint32_t* bnd,
                                                               long long bnd_stride, unsigned long long* next_pair) {
  __shared__ BatchWarpSmem sm[8];
  WarpCtx w{(int)(threadIdx.x & 31)};
  const int wi = (int)(threadIdx.x >> 5);
  const long long warp = (long long)blockIdx.x * 8 + wi;
  batch_warp<R, MODE, 32, true>(P, w, warp, (long long)gridDim.x * 8, &sm[wi], bnd + warp * bnd_stride, next_pair);
}
#endif

constexpr int kBatchRowChoices[] = {2, 4, 6, 8, 10, 12, 16};
constexpr int kNumBatchRowChoices = 7;
const void* batch_kernel(int R, int mode, int G);
const void* long_batch_kernel(int R, int mode);

}  // namespace swb
