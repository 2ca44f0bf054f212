// swb_banded.cuh -- banded Gotoh local alignment for batches of long pairs (BASELINE config 5).
//
// Semantics (SURVEY.md 8c; oracle: oracle_gotoh_banded): cell (i,j), 1-based, is in band iff
// band_lo <= j-i <= band_lo+63; out-of-band cells are H=E=F=0 and excluded from the max, i.e. main.cpp:57-63
// evaluated on in-band cells only.  The reference has no banded mode.
//
// Geometry.  The 64 diagonals k = j-i of a pair are spread over 16 threads.  Thread u holds four of them in two
// packed register sets: A = (2u, 2u+32) and B = (2u+1, 2u+33) (offsets from band_lo; lo half, hi half).  The sweep
// goes over anti-diagonals t = i+j; on one anti-diagonal only the diagonals with k = t (mod 2) have a cell, so steps
// alternate A, B, A, B and every packed instruction does two useful cells.  A cell's left neighbour is diagonal k-1
// and its upper neighbour diagonal k+1, both on the previous anti-diagonal: for set A the upper neighbours are the
// thread's own B registers and the left neighbours are thread u-1's B registers -- BOTH halves at once, because the
// two halves of a register are 32 diagonals apart -- so one __shfl_sync per step moves a whole register and no
// half-word merging is needed (set B: left = own A, upper = thread u+1's A).  The seam between diagonal 31 and 32
// rides on the same rotation: thread 15 sends (border, its B.lo) to thread 0, thread 0 sends (its A.hi, border) to
// thread 15, one PRMT with a per-thread selector.  The diagonal neighbour is the cell's own register two steps
// ago.  Two pairs per warp.  Substitution scores: one PRMT per cell vector from two shared-memory rings filled
// cooperatively per pair, a 4-byte score table per column symbol (as in the pair engine) and a PRMT selector per
// row pair (rows y and y-16: the hi half is 16 rows up and 16 columns right of the lo half).
#pragma once
#include "swb_engine.cuh"

#ifndef SWB_BANDED_UNROLL
#define SWB_BANDED_UNROLL 4
#endif
namespace swb {
constexpr int kSwbBandedUnroll = SWB_BANDED_UNROLL;   // step-loop unroll factor

constexpr int kBandRing = 128;     // ring entries (tables per column / selectors per row), kept twice
constexpr int kBandThreads = 16;   // threads per pair
constexpr int kBandWidth = 64;     // diagonals per pair

struct BandedParams {
  const uint64_t* a_words;   // seq1 (columns j), 2-bit packed, a_stride words per pair
  const uint64_t* b_words;   // seq2 (rows i)
  const int* a_len;
  const int* b_len;
  long long a_stride, b_stride;
  long long npairs;
  int band_lo;               // band is band_lo <= j-i <= band_lo+W-1 (W: the kernel's width)
  int* scores;
  int match, mismatch, gap_init, gap_ext;
};

// The two pairs of a warp read the same ring offsets in the same instruction: 16 words of padding put the
// second pair's ring 16 banks away from the first one's, so the 2 x 16 threads hit 32 different banks
// (without it every LDS of the step loop was a 2-way bank conflict and the LSU the bottleneck).
struct BandedWarpSmem {
  uint32_t tab[2][2 * kBandRing + 16];   // [pair in warp][ring]: score table of column x at slot x & 127
  uint32_t sel[2][2 * kBandRing + 16];   // selector of rows (y, y-16) at slot y & 127
};

SWB_HD uint32_t packed_code(const uint64_t* words, int pos, int len) {
  return (pos >= 0 && pos < len) ? (uint32_t)(words[pos >> 5] >> (2 * (pos & 31))) & 3u : 4u;
}

// word i of a pair's packed sequence, the index clamped to the pair's words (0 for an empty layout)
SWB_HD uint64_t packed_word(const uint64_t* words, long long stride, int i) {
  const long long k = i < 0 ? 0 : (i < stride ? i : stride - 1);
  return stride > 0 ? words[k] : 0ull;
}
// 64 bits starting at bit sh (0 .. 62) of the 128-bit value hi:lo
SWB_HD uint64_t funnel64(uint64_t lo, uint64_t hi, int sh) { return (lo >> sh) | ((hi << 1) << (63 - sh)); }

template <int MODE>
SWB_HD void banded_warp(const BandedParams& P, const WarpCtx& w, long long warp_id, long long num_warps, BandedWarpSmem* sm) {
  const int lane = w.lane;
  const int u = lane & 15, grp = lane >> 4;
  const int src_prev = grp * 16 + ((u + 15) & 15);     // A-step: registers come from thread u-1 (rotating)
  const int src_next = grp * 16 + ((u + 1) & 15);      // B-step: registers come from thread u+1 (rotating)
  const uint32_t nopen = pack2(-P.gap_init), next = pack2(-P.gap_ext);
  const uint32_t padb = (uint32_t)(P.mismatch + P.gap_init) & 0xFFu;
  const uint32_t padw = padb * 0x01010101u;
  const uint32_t flip = padb ^ ((uint32_t)(P.match + P.gap_init) & 0xFFu);
  const uint32_t padsel = mk_sel16(4u, 4u);
  // what a thread sends: its register as is, except at the seam (prmt(x, nopen, sel): bytes 0-3 = x, 4-7 = nopen)
  const uint32_t sel_left = u == 15 ? 0x1054u : 0x3210u;   // thread 15 -> thread 0: (border, B.lo = diagonal 31)
  const uint32_t sel_up = u == 0 ? 0x7632u : 0x3210u;      // thread 0 -> thread 15: (A.hi = diagonal 32, border)
  uint32_t* tab = sm->tab[grp];
  uint32_t* sel = sm->sel[grp];
  const long long ngroups = (P.npairs + 1) / 2;
  // first anti-diagonal handled by register set A: the largest t <= 2 with t = band_lo (mod 2)
  const int tA0 = 2 - ((2 - P.band_lo) & 1);
  const int I0 = (tA0 - P.band_lo) / 2, J0 = (tA0 + P.band_lo) / 2;      // exact: both numerators are even

  for (long long pg = warp_id; pg < ngroups; pg += num_warps) {
    const long long pair = pg * 2 + grp;
    const bool valid = pair < P.npairs;
    const int n = valid ? P.a_len[pair] : 0, m = valid ? P.b_len[pair] : 0;
    const uint64_t* aw = P.a_words + (valid ? pair : 0) * P.a_stride;
    const uint64_t* bw = P.b_words + (valid ? pair : 0) * P.b_stride;
    const int NH = (n > 0 && m > 0) ? (n + m - tA0) / 2 + 1 : 0;         // double steps (one A + one B anti-diagonal)
    const int maxNH = w.reduce_max(NH);
    const int nchunks = (maxNH + kChunk - 1) / kChunk;

    // state of the 4 diagonals: H-open, E, F of register sets A and B; all cells start as border (H 0, E/F <= 0)
    uint32_t HoA = nopen, EA = nopen, FA = nopen, HoB = nopen, EB = nopen, FB = nopen;
    uint32_t best = 0;
    // 0-based sequence positions of this thread's A.lo cell at double step h: row y = Y0 + h, column x = X0 + h;
    // A.hi: (y - 16, x + 16); B.lo: (y, x + 1); B.hi: (y - 16, x + 17)
    const int Y0 = I0 - u - 1, X0 = J0 + u - 1;

    // ---- rings: everything pad, then selectors for rows [Yc-32, Yc) and tables for columns [Xc, Xc+32) of chunk 0
    const int Yc0 = I0 - 1, Xc0 = J0 - 1;                                  // thread 0's positions at h = 0
    w.sync();
    for (int k = u; k < 2 * kBandRing; k += 16) { tab[k] = padw; sel[k] = padsel; }
    w.sync();
    for (int k = u; k < kChunk; k += 16) {
      const int y = Yc0 - kChunk + k;
      const uint32_t sv = mk_sel16(packed_code(bw, y, m), packed_code(bw, y - 16, m));
      sel[y & (kBandRing - 1)] = sv; sel[(y & (kBandRing - 1)) + kBandRing] = sv;
      const int x = Xc0 + k;
      const uint32_t tv = table_word(packed_code(aw, x, n), padw, flip);
      tab[x & (kBandRing - 1)] = tv; tab[(x & (kBandRing - 1)) + kBandRing] = tv;
    }

    for (int c = 0; c < nchunks; ++c) {
      // ---- this chunk reads rows [Yc-15, Yc+32) and columns [Xc, Xc+64): add rows [Yc, Yc+32), columns [Xc+32, Xc+64)
      const int Yc = Yc0 + c * kChunk, Xc = Xc0 + c * kChunk;
      for (int k = u; k < kChunk; k += 16) {
        const int y = Yc + k;
        const uint32_t sv = mk_sel16(packed_code(bw, y, m), packed_code(bw, y - 16, m));
        sel[y & (kBandRing - 1)] = sv; sel[(y & (kBandRing - 1)) + kBandRing] = sv;
        const int x = Xc + kChunk + k;
        const uint32_t tv = table_word(packed_code(aw, x, n), padw, flip);
        tab[x & (kBandRing - 1)] = tv; tab[(x & (kBandRing - 1)) + kBandRing] = tv;
      }
      w.sync();
      const uint32_t* selp = sel + ((Y0 + c * kChunk) & (kBandRing - 1));
      const uint32_t* tabp = tab + ((X0 + c * kChunk) & (kBandRing - 1));
      uint32_t a0 = tabp[0], b0 = tabp[16];
#pragma unroll (kSwbBandedUnroll)
      for (int h = 0; h < kChunk; ++h) {
        const uint32_t sv = selp[h];
        const uint32_t a1 = tabp[h + 1], b1 = tabp[h + 17];
        const uint32_t sA = prmt(a0, b0, sv);        // A.lo: row y, column x ; A.hi: row y-16, column x+16
        const uint32_t sB = prmt(a1, b1, sv);        // B.lo: row y, column x+1 ; B.hi: row y-16, column x+17
        a0 = a1; b0 = b1;
        // ---------------- anti-diagonal of set A: left neighbours = thread u-1's B, upper neighbours = own B
        {
          uint32_t h2;
          const uint32_t leftHo = w.shfl(prmt(HoB, nopen, sel_left), src_prev);
          if (MODE == 0) {
            const uint32_t leftE = w.shfl(prmt(EB, nopen, sel_left), src_prev);
            const uint32_t E = addmax16x2(leftE, next, leftHo);
            const uint32_t F = addmax16x2(FB, next, HoB);
            const uint32_t d = add16x2(HoA, sA);
            h2 = max3relu16x2(d, E, F);
            EA = E; FA = F;
          } else {
            h2 = max16x2(addmaxrelu16x2(HoA, sA, leftHo), HoB);
          }
          HoA = add16x2(h2, nopen);
          best = max16x2(best, h2);
        }
        // ---------------- anti-diagonal of set B: left neighbours = own A, upper neighbours = thread u+1's A
        {
          uint32_t h2;
          const uint32_t upHo = w.shfl(prmt(HoA, nopen, sel_up), src_next);
          if (MODE == 0) {
            const uint32_t upF = w.shfl(prmt(FA, nopen, sel_up), src_next);
            const uint32_t E = addmax16x2(EA, next, HoA);
            const uint32_t F = addmax16x2(upF, next, upHo);
            const uint32_t d = add16x2(HoB, sB);
            h2 = max3relu16x2(d, E, F);
            EB = E; FB = F;
          } else {
            h2 = max16x2(addmaxrelu16x2(HoB, sB, HoA), upHo);
          }
          HoB = add16x2(h2, nopen);
          best = max16x2(best, h2);
        }
      }
    }
    int mx = (int)(short)(best & 0xFFFFu), mh = (int)(short)(best >> 16);
    mx = mx > mh ? mx : mh;
#pragma unroll
    for (int d = 1; d < 16; d <<= 1) {
      const int o = (int)w.shfl((uint32_t)mx, lane ^ d);
      mx = mx > o ? mx : o;
    }
    if (valid && u == 0) P.scores[pair] = mx;
  }
}

#ifdef __CUDACC__
template <int MODE>
__global__ void __launch_bounds__(256, 4) sw_banded_kernel(const __grid_constant__ BandedParams P) {
  __shared__ BandedWarpSmem sm[8];
  WarpCtx w{(int)(threadIdx.x & 31)};
  const int wi = (int)(threadIdx.x >> 5);
  banded_warp<MODE>(P, w, (long long)blockIdx.x * 8 + wi, (long long)gridDim.x * 8, &sm[wi]);
}
#endif

const void* banded_kernel(int mode);

// =================================================================================================
//  Round 2: 8 threads per pair, four packed register sets per thread.
//  Thread u holds the diagonals 4u+s (lo half) and 4u+s+32 (hi half), s = 0..3, as sets S0..S3.  On an even
//  anti-diagonal S0 and S2 have a cell, on an odd one S1 and S3.  Only the two OUTER sets talk to a neighbouring
//  thread (S0's left neighbour is thread u-1's S3, S3's upper neighbour is thread u+1's S0); S1 and S2 find both
//  neighbours in the thread's own registers.  So a double step computes FOUR cell vectors with the shuffles of the
//  16-thread layout's two (2 in linear mode, 4 affine) and three shared-memory loads instead of six: 6.75 instead of
//  8.5 instructions per cell vector (linear), 10.75 instead of 12.5 (affine).  Four pairs per warp.
//  Positions (0-based) of S0.lo at double step h: row y = I0 - 2u - 1 + h, column x = J0 + 2u - 1 + h;
//  S1.lo: (y, x+1); S2.lo: (y-1, x+1); S3.lo: (y-1, x+2); hi halves: 16 rows up, 16 columns right.
// =================================================================================================
constexpr int kBand8Threads = 8;
struct BandedWarpSmem8 {
  uint32_t tab[4][2 * kBandRing + 8];    // 8 words of padding: the four pairs of a warp sit 8 banks apart
  uint32_t sel[4][2 * kBandRing + 8];
};

template <int MODE>
SWB_HD void banded_warp8(const BandedParams& P, const WarpCtx& w, long long warp_id, long long num_warps, BandedWarpSmem8* sm) {
  const int lane = w.lane;
  const int u = lane & 7, grp = lane >> 3;
  const int src_prev = grp * 8 + ((u + 7) & 7);        // even step: S0's left neighbours come from thread u-1 (rotating)
  const int src_next = grp * 8 + ((u + 1) & 7);        // odd step: S3's upper neighbours come from thread u+1 (rotating)
  const uint32_t nopen = pack2(-P.gap_init), next = pack2(-P.gap_ext);
  const uint32_t padb = (uint32_t)(P.mismatch + P.gap_init) & 0xFFu;
  const uint32_t padw = padb * 0x01010101u;
  const uint32_t flip = padb ^ ((uint32_t)(P.match + P.gap_init) & 0xFFu);
  const uint32_t padsel = mk_sel16(4u, 4u);
  // the seam between diagonal 31 and 32 rides on the rotation (prmt(x, nopen, sel): bytes 0-3 = x, 4-7 = nopen)
  const uint32_t sel_left = u == 7 ? 0x1054u : 0x3210u;    // thread 7 -> thread 0: (border, S3.lo = diagonal 31)
  const uint32_t sel_up = u == 0 ? 0x7632u : 0x3210u;      // thread 0 -> thread 7: (S0.hi = diagonal 32, border)
  uint32_t* tab = sm->tab[grp];
  uint32_t* sel = sm->sel[grp];
  const long long ngroups = (P.npairs + 3) / 4;
  const int tA0 = 2 - ((2 - P.band_lo) & 1);                             // first even-set anti-diagonal (see banded_warp)
  const int I0 = (tA0 - P.band_lo) / 2, J0 = (tA0 + P.band_lo) / 2;

  for (long long pg = warp_id; pg < ngroups; pg += num_warps) {
    const long long pair = pg * 4 + grp;
    const bool valid = pair < P.npairs;
    const int n = valid ? P.a_len[pair] : 0, m = valid ? P.b_len[pair] : 0;
    const uint64_t* aw = P.a_words + (valid ? pair : 0) * P.a_stride;
    const uint64_t* bw = P.b_words + (valid ? pair : 0) * P.b_stride;
    const int NH = (n > 0 && m > 0) ? (n + m - tA0) / 2 + 1 : 0;
    const int maxNH = w.reduce_max(NH);
    const int nchunks = (maxNH + kChunk - 1) / kChunk;

    uint32_t Ho[4], E[4], F[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { Ho[k] = nopen; E[k] = nopen; F[k] = nopen; }
    uint32_t best = 0;
    const int Y0 = I0 - 2 * u - 1, X0 = J0 + 2 * u - 1;

    // ---- rings: everything pad, then selectors for rows [Yc-32, Yc) and tables for columns [Xc, Xc+32) of chunk 0
    const int Yc0 = I0 - 1, Xc0 = J0 - 1;                                  // thread 0's positions at h = 0
    w.sync();
    for (int k = u; k < 2 * kBandRing; k += 8) { tab[k] = padw; sel[k] = padsel; }
    w.sync();
    for (int k = u; k < kChunk; k += 8) {
      const int y = Yc0 - kChunk + k;
      const uint32_t sv = mk_sel16(packed_code(bw, y, m), packed_code(bw, y - 16, m));
      sel[y & (kBandRing - 1)] = sv; sel[(y & (kBandRing - 1)) + kBandRing] = sv;
      const int x = Xc0 + k;
      const uint32_t tv = table_word(packed_code(aw, x, n), padw, flip);
      tab[x & (kBandRing - 1)] = tv; tab[(x & (kBandRing - 1)) + kBandRing] = tv;
    }

    for (int c = 0; c < nchunks; ++c) {
      // ---- this chunk reads rows [Yc-16, Yc+32) and columns [Xc, Xc+64): add rows [Yc, Yc+32), columns [Xc+32, Xc+64)
      const int Yc = Yc0 + c * kChunk, Xc = Xc0 + c * kChunk;
      for (int k = u; k < kChunk; k += 8) {
        const int y = Yc + k;
        const uint32_t sv = mk_sel16(packed_code(bw, y, m), packed_code(bw, y - 16, m));
        sel[y & (kBandRing - 1)] = sv; sel[(y & (kBandRing - 1)) + kBandRing] = sv;
        const int x = Xc + kChunk + k;
        const uint32_t tv = table_word(packed_code(aw, x, n), padw, flip);
        tab[x & (kBandRing - 1)] = tv; tab[(x & (kBandRing - 1)) + kBandRing] = tv;
      }
      w.sync();
      // ring windows of this thread: selp[h] = selector of row y; tabp[h] = table of column x (both read up to +18 / -1)
      const uint32_t* selp = sel + ((Y0 + c * kChunk - 1) & (kBandRing - 1)) + 1;
      const uint32_t* tabp = tab + ((X0 + c * kChunk) & (kBandRing - 1));
      uint32_t a0 = tabp[0], a1 = tabp[1], b0 = tabp[16], b1 = tabp[17];
      uint32_t svp = selp[-1];                                            // selector of row y - 1
#pragma unroll (kSwbBandedUnroll)
      for (int h = 0; h < kChunk; ++h) {
        const uint32_t sv = selp[h];
        const uint32_t a2 = tabp[h + 2], b2 = tabp[h + 18];
        const uint32_t s0 = prmt(a0, b0, sv);        // S0: row y,   column x
        const uint32_t s1 = prmt(a1, b1, sv);        // S1: row y,   column x+1
        const uint32_t s2 = prmt(a1, b1, svp);       // S2: row y-1, column x+1
        const uint32_t s3 = prmt(a2, b2, svp);       // S3: row y-1, column x+2
        a0 = a1; a1 = a2; b0 = b1; b1 = b2; svp = sv;
        // ---------------- even anti-diagonal: S0 (left = thread u-1's S3, up = own S1), S2 (left = own S1, up = own S3)
        {
          const uint32_t leftHo = w.shfl(prmt(Ho[3], nopen, sel_left), src_prev);
          uint32_t h0, h2;
          if (MODE == 0) {
            const uint32_t leftE = w.shfl(prmt(E[3], nopen, sel_left), src_prev);
            const uint32_t E0 = addmax16x2(leftE, next, leftHo), F0 = addmax16x2(F[1], next, Ho[1]);
            const uint32_t E2 = addmax16x2(E[1], next, Ho[1]), F2 = addmax16x2(F[3], next, Ho[3]);
            h0 = max3relu16x2(add16x2(Ho[0], s0), E0, F0);
            h2 = max3relu16x2(add16x2(Ho[2], s2), E2, F2);
            E[0] = E0; F[0] = F0; E[2] = E2; F[2] = F2;
          } else {
            h0 = max16x2(addmaxrelu16x2(Ho[0], s0, leftHo), Ho[1]);
            h2 = max16x2(addmaxrelu16x2(Ho[2], s2, Ho[1]), Ho[3]);
          }
          Ho[0] = add16x2(h0, nopen); Ho[2] = add16x2(h2, nopen);
          best = max3_16x2(best, h0, h2);
        }
        // ---------------- odd anti-diagonal: S1 (left = own S0, up = own S2), S3 (left = own S2, up = thread u+1's S0)
        {
          const uint32_t upHo = w.shfl(prmt(Ho[0], nopen, sel_up), src_next);
          uint32_t h1, h3;
          if (MODE == 0) {
            const uint32_t upF = w.shfl(prmt(F[0], nopen, sel_up), src_next);
            const uint32_t E1 = addmax16x2(E[0], next, Ho[0]), F1 = addmax16x2(F[2], next, Ho[2]);
            const uint32_t E3 = addmax16x2(E[2], next, Ho[2]), F3 = addmax16x2(upF, next, upHo);
            h1 = max3relu16x2(add16x2(Ho[1], s1), E1, F1);
            h3 = max3relu16x2(add16x2(Ho[3], s3), E3, F3);
            E[1] = E1; F[1] = F1; E[3] = E3; F[3] = F3;
          } else {
            h1 = max16x2(addmaxrelu16x2(Ho[1], s1, Ho[0]), Ho[2]);
            h3 = max16x2(addmaxrelu16x2(Ho[3], s3, Ho[2]), upHo);
          }
          Ho[1] = add16x2(h1, nopen); Ho[3] = add16x2(h3, nopen);
          best = max3_16x2(best, h1, h3);
        }
      }
    }
    int mx = (int)(short)(best & 0xFFFFu), mh = (int)(short)(best >> 16);
    mx = mx > mh ? mx : mh;
#pragma unroll
    for (int d = 1; d < 8; d <<= 1) {
      const int o = (int)w.shfl((uint32_t)mx, lane ^ d);
      mx = mx > o ? mx : o;
    }
    if (valid && u == 0) P.scores[pair] = mx;
  }
}

#ifdef __CUDACC__
template <int MODE>
__global__ void __launch_bounds__(128, 6) sw_banded8_kernel(const __grid_constant__ BandedParams P) {
  __shared__ BandedWarpSmem8 sm[4];
  WarpCtx w{(int)(threadIdx.x & 31)};
  const int wi = (int)(threadIdx.x >> 5);
  banded_warp8<MODE>(P, w, (long long)blockIdx.x * 4 + wi, (long long)gridDim.x * 4, &sm[wi]);
}
#endif

const void* banded8_kernel(int mode);

// =================================================================================================
//  Round 2, second step: the same layout for any even number S of packed register sets per thread (32 / S threads
//  per pair, S pairs per warp); instantiated for S = 8: four threads per pair, eight pairs per warp.
//  Thread u holds the diagonals S*u + s (lo half) and S*u + s + 32 (hi half), s = 0 .. S-1.  On an even anti-diagonal
//  the even sets have a cell, on an odd one the odd sets; only set 0 (left neighbour: thread u-1's set S-1) and set
//  S-1 (upper neighbour: thread u+1's set 0) talk to another thread, so a double step computes S cell vectors with
//  the same 2 (linear) / 4 (affine) shuffles and 3 shared-memory loads as before: 5.4 instead of 6.75 instructions
//  per cell vector (linear), 9.4 instead of 10.75 (affine).
//  Positions (0-based) at double step h, with y = I0 - (S/2) u - 1 + h and x = J0 + (S/2) u - 1 + h:
//  set 2e: row y - e, column x + e; set 2e+1: row y - e, column x + e + 1; hi halves 16 rows up, 16 columns right.
//
//  Wider bands (W = 128, 256, 512 diagonals; DESIGN.md 4f) use the same layout with S = 8 and TP = W / 16 threads per
//  pair (32 / TP pairs per warp): thread u holds diagonals S*u + s and S*u + s + W/2, so a register's hi half is W/4 rows
//  up and W/4 columns right of its lo half and a selector pairs rows y and y - W/4.  The seam between diagonals W/2 - 1
//  and W/2 rides on the rotation between the last thread and thread 0 with the same two selectors.  A chunk reads rows
//  [Yc - W/4 + 1, Yc + 32) and columns [Xc, Xc + W/2 + 32) while the previous chunk's reads may still be in flight, so
//  the rings hold W/4 + 64 rows and W/2 + 64 columns (kBandRingFor).  The selectors of wide bands are refilled by the
//  guarded per-symbol path; the column tables keep the rolling window.
// =================================================================================================
// ring entries of a W-diagonal band: a power of two >= W/2 + 64 (128 for W = 64 and 128, 256 for 256, 512 for 512)
template <int W>
constexpr int kBandRingFor = W <= 128 ? kBandRing : (W <= 256 ? 256 : 512);

template <int S, int W = kBandWidth>
struct BandedWarpSmemS {
  // The pairs of a warp read the same ring offsets in the same instruction: pair g's rings start (g mod S/2) + 16 (g / (S/2))
  // words into their row, so that the 32 threads (offsets (S/2) u inside a pair) hit 32 different banks.  (From W = 256 on,
  // threads u and u + 8 of one pair read 32 words apart: 2-way, at W = 512 4-way conflicts that no offset removes.)
  static constexpr int kPairs = 32 * 2 * S / W, kRing = kBandRingFor<W>;
  uint32_t tab[kPairs][2 * kRing + 32];
  uint32_t sel[kPairs][2 * kRing + 32];
};

template <int MODE, int S, int W = kBandWidth>
SWB_HD void banded_warpS(const BandedParams& P, const WarpCtx& w, long long warp_id, long long num_warps, BandedWarpSmemS<S, W>* sm) {
  static_assert(S >= 4 && S <= 16 && (S & (S - 1)) == 0, "register sets per thread: 4, 8 or 16");
  static_assert(W == kBandWidth || (S == 8 && (W == 128 || W == 256 || W == 512)), "band width: 64, or 128 / 256 / 512 with S = 8");
  constexpr int TP = W / (2 * S), H2 = S / 2, G = 32 / TP;      // threads per pair, pairs per warp
  constexpr int Q = W / 4;                                      // rows up / columns right of a register's hi half
  constexpr int RING = kBandRingFor<W>;
  constexpr int PRE = Q > kChunk ? Q : kChunk;                  // rows below the first chunk the rings start with
  constexpr bool ROW_WINDOW = Q == 16;                          // rows y and y - 16 come from one 64-bit funnel
  const int lane = w.lane;
  const int u = lane & (TP - 1), grp = lane / TP;
  const int src_prev = grp * TP + ((u + TP - 1) & (TP - 1));   // even step: set 0's left neighbours come from thread u-1 (rotating)
  const int src_next = grp * TP + ((u + 1) & (TP - 1));        // odd step: set S-1's upper neighbours come from thread u+1 (rotating)
  const uint32_t nopen = pack2(-P.gap_init), next = pack2(-P.gap_ext);
  const uint32_t padb = (uint32_t)(P.mismatch + P.gap_init) & 0xFFu;
  const uint32_t padw = padb * 0x01010101u;
  const uint32_t flip = padb ^ ((uint32_t)(P.match + P.gap_init) & 0xFFu);
  const uint32_t padsel = mk_sel16(4u, 4u);
  // the seam between diagonal 31 and 32 rides on the rotation (prmt(x, nopen, sel): bytes 0-3 = x, 4-7 = nopen)
  const uint32_t sel_left = u == TP - 1 ? 0x1054u : 0x3210u;   // last thread -> thread 0: (border, its set S-1 lo = diagonal 31)
  const uint32_t sel_up = u == 0 ? 0x7632u : 0x3210u;          // thread 0 -> last thread: (its set 0 hi = diagonal 32, border)
  uint32_t* tab = sm->tab[grp] + (grp % H2) + 16 * (grp / H2);
  uint32_t* sel = sm->sel[grp] + (grp % H2) + 16 * (grp / H2);
  const long long ngroups = (P.npairs + G - 1) / G;
  const int tA0 = 2 - ((2 - P.band_lo) & 1);                             // first even-set anti-diagonal (see banded_warp)
  const int I0 = (tA0 - P.band_lo) / 2, J0 = (tA0 + P.band_lo) / 2;

  for (long long pg = warp_id; pg < ngroups; pg += num_warps) {
    const long long pair = pg * G + grp;
    const bool valid = pair < P.npairs;
    const int n = valid ? P.a_len[pair] : 0, m = valid ? P.b_len[pair] : 0;
    const uint64_t* aw = P.a_words + (valid ? pair : 0) * P.a_stride;
    const uint64_t* bw = P.b_words + (valid ? pair : 0) * P.b_stride;
    const int NH = (n > 0 && m > 0) ? (n + m - tA0) / 2 + 1 : 0;
    const int maxNH = w.reduce_max(NH);
    const int nchunks = (maxNH + kChunk - 1) / kChunk;

    uint32_t Ho[S], E[S], F[S];
#pragma unroll
    for (int k = 0; k < S; ++k) { Ho[k] = nopen; E[k] = nopen; F[k] = nopen; }
    uint32_t best = 0;

    // ---- rings (slot of row y: (y - Yc0) & (RING-1), of column x: (x - Xc0) & (RING-1) -- a chunk's 32 new entries
    // never wrap): everything pad, then selectors for rows [Yc0-PRE, Yc0) and tables for columns [Xc0, Xc0+W/2)
    const int Yc0 = I0 - 1, Xc0 = J0 - 1;                                  // thread 0's positions at h = 0
    w.sync();
    for (int k = u; k < 2 * RING; k += TP) { tab[k] = padw; sel[k] = padsel; }
    w.sync();
    for (int k = u; k < W / 2; k += TP) {
      if (k < PRE) {
        const int y = Yc0 - PRE + k;
        const uint32_t sv = mk_sel16(packed_code(bw, y, m), packed_code(bw, y - Q, m));
        sel[(RING - PRE) + k] = sv; sel[(RING - PRE) + k + RING] = sv;
      }
      const int x = Xc0 + k;
      const uint32_t tv = table_word(packed_code(aw, x, n), padw, flip);
      tab[k] = tv; tab[k + RING] = tv;
    }
    // Rolling 32-symbol windows of the packed sequences (64 bits each), so that a chunk whose new rows and columns lie
    // inside the sequences costs ONE 64-bit load per sequence, issued a chunk ahead, instead of 24 guarded ones per thread
    // (the refill was 39 % of this kernel's stall samples, most of them waiting for those loads):
    //   RA = rows [Yc-16, Yc+16) of the coming chunk, RN = the same for the chunk after it, TC = columns [Xc+W/2, Xc+W/2+32).
    // Word indices are clamped to the pair's words: a window that overlaps the outside holds garbage there and is not
    // used (such chunks take the guarded per-symbol path below).
    const int wr_i = (Yc0 - 16) >> 5, wr_sh = 2 * ((Yc0 - 16) & 31);
    const int wc_i = (Xc0 + W / 2) >> 5, wc_sh = 2 * ((Xc0 + W / 2) & 31);
    uint64_t RA, RN, r_last, TC, c_last;
    {
      const uint64_t r0 = packed_word(bw, P.b_stride, wr_i), r1 = packed_word(bw, P.b_stride, wr_i + 1);
      r_last = packed_word(bw, P.b_stride, wr_i + 2);
      RA = funnel64(r0, r1, wr_sh); RN = funnel64(r1, r_last, wr_sh);
      const uint64_t c0 = packed_word(aw, P.a_stride, wc_i);
      c_last = packed_word(aw, P.a_stride, wc_i + 1);
      TC = funnel64(c0, c_last, wc_sh);
    }
    const int su = 2 * H2 * u;                                             // W = 64: this thread's entries are k = H2 u + j + 16 i
                                                                           // (the offsets the step loop reads with: no bank conflicts)
    for (int c = 0; c < nchunks; ++c) {
      // ---- this chunk reads rows [Yc-Q, Yc+32) and columns [Xc, Xc+W/2+32): add rows [Yc, Yc+32), columns [Xc+W/2, Xc+W/2+32)
      const int Yc = Yc0 + c * kChunk, Xc = Xc0 + c * kChunk;
      const uint64_t r_new = packed_word(bw, P.b_stride, wr_i + c + 3);    // consumed at the end of the chunk
      const uint64_t c_new = packed_word(aw, P.a_stride, wc_i + c + 2);
      uint32_t* const selw = sel + ((c * kChunk) & (RING - 1));
      uint32_t* const tabw = tab + ((c * kChunk + W / 2) & (RING - 1));
      if (ROW_WINDOW && Yc >= 16 && Yc + kChunk <= m) {
        const uint32_t a_lo = (uint32_t)RA, b_lo = (uint32_t)(RA >> 32), b_hi = (uint32_t)RN;   // rows y - 16: RA; rows y: RA.hi, RN.lo
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const uint32_t wb = (i ? b_hi : b_lo) >> su, wa = (i ? b_lo : a_lo) >> su;
#pragma unroll
          for (int j = 0; j < H2; ++j) {
            const uint32_t sv = 0xC480u + ((wb >> (2 * j)) & 3u) * 0x11u + ((wa >> (2 * j)) & 3u) * 0x1100u;   // = mk_sel16 of two real codes
            selw[H2 * u + j + 16 * i] = sv; selw[H2 * u + j + 16 * i + RING] = sv;
          }
        }
      } else {
        for (int k = u; k < kChunk; k += TP) {
          const int y = Yc + k;
          const uint32_t sv = mk_sel16(packed_code(bw, y, m), packed_code(bw, y - Q, m));
          selw[k] = sv; selw[k + RING] = sv;
        }
      }
      if (Xc + W / 2 >= 0 && Xc + W / 2 + kChunk <= n) {
        if constexpr (ROW_WINDOW) {
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const uint32_t wt = (i ? (uint32_t)(TC >> 32) : (uint32_t)TC) >> su;
#pragma unroll
            for (int j = 0; j < H2; ++j) {
              const uint32_t tv = padw ^ (flip << (8u * ((wt >> (2 * j)) & 3u)));
              tabw[H2 * u + j + 16 * i] = tv; tabw[H2 * u + j + 16 * i + RING] = tv;
            }
          }
        } else {                                                           // W > 64: 32 / TP consecutive entries a thread
#pragma unroll
          for (int j = 0; j < kChunk / TP; ++j) {
            const int k = (kChunk / TP) * u + j;
            const uint32_t tv = padw ^ (flip << (8u * ((uint32_t)(TC >> (2 * k)) & 3u)));
            tabw[k] = tv; tabw[k + RING] = tv;
          }
        }
      } else {
        for (int k = u; k < kChunk; k += TP) {
          const int x = Xc + W / 2 + k;
          const uint32_t tv = table_word(packed_code(aw, x, n), padw, flip);
          tabw[k] = tv; tabw[k + RING] = tv;
        }
      }
      RA = RN; RN = funnel64(r_last, r_new, wr_sh); r_last = r_new;
      TC = funnel64(c_last, c_new, wc_sh); c_last = c_new;
      w.sync();
      // ring windows of this thread: selp[h] = selector of row y (read back to -(S/2 - 1)); tabp[h] = table of column x
      const uint32_t* selp = sel + ((c * kChunk - H2 * u - (H2 - 1)) & (RING - 1)) + (H2 - 1);
      const uint32_t* tabp = tab + ((c * kChunk + H2 * u) & (RING - 1));
      uint32_t a[H2 + 1], b[H2 + 1], sv[H2];        // columns x .. x + S/2 (and Q further right), rows y .. y - S/2 + 1
#pragma unroll
      for (int e = 0; e < H2; ++e) { a[e] = tabp[e]; b[e] = tabp[e + Q]; }
#pragma unroll
      for (int e = 1; e < H2; ++e) sv[e] = selp[-e];
#pragma unroll (2)
      for (int h = 0; h < kChunk; ++h) {
        sv[0] = selp[h];
        a[H2] = tabp[h + H2]; b[H2] = tabp[h + H2 + Q];
        uint32_t sub[S];
#pragma unroll
        for (int e = 0; e < H2; ++e) {
          sub[2 * e] = prmt(a[e], b[e], sv[e]);                 // set 2e:   row y - e, column x + e
          sub[2 * e + 1] = prmt(a[e + 1], b[e + 1], sv[e]);     // set 2e+1: row y - e, column x + e + 1
        }
#pragma unroll
        for (int e = 0; e < H2; ++e) { a[e] = a[e + 1]; b[e] = b[e + 1]; }
#pragma unroll
        for (int e = H2 - 1; e >= 1; --e) sv[e] = sv[e - 1];
        // ---------------- even anti-diagonal: sets 2e (left = set 2e-1, for e = 0 thread u-1's set S-1; up = set 2e+1)
        {
          const uint32_t leftHo0 = w.shfl(prmt(Ho[S - 1], nopen, sel_left), src_prev);
          uint32_t leftE0 = 0;
          if (MODE == 0) leftE0 = w.shfl(prmt(E[S - 1], nopen, sel_left), src_prev);
          uint32_t hv[H2];
#pragma unroll
          for (int e = 0; e < H2; ++e) {
            const int k = 2 * e;
            const uint32_t lHo = e == 0 ? leftHo0 : Ho[k - 1];
            if (MODE == 0) {
              const uint32_t lE = e == 0 ? leftE0 : E[k - 1];
              const uint32_t En = addmax16x2(lE, next, lHo), Fn = addmax16x2(F[k + 1], next, Ho[k + 1]);
              hv[e] = max3relu16x2(add16x2(Ho[k], sub[k]), En, Fn);
              E[k] = En; F[k] = Fn;
            } else {
              hv[e] = max16x2(addmaxrelu16x2(Ho[k], sub[k], lHo), Ho[k + 1]);
            }
          }
#pragma unroll
          for (int e = 0; e < H2; ++e) Ho[2 * e] = add16x2(hv[e], nopen);
#pragma unroll
          for (int e = 0; e < H2; e += 2) best = max3_16x2(best, hv[e], hv[e + 1]);
        }
        // ---------------- odd anti-diagonal: sets 2e+1 (left = set 2e; up = set 2e+2, for the last one thread u+1's set 0)
        {
          const uint32_t upHoL = w.shfl(prmt(Ho[0], nopen, sel_up), src_next);
          uint32_t upFL = 0;
          if (MODE == 0) upFL = w.shfl(prmt(F[0], nopen, sel_up), src_next);
          uint32_t hv[H2];
#pragma unroll
          for (int e = 0; e < H2; ++e) {
            const int k = 2 * e + 1;
            const uint32_t uHo = k == S - 1 ? upHoL : Ho[k + 1 < S ? k + 1 : 0];
            if (MODE == 0) {
              const uint32_t uF = k == S - 1 ? upFL : F[k + 1 < S ? k + 1 : 0];
              const uint32_t En = addmax16x2(E[k - 1], next, Ho[k - 1]), Fn = addmax16x2(uF, next, uHo);
              hv[e] = max3relu16x2(add16x2(Ho[k], sub[k]), En, Fn);
              E[k] = En; F[k] = Fn;
            } else {
              hv[e] = max16x2(addmaxrelu16x2(Ho[k], sub[k], Ho[k - 1]), uHo);
            }
          }
#pragma unroll
          for (int e = 0; e < H2; ++e) Ho[2 * e + 1] = add16x2(hv[e], nopen);
#pragma unroll
          for (int e = 0; e < H2; e += 2) best = max3_16x2(best, hv[e], hv[e + 1]);
        }
      }
    }
    int mx = (int)(short)(best & 0xFFFFu), mh = (int)(short)(best >> 16);
    mx = mx > mh ? mx : mh;
#pragma unroll
    for (int d = 1; d < TP; d <<= 1) {
      const int o = (int)w.shfl((uint32_t)mx, lane ^ d);
      mx = mx > o ? mx : o;
    }
    if (valid && u == 0) P.scores[pair] = mx;
  }
}

#ifdef __CUDACC__
template <int MODE>
__global__ void __launch_bounds__(64, 6) sw_banded4_kernel(const __grid_constant__ BandedParams P) {
  __shared__ BandedWarpSmemS<8> sm[2];
  WarpCtx w{(int)(threadIdx.x & 31)};
  const int wi = (int)(threadIdx.x >> 5);
  banded_warpS<MODE, 8>(P, w, (long long)blockIdx.x * 2 + wi, (long long)gridDim.x * 2, &sm[wi]);
}
#endif

const void* banded4_kernel(int mode);

#ifdef __CUDACC__
// Two threads per pair with sixteen register sets each (sixteen pairs per warp, one warp per CTA: the rings of sixteen
// pairs are 36 KB of shared memory).  Half the shuffles, border PRMTs and ring loads per cell of the layout above.
template <int MODE>
__global__ void __launch_bounds__(32, 6) sw_banded2_kernel(const __grid_constant__ BandedParams P) {
  __shared__ BandedWarpSmemS<16> sm;
  WarpCtx w{(int)(threadIdx.x & 31)};
  banded_warpS<MODE, 16>(P, w, (long long)blockIdx.x, (long long)gridDim.x, &sm);
}
#endif

const void* banded2_kernel(int mode);

#ifdef __CUDACC__
// Bands of W = 128, 256 or 512 diagonals: W / 16 threads per pair with eight register sets each, 1024 / W pairs per CTA.
template <int MODE, int W>
__global__ void __launch_bounds__(64, 6) sw_banded_wide_kernel(const __grid_constant__ BandedParams P) {
  __shared__ BandedWarpSmemS<8, W> sm[2];
  WarpCtx w{(int)(threadIdx.x & 31)};
  const int wi = (int)(threadIdx.x >> 5);
  banded_warpS<MODE, 8, W>(P, w, (long long)blockIdx.x * 2 + wi, (long long)gridDim.x * 2, &sm[wi]);
}
#endif

const void* banded_wide_kernel(int mode, int width);   // null for a width without a kernel

}  // namespace swb
