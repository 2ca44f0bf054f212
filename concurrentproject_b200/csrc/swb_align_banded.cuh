// swb_align_banded.cuh -- score, span and CIGAR for every pair of a banded batch (swb200_align_banded_batch,
// swb200_batch_align_banded): the best local alignment all of whose cells lie in the band B, band_lo <= j - i <= band_hi
// (W = 64 K diagonals, K = 1, 2, 4 or 8; i is the row in seq2, j the column in seq1).
//
// One warp per pair.  A 10 kb pair's direction nibbles take ~16 B x (len1 + len2) = 320 KB, so a thread per pair (as in
// swb_align_batch.cuh) would need gigabytes in flight; a warp needs 32x less, and its storage grows with the resident
// warps, never with the batch.  Lane l owns diagonals lo + 2l and lo + 2l + 1 (32-bit values, no packing).  The sweep
// runs over anti-diagonals t = i + j; on each one exactly one of a lane's two diagonals has a cell (the first one when
// t - lo is even), so every lane computes one cell per step.  A cell's upper neighbour is diagonal k + 1 and its left
// neighbour diagonal k - 1, both on the previous anti-diagonal: on an even step the upper one is the lane's own second
// register and the left one lane l-1's second register (one shfl for H, one for E); on an odd step the left one is the
// lane's own first register and the upper one lane l+1's first register (H and F).  The diagonal neighbour is the
// cell's own register of two steps ago.  This is the geometry of swb_banded.cuh, in 32-bit lanes.
//
// Wider bands (K > 1, DESIGN.md 4f): lane l owns the 2K consecutive diagonals lo + 2Kl .. lo + 2Kl + 2K - 1, of which K
// have a cell on each anti-diagonal.  Neighbours inside the lane stay in registers; only the lane's outer diagonals use
// the two shfls above.  A lane writes K nibbles per anti-diagonal, so one direction word holds 8 / K anti-diagonals.
//
//   pass 1  local recurrence over the pair, band lo = band_lo: the end cell (max H, then the smallest j, then the
//           smallest i; out-of-band cells are H = E = F = 0, as in oracle_gotoh_banded);
//   pass 2  anchored recurrence over the reversed prefixes seq1[..j_end], seq2[..i_end] in the mirrored band
//           lo' = (j_end - i_end) - band_hi (cells outside it are unreachable): its maximum is the score again and
//           sits at the start cell (the largest j_start, then the largest i_start);
//   pass 3  anchored recurrence over the span rectangle in the band lo'' = band_lo - (j_start - i_start), writing one
//           nibble per lane per anti-diagonal exactly as align_dp does (diagonal before E before F; a gap counts as
//           extended only where extending is strictly better than opening): every 8 anti-diagonals each lane stores a
//           32-bit word, one coalesced 128-byte line per warp.  Then one lane walks back from the rectangle's last cell
//           while the warp stages blocks of lines through shared memory ahead of it (the walk only moves to lower
//           anti-diagonals), run-length encodes, splits '=' / 'X' and re-scores with main.cpp's costs.
//
// Passes 1 + 2 are one kernel, pass 3 + walk another: each warp owns a fixed direction slot; a span larger than the slot
// takes a piece of the shared pool (one atomic add) or goes to the pending list for the next round (swb200.cu runs the
// rounds of both batch alignments the same way).  Error bits, op codes and the '1I1I' split when gap_ext > gap_init are
// those of swb_align_batch.cuh.  Everything per pair is SWB_HD on a WarpCtx, so tests/emu/align_banded_emu.cu runs the
// same bodies with one pthread per lane.
#pragma once
#include "swb_align_batch.cuh"

namespace swb {

constexpr int kBandAlignWarps = 4;          // warps per CTA
constexpr int kBandStageLines = 32;         // direction lines (8 anti-diagonals x 32 lanes each) the walk has staged

struct AlignBandedParams {
  const uint64_t* a_words;   // seq1 (columns j), 2-bit packed: a batch packed with keep_order = 1 (q = seq1, t = seq2)
  const uint64_t* b_words;   // seq2 (rows i)
  const int* a_len;
  const int* b_len;
  long long a_stride, b_stride;
  long long npairs;
  int band_lo;               // the band is band_lo <= j - i <= band_lo + 64 K - 1 (K: the kernels' template argument)
  int match, mismatch, gap_init, gap_ext;
  int* scores;               // per pair
  int* spans;                // per pair {i_start, j_start, i_end, j_end}, 1-based
  long long nwarps;          // warps of the first launch (the stride of the pair loop; slot w belongs to warp w)
  // pass 3
  uint32_t* slot;            // slot_words 32-bit words per warp, warp w's at slot + w * slot_words
  long long slot_words;
  uint32_t* pool;            // shared pool for spans larger than a slot
  long long pool_words;
  unsigned long long* pool_used;
  const int* todo;           // pairs to trace (null: 0 .. ntodo-1)
  long long ntodo;
  int* pending;              // pairs the pool could not take this round
  int* npending;
  uint32_t* ops;             // ops_stride words per pair
  int ops_stride;
  int* ops_count;            // per pair: number of operations, -(number) if more than ops_stride
  int* err;                  // kAlignErr* bits
  unsigned long long* cells; // in-band cells the passes computed (one atomic add per lane and launch)
};

// 32-bit direction words a lx x ly span takes: one line of 32 words per 8 / K anti-diagonals t = 0 .. lx + ly
template <int K = 1>
SWB_HD long long band_dir_words(int lx, int ly) { return 32LL * (((long long)lx + ly) / (8 / K) + 1); }

// the end / start cell's tie rule: the larger H; among equal H > 0 the smaller x (j), then the smaller y (i)
SWB_HD bool band_better(int h, int x, int y, int bh, int bx, int by) {
  return h > bh || (h == bh && h > 0 && (x < bx || (x == bx && y < by)));
}

// One recurrence over X (columns x = 1..X.len) x Y (rows y = 1..Y.len), restricted to the 64 K diagonals
// lo <= x - y <= lo + 64 K - 1; the same result in every lane.
//   MODE 0: local, returns the maximum and its cell;  MODE 1: anchored from (0, 0) (which must lie in the band), the same;
//   MODE 2: anchored with direction nibbles into dirs (band_dir_words<K>(X.len, Y.len) words), returns H at (X.len, Y.len).
// *cells += the in-band cells of the rectangle this lane computed.
template <int MODE, int K = 1>
SWB_HD int band_dp(const AlignBandedParams& P, const WarpCtx& w, const AlignSeq& X, const AlignSeq& Y, int lo, uint32_t* dirs,
                   int* bx, int* by, long long* cells) {
  constexpr bool ANCH = MODE >= 1, DIRS = MODE == 2;
  const int nx = X.len, ny = Y.len, lane = w.lane;
  const int gi = P.gap_init, ge = P.gap_ext, gmin = gi < ge ? gi : ge;
  const int ma = P.match, mi = P.mismatch;
  constexpr int W = 64 * K, TW = 8 / K, TWS = K == 1 ? 3 : (K == 2 ? 2 : (K == 4 ? 1 : 0));   // TW = 2^TWS anti-diagonals a word, 2K = 2^(4-TWS)
  const int OUT = ANCH ? kAlignNeg : 0;          // H, E, F outside the band or the rectangle (anchored: borders aside)
  *bx = 0; *by = 0;
  // the diagonals that have cells, and the anti-diagonals t0 .. t1 they span
  const int klo = lo > 1 - ny ? lo : 1 - ny, khi = lo + (W - 1) < nx - 1 ? lo + (W - 1) : nx - 1;
  if (nx <= 0 || ny <= 0 || klo > khi) return 0;
  const int t0 = 2 + (klo > 0 ? klo : (khi < 0 ? -khi : 0));
  const int kc = nx - ny < klo ? klo : (nx - ny > khi ? khi : nx - ny);
  const int t1 = nx + ny - (nx - ny - kc > 0 ? nx - ny - kc : kc - (nx - ny));
  const int kA = lo + 2 * K * lane;              // this lane's first diagonal; kA + 2K - 1 its last
  const int up_src = (lane + 1) & 31, left_src = (lane + 31) & 31;
  // diagonal kA + q in hv[q], ev[q], fv[q]
  int hv[2 * K], ev[2 * K], fv[2 * K];
#pragma unroll
  for (int q = 0; q < 2 * K; ++q) { hv[q] = OUT; ev[q] = OUT; fv[q] = OUT; }
  int best = 0, bxx = 0, byy = 0;
  long long nc = 0;
  uint32_t dword = 0;
  // two steps before t0 every cell is a border cell or outside: the registers hold correct neighbours from then on
  for (int t = t0 - 2; t <= t1; ++t) {
    const bool odd = ((t - lo) & 1) != 0;
    const int nh = (int)w.shfl((uint32_t)(odd ? hv[0] : hv[2 * K - 1]), odd ? up_src : left_src);
    const int ng = (int)w.shfl((uint32_t)(odd ? fv[0] : ev[2 * K - 1]), odd ? up_src : left_src);
    const bool edge = odd ? lane == 31 : lane == 0;          // diagonal lo + W / lo - 1: outside the band
    const int xh = edge ? OUT : nh, xg = edge ? OUT : ng;
    int hn[K], en[K], fn[K];
    uint32_t nib = 0;
#pragma unroll
    for (int c = 0; c < K; ++c) {
      // the cell on diagonal kA + q, q = 2c + odd: left = q - 1, up = q + 1 (both of the previous step), diagonal = q itself
      const int qa = 2 * c, qb = 2 * c + 1;
      const int lh = odd ? hv[qa] : (c == 0 ? xh : hv[c == 0 ? 0 : qa - 1]);          // left (y, x-1)
      const int lg = odd ? ev[qa] : (c == 0 ? xg : ev[c == 0 ? 0 : qa - 1]);
      const int uh = odd ? (c == K - 1 ? xh : hv[c == K - 1 ? 0 : qb + 1]) : hv[qb];  // up (y-1, x)
      const int ug = odd ? (c == K - 1 ? xg : fv[c == K - 1 ? 0 : qb + 1]) : fv[qb];
      const int dh = odd ? hv[qb] : hv[qa];                                           // diagonal (y-1, x-1)
      const int k = kA + (odd ? qb : qa);
      const int x = (t + k) >> 1, y = (t - k) >> 1;            // t + k is even
      const bool in = x >= 1 && x <= nx && y >= 1 && y <= ny;
      const int s = align_code(X, in ? x - 1 : 0) == align_code(Y, in ? y - 1 : 0) ? ma : mi;
      const int e_ext = lg - ge, e_open = lh - gi, f_ext = ug - ge, f_open = uh - gi;
      int e = imax2(e_ext, e_open), f = imax2(f_ext, f_open);
      const int d = dh + s;
      int h = imax2(d, imax2(e, f));
      if (!ANCH) h = imax2(h, 0);
      if (!in) {
        e = OUT; f = OUT; h = OUT;
        if (ANCH && x >= 0 && y >= 0 && (x == 0 || y == 0)) h = x + y == 0 ? 0 : -(gi + (x + y - 1) * gmin);
      }
      nc += in ? 1 : 0;
      if (DIRS) {
        const uint32_t src = h == d ? 0u : (h == e ? 1u : 2u);
        nib |= (src | (e_ext > e_open ? 4u : 0u) | (f_ext > f_open ? 8u : 0u)) << (4 * c);
      } else if (in && band_better(h, x, y, best, bxx, byy)) {
        best = h; bxx = x; byy = y;
      }
      hn[c] = h; en[c] = e; fn[c] = f;
    }
    if (DIRS) {
      dword |= nib << (4 * K * (t & (TW - 1)));
      if ((t & (TW - 1)) == TW - 1 || t == t1) { dirs[(long long)(t >> TWS) * 32 + lane] = dword; dword = 0; }
    }
#pragma unroll
    for (int c = 0; c < K; ++c) {
      if (odd) { hv[2 * c + 1] = hn[c]; ev[2 * c + 1] = en[c]; fv[2 * c + 1] = fn[c]; }
      else { hv[2 * c] = hn[c]; ev[2 * c] = en[c]; fv[2 * c] = fn[c]; }
    }
  }
  *cells += nc;
  if constexpr (DIRS) {
    // H(nx, ny) is the last cell of diagonal nx - ny, computed at t1 = nx + ny
    const int kl = nx - ny - lo, q = kl & (2 * K - 1);
    int hq = hv[0];
#pragma unroll
    for (int r = 1; r < 2 * K; ++r) hq = q == r ? hv[r] : hq;
    return (int)w.shfl((uint32_t)hq, kl >> (4 - TWS));
  } else {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int oh = (int)w.shfl((uint32_t)best, lane ^ o), ox = (int)w.shfl((uint32_t)bxx, lane ^ o);
      const int oy = (int)w.shfl((uint32_t)byy, lane ^ o);
      if (band_better(oh, ox, oy, best, bxx, byy)) { best = oh; bxx = ox; byy = oy; }
    }
    *bx = bxx; *by = byy;
    return best;
  }
}

// Passes 1 and 2 for pair k: score and span.  Returns this lane's in-band cells.
template <int K = 1>
SWB_HD long long band_span_pair(const AlignBandedParams& P, const WarpCtx& w, long long k) {
  const int n = P.a_len[k], m = P.b_len[k];
  const uint64_t* aw = P.a_words + k * P.a_stride;
  const uint64_t* bw = P.b_words + k * P.b_stride;
  long long nc = 0;
  int je = 0, ie = 0, rj = 0, ri = 0;
  const int s = band_dp<0, K>(P, w, AlignSeq{aw, 0, n, false}, AlignSeq{bw, 0, m, false}, P.band_lo, nullptr, &je, &ie, &nc);
  int s2 = s;
  if (s > 0)
    s2 = band_dp<1, K>(P, w, AlignSeq{aw, 0, je, true}, AlignSeq{bw, 0, ie, true}, (je - ie) - (P.band_lo + (64 * K - 1)), nullptr,
                       &rj, &ri, &nc);
  if (w.lane == 0) {
    int* span = P.spans + 4 * k;
    P.scores[k] = s;
    const bool ok = s > 0 && s2 == s;
    span[0] = ok ? ie - ri + 1 : 0; span[1] = ok ? je - rj + 1 : 0; span[2] = ok ? ie : 0; span[3] = ok ? je : 0;
    if (s2 != s) atomic_or_i32(P.err, kAlignErrStart);
  }
  return nc;
}

// The run-length encoder of the warp walks (band_walk, long_walk).  Operations arrive last-first; WRITE = false counts
// them and re-scores, WRITE = true stores them first-first (ops[n - 1 - t]).  tot sums main.cpp's costs of the runs.
// emit(..., opened = true) for a gap that was opened ends its run when gap_ext > gap_init (two gaps, not one extended).
template <bool WRITE>
struct OpEncoder {
  int match, mismatch, gap_init, gap_ext;
  uint32_t* ops;
  int n;
  int nops = 0, run = 0;
  uint32_t cur = 0;
  bool brk = false;
  long long tot = 0;
  SWB_HD void flush() {
    if (run <= 0) return;
    if (cur == kOpEq) tot += (long long)run * match;
    else if (cur == kOpX) tot += (long long)run * mismatch;
    else tot -= gap_init + (long long)(run - 1) * gap_ext;
    if (WRITE) ops[n - 1 - nops] = ((uint32_t)run << 4) | cur;
    ++nops;
  }
  SWB_HD void emit(uint32_t op, int cnt, bool opened = false) {
    if (op == cur && !brk) run += cnt;
    else { flush(); cur = op; run = cnt; }
    brk = opened && gap_ext > gap_init;
  }
};

// The walk over the direction lines of a span (band lo, X / Y as pass 3 saw them) from its last cell back to (0, 0).
// Lane 0 walks; before it runs out of staged lines the warp copies the next kBandStageLines lines below into stage.
// Operations come out last-first (OpEncoder).  Returns the count and *total in every lane; a step out of the band
// poisons *total.
template <bool WRITE, int K = 1>
SWB_HD int band_walk(const AlignBandedParams& P, const WarpCtx& w, const uint32_t* dirs, const AlignSeq& X, const AlignSeq& Y,
                     int lo, uint32_t* stage, int n, uint32_t* ops, int* total) {
  constexpr int TWS = K == 1 ? 3 : (K == 2 ? 2 : (K == 4 ? 1 : 0));   // a direction line holds 2^TWS = 8 / K anti-diagonals
  const int lane = w.lane;
  int x = X.len, y = Y.len, state = 0;
  bool outside = false;
  OpEncoder<WRITE> enc{P.match, P.mismatch, P.gap_init, P.gap_ext, ops, n};
  for (;;) {
    const int top = (int)w.shfl((uint32_t)((x + y) >> TWS), 0);
    const int base = top - kBandStageLines + 1 > 0 ? top - kBandStageLines + 1 : 0;
    w.sync();
    for (int q = 0; q < kBandStageLines && base + q <= top; ++q) stage[q * 32 + lane] = dirs[(long long)(base + q) * 32 + lane];
    w.sync();
    int done = 1;
    if (lane == 0) {
      while (x > 0 && y > 0) {
        const int t = x + y;
        if ((t >> TWS) < base) break;
        const unsigned kl = (unsigned)(x - y - lo);
        if (kl > 64u * K - 1) { outside = true; break; }
        // lane kl / 2K, nibble K (t mod 8/K) + (kl mod 2K) / 2
        const uint32_t nib = K * (t & ((1 << TWS) - 1)) + ((kl & (2 * K - 1)) >> 1);
        const uint32_t d = (stage[((t >> TWS) - base) * 32 + (int)(kl >> (4 - TWS))] >> (4 * nib)) & 0xFu;
        if (state == 0) {
          const uint32_t src = d & 3u;
          if (src == 0) { enc.emit(align_code(X, x - 1) == align_code(Y, y - 1) ? kOpEq : kOpX, 1); --x; --y; }
          else state = (int)src;
        } else if (state == 1) {                   // E: a base of seq1 against a gap
          const bool opened = !(d & 4u);
          enc.emit(kOpIns, 1, opened);
          state = opened ? 0 : 1;
          --x;
        } else {                                   // F: a base of seq2 against a gap
          const bool opened = !(d & 8u);
          enc.emit(kOpDel, 1, opened);
          state = opened ? 0 : 2;
          --y;
        }
      }
      done = outside || !(x > 0 && y > 0);
    }
    if (w.shfl((uint32_t)done, 0)) break;
  }
  int tl = 0;
  if (lane == 0) {
    // the rest runs along row 0 or column 0 of the span: leading gaps, in the band because (0, 0) and (x, y) are
    if (x > 0) enc.emit(kOpIns, x);
    if (y > 0) enc.emit(kOpDel, y);
    enc.flush();
    tl = outside ? kAlignNeg : (int)enc.tot;
  }
  *total = (int)w.shfl((uint32_t)tl, 0);
  return (int)w.shfl((uint32_t)enc.nops, 0);
}

// Pass 3 and the walk for pair k (score and span from band_span_pair).  Returns this lane's in-band cells, or -1 if the
// pair must wait for the next round (pool exhausted).
template <int K = 1>
SWB_HD long long band_trace_pair(const AlignBandedParams& P, const WarpCtx& w, long long k, long long warp, uint32_t* stage) {
  const int s = P.scores[k];
  if (s <= 0) { if (w.lane == 0) P.ops_count[k] = 0; return 0; }
  const int* span = P.spans + 4 * k;
  const int is = span[0], js = span[1], ie = span[2], je = span[3];
  const int lx = je - js + 1, ly = ie - is + 1, lo = P.band_lo - (js - is);
  const long long words = band_dir_words<K>(lx, ly);
  uint32_t* dirs;
  if (words <= P.slot_words) {
    dirs = P.slot + warp * P.slot_words;
  } else {
    unsigned long long at = 0;
    if (w.lane == 0) at = align_atomic_add(P.pool_used, (unsigned long long)words);
    at = (unsigned long long)w.shfl((uint32_t)at, 0) | ((unsigned long long)w.shfl((uint32_t)(at >> 32), 0) << 32);
    if ((long long)at + words > P.pool_words) {
      if (w.lane == 0) P.pending[align_atomic_inc(P.npending)] = (int)k;
      return -1;
    }
    dirs = P.pool + at;
  }
  const AlignSeq X{P.a_words + k * P.a_stride, js - 1, lx, false}, Y{P.b_words + k * P.b_stride, is - 1, ly, false};
  long long nc = 0;
  int unused0 = 0, unused1 = 0;
  const int h = band_dp<2, K>(P, w, X, Y, lo, dirs, &unused0, &unused1, &nc);
  if (h != s) {
    if (w.lane == 0) { atomic_or_i32(P.err, kAlignErrTrace); P.ops_count[k] = 0; }
    return nc;
  }
  int total = 0;
  const int n = band_walk<false, K>(P, w, dirs, X, Y, lo, stage, 0, nullptr, &total);
  if (total != s) {
    if (w.lane == 0) { atomic_or_i32(P.err, kAlignErrRescore); P.ops_count[k] = 0; }
    return nc;
  }
  if (n > P.ops_stride) { if (w.lane == 0) P.ops_count[k] = -n; return nc; }
  band_walk<true, K>(P, w, dirs, X, Y, lo, stage, n, P.ops + k * (long long)P.ops_stride, &total);
  if (w.lane == 0) P.ops_count[k] = n;
  return nc;
}

#if defined(__CUDACC__) && defined(SWB_ALIGN_BANDED_KERNELS)   // defined in swb_align_banded.cu only: one definition
template <int K>
__global__ void __launch_bounds__(32 * kBandAlignWarps) align_banded_span_kernel(const __grid_constant__ AlignBandedParams P) {
  const WarpCtx w{(int)(threadIdx.x & 31)};
  const long long warp = (long long)blockIdx.x * kBandAlignWarps + threadIdx.x / 32;
  long long cells = 0;
  for (long long k = warp; k < P.npairs; k += P.nwarps) cells += band_span_pair<K>(P, w, k);
  if (cells) atomicAdd(P.cells, (unsigned long long)cells);
}
// __maxnreg__: without a register limit ptxas gives K = 2 64 registers and 20 bytes of spills
template <int K>
__global__ void __launch_bounds__(32 * kBandAlignWarps) __maxnreg__(K == 2 ? 128 : 255) align_banded_trace_kernel(const __grid_constant__ AlignBandedParams P) {
  __shared__ uint32_t stage[kBandAlignWarps][kBandStageLines * 32];
  const WarpCtx w{(int)(threadIdx.x & 31)};
  const long long warp = (long long)blockIdx.x * kBandAlignWarps + threadIdx.x / 32;
  long long cells = 0;
  for (long long t = warp; t < P.ntodo; t += P.nwarps) {
    const long long c = band_trace_pair<K>(P, w, P.todo ? P.todo[t] : t, warp, stage[threadIdx.x / 32]);
    cells += c > 0 ? c : 0;
  }
  if (cells) atomicAdd(P.cells, (unsigned long long)cells);
}
#endif

// host launchers (swb_align_banded.cu) for K = 1, 2, 4, 8; blocks x kBandAlignWarps warps must not exceed P.nwarps
void launch_align_banded_span(const AlignBandedParams& P, int K, int blocks, cudaStream_t s);
void launch_align_banded_trace(const AlignBandedParams& P, int K, int blocks, cudaStream_t s);
const void* align_banded_trace_kernel_ptr(int K);

}  // namespace swb
