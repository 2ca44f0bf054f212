// swb_align_batch.cuh -- score, span and CIGAR for every pair of a batch (swb200_align_batch, swb200_batch_align).
//
// One thread per pair.  A read pair is small (150 x 1000 cells), so a thread can afford the whole pair, and a warp then
// holds 32 independent pairs: no shuffles, no barriers, no hand-off between lanes.  The pair is read from the packed
// batch (swb_batch.cuh: the shorter sequence is Q, the longer T, both 2-bit).  Inside a pass the thread sweeps strips of
// kAlignStrip columns of T, one strip in registers, down all rows of Q; the left boundary of the strip (H and the gap
// along T, per Q row) lives in a per-thread column buffer in HBM, interleaved over threads so that a warp whose pairs have
// equal shapes reads and writes it coalesced.  32-bit arithmetic throughout.
//
//   pass 1  local recurrence of main.cpp:57-63 over the pair, tracking the end cell (max H, then the smallest position in
//           seq1, then the smallest in seq2 -- oracle_gotoh_end's rule, in seq1/seq2 terms whichever sequence is Q);
//   pass 2  the anchored recurrence over the reversed prefixes that end at the end cell; its maximum is the score again and
//           sits at the start cell (oracle_gotoh_span);
//   pass 3  the anchored recurrence over the span rectangle, recording 4 bits per cell exactly as engine_warp_s32 with
//           DIRS does (source of H: diagonal before E before F; E / F extended only where strictly better than opening);
//           then the walk back from the rectangle's last cell, run-length encoding, '=' / 'X' split and the re-score with
//           main.cpp's costs, all in the same thread.
//
// Passes 1 + 2 are one kernel (align_span_kernel); pass 3 + walk another (align_trace_kernel), because the direction
// nibbles need storage whose size only the spans tell: each thread owns a fixed slot (slot_words 64-bit words, interleaved
// like the column buffer) that is reused for every pair it handles; a pair whose rectangle needs more takes a piece of a
// shared pool (one atomic add); a pair that finds the pool exhausted goes to a pending list that the host runs again with
// the pool emptied.  The first taker of an empty pool always fits (the pool is at least the largest rectangle).
//
// Ties and gap accounting are those of swb200_align.  One refinement: when gap_ext > gap_init the recurrence never extends
// a gap (opening again is cheaper), so two neighbouring gap characters are two gaps; they are then reported as two
// operations ("1I1I"), which re-score to the score with main.cpp's costs.  For gap_ext <= gap_init the operations are
// exactly swb200_align's.
//
// Every function that runs per pair is SWB_HD, so tests/emu/align_batch_emu.cu runs the same bodies on CPU threads.
#pragma once
#include "swb_device.cuh"

namespace swb {

constexpr int kAlignStrip = 16;                 // T columns per register strip: 16 nibbles = one 64-bit direction word
constexpr int kAlignNeg = -(1 << 29);           // "minus infinity" of the anchored borders (no s32 overflow)

// ops: count << 4 | op, BAM numbering
constexpr uint32_t kOpIns = 1, kOpDel = 2, kOpEq = 7, kOpX = 8;

// error bits (AlignBatchParams::err)
constexpr int kAlignErrStart = 1;               // pass 2 did not reproduce the score
constexpr int kAlignErrTrace = 2;               // pass 3 did not reproduce the score at the rectangle's last cell
constexpr int kAlignErrRescore = 4;             // the walked alignment does not re-score to the score

struct AlignBatchParams {
  const uint64_t* q_words;   // packed batch (swb_batch.cuh BatchParams): Q = the shorter sequence
  const uint64_t* t_words;
  const int* q_len;
  const int* t_len;
  const int* len1;           // the caller's seq1 lengths: pair k was swapped (Q = seq2) iff len1[k] != q_len[k]
  long long q_stride, t_stride;
  long long npairs;
  int match, mismatch, gap_init, gap_ext;
  int* scores;               // per pair
  int* spans;                // per pair {i_start, j_start, i_end, j_end}, 1-based, i in seq2, j in seq1
  int2* col;                 // column buffer: (max_short + 1) entries per thread, entry y of thread t at col[y * nthreads + t]
  long long nthreads;        // threads of the launch (the interleave stride of col and slot)
  // pass 3
  uint64_t* slot;            // slot_words per thread, word w of thread t at slot[w * nthreads + t]
  long long slot_words;
  uint64_t* pool;            // shared pool for rectangles larger than a slot
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
  unsigned long long* cells; // cells the passes computed (one atomic add per thread and launch)
  // the long-pair kernels (swb_align_long.cuh) only: col is one boundary row of row_stride entries per launched warp,
  // warp w's at col + w * row_stride, slot_words counts per warp, and warps draw pairs from the counter *next
  long long row_stride;
  unsigned long long* next;
};

// A view of 2-bit symbols: positions [0, len) of words at off (forward) or of off + len - 1 downwards (reversed).
struct AlignSeq {
  const uint64_t* w;
  int off, len;
  bool rev;
};
SWB_HD uint32_t align_code(const AlignSeq& s, int p) {
  const int a = s.rev ? s.off + s.len - 1 - p : s.off + p;
  return (uint32_t)(s.w[a >> 5] >> (2 * (a & 31))) & 3u;
}

SWB_HD unsigned long long align_atomic_add(unsigned long long* p, unsigned long long v) {
#if SWB_DEVICE_CODE
  return atomicAdd(p, v);
#else
  return reinterpret_cast<std::atomic<unsigned long long>*>(p)->fetch_add(v);
#endif
}
SWB_HD int align_atomic_inc(int* p) {
#if SWB_DEVICE_CODE
  return atomicAdd(p, 1);
#else
  return reinterpret_cast<std::atomic<int>*>(p)->fetch_add(1);
#endif
}

SWB_HD int imax2(int a, int b) { return a > b ? a : b; }

// 64-bit words of direction nibbles a rectangle of lx T columns x ly Q rows takes
SWB_HD long long align_dir_words(int lx, int ly) { return (long long)((lx + kAlignStrip - 1) / kAlignStrip) * ly; }

// One recurrence over X (T side, columns x = 1..X.len) x Y (Q side, rows y = 1..Y.len).
//   MODE 0: local (main.cpp:57-63), returns the maximum and its cell;  MODE 1: anchored, the same;
//   MODE 2: anchored with direction nibbles, returns H at (X.len, Y.len).
//   SWP: seq1 is X (the pair was swapped); picks the tie rule's order and which gap is E (consumes seq1) and which F.
template <int MODE, bool SWP>
SWB_HD int align_dp(const AlignBatchParams& P, const AlignSeq& X, const AlignSeq& Y, long long tid, uint64_t* dirs,
                    long long dstride, int* bx, int* by) {
  constexpr int S = kAlignStrip;
  constexpr bool ANCH = MODE >= 1, DIRS = MODE == 2;
  const int LX = X.len, LY = Y.len;
  const int gi = P.gap_init, ge = P.gap_ext, gmin = gi < ge ? gi : ge;
  const int ma = P.match, mi = P.mismatch;
  int2* col = P.col + tid;
  const long long cs = P.nthreads;
  // left border (x = 0): H(0, y), and the gap along T there (impossible in the anchored matrix)
  for (int y = 0; y <= LY; ++y) {
    int2 v = make_int2(0, 0);
    if (ANCH) v = make_int2(y == 0 ? 0 : -(gi + (y - 1) * gmin), kAlignNeg);
    col[y * cs] = v;
  }
  int best = 0, bi = 0, bj = 0;          // the tie rule's coordinates: j in seq1, i in seq2
  for (int x0 = 0; x0 < LX; x0 += S) {
    uint32_t xc[S];
    int hp[S], gy[S];                    // H(x, y-1), gap along Q at (x, y-1)
#pragma unroll
    for (int r = 0; r < S; ++r) {
      const int x = x0 + r + 1;
      xc[r] = x <= LX ? align_code(X, x - 1) : 4u;
      hp[r] = ANCH ? -(gi + (x - 1) * gmin) : 0;
      gy[r] = ANCH ? kAlignNeg : 0;
    }
    int hd = col[0].x;                   // H(x0, y-1)
    for (int y = 1; y <= LY; ++y) {
      const uint32_t yc = align_code(Y, y - 1);
      const int2 c = col[y * cs];
      int hleft = c.x, gx = c.y;         // H(x-1, y), gap along T at (x-1, y)
      int hdiag = hd;
      hd = c.x;
      uint64_t dword = 0;
#pragma unroll
      for (int r = 0; r < S; ++r) {
        const int s = xc[r] == yc ? ma : mi;
        const int gx_ext = gx - ge, gx_open = hleft - gi;
        const int gy_ext = gy[r] - ge, gy_open = hp[r] - gi;
        gx = imax2(gx_ext, gx_open);
        const int gyv = imax2(gy_ext, gy_open);
        const int d = hdiag + s;
        int h = imax2(d, imax2(gx, gyv));
        if (!ANCH) h = imax2(h, 0);
        if (DIRS) {
          const int e = SWP ? gx : gyv;                       // E: a base of seq1 against a gap
          const bool e_ext = SWP ? gx_ext > gx_open : gy_ext > gy_open;
          const bool f_ext = SWP ? gy_ext > gy_open : gx_ext > gx_open;
          const uint32_t src = h == d ? 0u : (h == e ? 1u : 2u);
          dword |= (uint64_t)(src | (e_ext ? 4u : 0u) | (f_ext ? 8u : 0u)) << (4 * r);
        } else {
          const int x = x0 + r + 1;
          const int j = SWP ? x : y, i = SWP ? y : x;
          if (x <= LX && (h > best || (h == best && h > 0 && (j < bj || (j == bj && i < bi))))) { best = h; bj = j; bi = i; }
        }
        hdiag = hp[r];
        hp[r] = h;
        gy[r] = gyv;
        hleft = h;
      }
      col[y * cs] = make_int2(hleft, gx);
      if (DIRS) dirs[((long long)(x0 / S) * LY + (y - 1)) * dstride] = dword;
    }
    const int xn = x0 + S;               // H(xn, 0) for the next strip
    col[0] = make_int2(ANCH ? -(gi + (xn - 1) * gmin) : 0, kAlignNeg);
    if (DIRS && x0 + S >= LX) {
      // H(LX, LY) sits in register (LX - 1 - x0) of the last strip
      int hl = 0;
#pragma unroll
      for (int r = 0; r < S; ++r) hl = r == LX - 1 - x0 ? hp[r] : hl;
      best = hl;
    }
  }
  if (!DIRS) { *bx = SWP ? bj : bi; *by = SWP ? bi : bj; }
  return best;
}

// Passes 1 and 2 for pair k: score and span.  Returns the cells computed.
SWB_HD long long align_span_pair(const AlignBatchParams& P, long long k, long long tid) {
  const int LQ = P.q_len[k], LT = P.t_len[k];
  const bool swp = P.len1[k] != LQ;
  int* span = P.spans + 4 * k;
  span[0] = span[1] = span[2] = span[3] = 0;
  P.scores[k] = 0;
  if (LQ == 0 || LT == 0) return 0;
  const uint64_t* qw = P.q_words + k * P.q_stride;
  const uint64_t* tw = P.t_words + k * P.t_stride;
  int xe = 0, ye = 0;
  const AlignSeq X{tw, 0, LT, false}, Y{qw, 0, LQ, false};
  const int s = swp ? align_dp<0, true>(P, X, Y, tid, nullptr, 0, &xe, &ye) : align_dp<0, false>(P, X, Y, tid, nullptr, 0, &xe, &ye);
  P.scores[k] = s;
  if (s <= 0) return (long long)LQ * LT;
  int rx = 0, ry = 0;
  const AlignSeq Xr{tw, 0, xe, true}, Yr{qw, 0, ye, true};
  const int s2 = swp ? align_dp<1, true>(P, Xr, Yr, tid, nullptr, 0, &rx, &ry) : align_dp<1, false>(P, Xr, Yr, tid, nullptr, 0, &rx, &ry);
  if (s2 != s) { atomic_or_i32(P.err, kAlignErrStart); return 0; }
  const int xs = xe - rx + 1, ys = ye - ry + 1;
  // seq1/seq2 terms: i in seq2, j in seq1
  span[0] = swp ? ys : xs; span[1] = swp ? xs : ys; span[2] = swp ? ye : xe; span[3] = swp ? xe : ye;
  return (long long)LQ * LT + (long long)xe * ye;
}

// The walk over the direction nibbles of a lx x ly rectangle, from its last cell back to (0, 0).  Operations come out
// last-first; WRITE = false counts them and re-scores, WRITE = true stores them first-first (ops[n - 1 - t]).
template <bool WRITE>
SWB_HD int align_walk(const AlignBatchParams& P, const uint64_t* dirs, long long dstride, const AlignSeq& X, const AlignSeq& Y,
                      bool swp, int n, uint32_t* ops, long long* total) {
  const int LX = X.len, LY = Y.len;
  const bool split = P.gap_ext > P.gap_init;
  int x = LX, y = LY, state = 0, nops = 0, run = 0;
  uint32_t cur = 0;
  bool brk = false;
  long long tot = 0;
  auto flush = [&]() {
    if (run <= 0) return;
    if (cur == kOpEq) tot += (long long)run * P.match;
    else if (cur == kOpX) tot += (long long)run * P.mismatch;
    else tot -= P.gap_init + (long long)(run - 1) * P.gap_ext;
    if (WRITE) ops[n - 1 - nops] = ((uint32_t)run << 4) | cur;
    ++nops;
  };
  auto emit = [&](uint32_t op, int cnt) {
    if (op == cur && !brk) { run += cnt; return; }
    flush();
    cur = op; run = cnt; brk = false;
  };
  while (x > 0 && y > 0) {
    const uint32_t d = (uint32_t)(dirs[((long long)((x - 1) / kAlignStrip) * LY + (y - 1)) * dstride] >> (4 * ((x - 1) % kAlignStrip))) & 0xFu;
    if (state == 0) {
      const uint32_t src = d & 3u;
      if (src == 0) { emit(align_code(X, x - 1) == align_code(Y, y - 1) ? kOpEq : kOpX, 1); --x; --y; }
      else state = (int)src;
    } else if (state == 1) {                     // E: a base of seq1 against a gap
      emit(kOpIns, 1);
      const bool opened = !(d & 4u);
      state = opened ? 0 : 1;
      if (swp) --x; else --y;
      brk = opened && split;
    } else {                                     // F: a base of seq2 against a gap
      emit(kOpDel, 1);
      const bool opened = !(d & 8u);
      state = opened ? 0 : 2;
      if (swp) --y; else --x;
      brk = opened && split;
    }
  }
  const int j = swp ? x : y, i = swp ? y : x;
  if (j > 0) emit(kOpIns, j);
  if (i > 0) emit(kOpDel, i);
  flush();
  *total = tot;
  return nops;
}

// Pass 3 and the walk for pair k (score and span from align_span_pair).  Returns the cells computed, or -1 if the pair
// must wait for the next round (pool exhausted).
SWB_HD long long align_trace_pair(const AlignBatchParams& P, long long k, long long tid) {
  const int s = P.scores[k];
  if (s <= 0) { P.ops_count[k] = 0; return 0; }
  const int LQ = P.q_len[k];
  const bool swp = P.len1[k] != LQ;
  const int* span = P.spans + 4 * k;
  // rectangle in Q/T terms: Q rows ys..ye, T columns xs..xe (1-based)
  const int ys = swp ? span[0] : span[1], ye = swp ? span[2] : span[3];
  const int xs = swp ? span[1] : span[0], xe = swp ? span[3] : span[2];
  const int lx = xe - xs + 1, ly = ye - ys + 1;
  const long long words = align_dir_words(lx, ly);
  uint64_t* dirs;
  long long dstride;
  if (words <= P.slot_words) { dirs = P.slot + tid; dstride = P.nthreads; }
  else {
    const unsigned long long at = align_atomic_add(P.pool_used, (unsigned long long)words);
    if ((long long)at + words > P.pool_words) { P.pending[align_atomic_inc(P.npending)] = (int)k; return -1; }
    dirs = P.pool + at; dstride = 1;
  }
  const AlignSeq X{P.t_words + k * P.t_stride, xs - 1, lx, false}, Y{P.q_words + k * P.q_stride, ys - 1, ly, false};
  int unused0 = 0, unused1 = 0;
  const int h = swp ? align_dp<2, true>(P, X, Y, tid, dirs, dstride, &unused0, &unused1)
                    : align_dp<2, false>(P, X, Y, tid, dirs, dstride, &unused0, &unused1);
  const long long cells = (long long)lx * ly;
  if (h != s) { atomic_or_i32(P.err, kAlignErrTrace); P.ops_count[k] = 0; return cells; }
  long long total = 0;
  const int n = align_walk<false>(P, dirs, dstride, X, Y, swp, 0, nullptr, &total);
  if (total != s) { atomic_or_i32(P.err, kAlignErrRescore); P.ops_count[k] = 0; return cells; }
  if (n > P.ops_stride) { P.ops_count[k] = -n; return cells; }
  align_walk<true>(P, dirs, dstride, X, Y, swp, n, P.ops + k * (long long)P.ops_stride, &total);
  P.ops_count[k] = n;
  return cells;
}

#if defined(__CUDACC__) && defined(SWB_ALIGN_BATCH_KERNELS)     // defined in swb_align_batch.cu only: one definition
__global__ void __launch_bounds__(256) align_span_kernel(const __grid_constant__ AlignBatchParams P) {
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long cells = 0;
  for (long long k = tid; k < P.npairs; k += P.nthreads) cells += align_span_pair(P, k, tid);
  if (cells) atomicAdd(P.cells, (unsigned long long)cells);
}
__global__ void __launch_bounds__(256) align_trace_kernel(const __grid_constant__ AlignBatchParams P) {
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long cells = 0;
  for (long long t = tid; t < P.ntodo; t += P.nthreads) {
    const long long c = align_trace_pair(P, P.todo ? P.todo[t] : t, tid);
    cells += c > 0 ? c : 0;
  }
  if (cells) atomicAdd(P.cells, (unsigned long long)cells);
}
#endif

// host launchers (swb_align_batch.cu); blocks x 256 threads must equal P.nthreads
void launch_align_span(const AlignBatchParams& P, int blocks, cudaStream_t s);
void launch_align_trace(const AlignBatchParams& P, int blocks, cudaStream_t s);

}  // namespace swb
