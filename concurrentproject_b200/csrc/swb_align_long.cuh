// swb_align_long.cuh -- score, span and CIGAR for every pair of a batch whose shorter side may exceed 1024
// (swb200_align_long_batch, swb200_batch_align_long).  DESIGN.md section 4e.
//
// One warp per pair, 32-bit lanes.  The pair is read from a batch packed with keep_order = 0 (Q = the shorter sequence,
// rows y; T = the longer, columns x); the caller's len1 tells whether the packer swapped it (SWP: seq1 is T), exactly as
// in swb_align_batch.cuh.  Q is cut into bands of 256 rows; lane l owns rows 8l + 1 .. 8l + 8 of a band and processes
// column x at step k = (x - 1) + l (a lane skew of one step).  H, the gap along Q and the diagonal travel down a lane's
// eight rows in registers; lane l takes {H, gap along Q} of the row above its first from lane l - 1's last row, made in
// the step before, by shfl.  Lane 0 takes it from the row above the band: the zero / border row in band 0, else the
// band above's bottom row, which lane 31 leaves per column in the warp's boundary row in device memory (8 B a column).
//
//   pass 1  local recurrence over the pair, tracking the end cell (max H, then the smallest position in seq1, then in
//           seq2, whichever of Q and T is seq1: the rule is applied as a comparison, never by visiting order, because
//           within a band the sweep goes column by column and a later band can hold an equal H at a smaller column);
//   pass 2  the anchored recurrence over the reversed prefixes that end at the end cell: its maximum is the score again
//           and sits at the start cell;
//   pass 3  the anchored recurrence over the span rectangle, recording align_dp's 4 direction bits per cell: one 32-bit
//           word of 8 nibbles per lane per step, dirs[(band * (lx + 31) + k) * 32 + lane] (walk_block's layout with
//           sk = 1), one coalesced 128-byte line per warp and step.  Then lane 0 walks back from the last cell while
//           the warp stages lines through shared memory ahead of it, and the operations are encoded, '=' / 'X' split and
//           re-scored as in swb_align_banded.cuh.
//
// Passes 1 + 2 are one kernel, pass 3 + walk another; warps draw pairs from a counter, so a warp that drew a short pair
// takes the next one while others still sweep long ones.  Direction storage: a slot per warp of the trace launch, else a
// piece of the shared pool, else the pending list of the next round (align_rounds_locked in swb200.cu).  Everything per
// pair is SWB_HD on a WarpCtx, so tests/emu/align_long_emu.cu runs the same bodies with one pthread per lane.
#pragma once
#include "swb_align_banded.cuh"

namespace swb {

constexpr int kLongAlignWarps = 4;          // warps per CTA
constexpr int kLongLaneRows = 8;            // Q rows per lane: one nibble each in a 32-bit direction word
constexpr int kLongBandRows = 32 * kLongLaneRows;
constexpr int kLongStageLines = 32;         // direction lines (one step each) the walk has staged

// 32-bit direction words a span of lx T columns x ly Q rows takes: ceil(ly / 256) bands of lx + 31 steps of 32 words
SWB_HD long long long_dir_words(int lx, int ly) {
  return (long long)((ly + kLongBandRows - 1) / kLongBandRows) * ((long long)lx + 31) * 32;
}

// Shared memory of one warp.  Rings indexed by 0-based column c: tc (T symbols, filled a chunk of 32 steps ahead),
// bin (the row above the band for lane 0, a chunk ahead), bout (lane 31's bottom row until its 128-byte line is stored).
struct LongWarpSmem {
  uint32_t tc[128];
  int2 bin[64];
  int2 bout[128];
};

// The next pair (or todo index) from the launch's counter, in every lane
SWB_HD long long long_take(const AlignBatchParams& P, const WarpCtx& w) {
  unsigned long long v = 0;
  if (w.lane == 0) v = atomic_fetch_add_u64(P.next, 1ull);
  return (long long)(((unsigned long long)w.shfl((uint32_t)(v >> 32), 0) << 32) | w.shfl((uint32_t)v, 0));
}

// the end / start cell's tie rule in x (T) / y (Q) terms: the larger H; among equal H > 0 the smaller position in seq1,
// then in seq2 (SWP: seq1 is x)
template <bool SWP>
SWB_HD bool long_better(int h, int x, int y, int bh, int bx, int by) {
  const int j = SWP ? x : y, i = SWP ? y : x, bj = SWP ? bx : by, bi = SWP ? by : bx;
  return h > bh || (h == bh && h > 0 && (j < bj || (j == bj && i < bi)));
}

// One recurrence over X (T side, columns x = 1..X.len) x Y (Q side, rows y = 1..Y.len); the same result in every lane.
//   MODE 0: local, returns the maximum and its cell;  MODE 1: anchored, the same;
//   MODE 2: anchored with direction nibbles into dirs (long_dir_words(X.len, Y.len) words), returns H at (X.len, Y.len).
// bnd: the warp's boundary row (X.len entries); *cells += the cells this lane computed.
template <int MODE, bool SWP>
SWB_HD int long_dp(const AlignBatchParams& P, const WarpCtx& w, const AlignSeq& X, const AlignSeq& Y, int2* bnd,
                   LongWarpSmem* sm, uint32_t* dirs, int* bx, int* by, long long* cells) {
  constexpr bool ANCH = MODE >= 1, DIRS = MODE == 2;
  constexpr int RW = kLongLaneRows;
  const int LX = X.len, LY = Y.len, lane = w.lane;
  const int gi = P.gap_init, ge = P.gap_ext, gmin = gi < ge ? gi : ge;
  const int ma = P.match, mi = P.mismatch;
  const int GOUT = ANCH ? kAlignNeg : 0;               // a gap on the border (impossible in the anchored matrix)
  *bx = 0; *by = 0;
  if (LX <= 0 || LY <= 0) return 0;
  const int nbands = (LY + kLongBandRows - 1) / kLongBandRows;
  const int nsteps = (LX + 31 + 31) / 32 * 32;         // whole chunks of 32 steps over k = 0 .. LX + 30
  const long long dsteps = (long long)LX + 31;         // steps a band of directions holds
  const int left = (lane + 31) & 31;
  auto tcode = [&](int c) -> uint32_t { return c >= 0 && c < LX ? align_code(X, c) : 0u; };
  int best = 0, bxx = 0, byy = 0, hlast = 0;
  long long nc = 0;
  for (int band = 0; band < nbands; ++band) {
    const int y0 = band * kLongBandRows + lane * RW;   // this lane's rows are y0 + 1 .. y0 + 8
    const bool carry = band + 1 < nbands;              // the next band reads this band's bottom row
    const int rows_in = LY - y0 < 0 ? 0 : (LY - y0 > RW ? RW : LY - y0);
    // the row above the band at column c (0-based): the border row in band 0, else the boundary row
    auto above = [&](int c) -> int2 {
      if (band > 0 && c < LX) return bnd[c];
      return make_int2(ANCH ? -(gi + c * gmin) : 0, GOUT);
    };
    uint32_t qc = 0;
    int hl[RW], gx[RW];                                // H(x - 1, y), gap along T at (x - 1, y): the left border first
#pragma unroll
    for (int r = 0; r < RW; ++r) {
      const int y = y0 + r + 1;
      qc |= (y <= LY ? align_code(Y, y - 1) : 0u) << (2 * r);
      hl[r] = ANCH ? -(gi + (y - 1) * gmin) : 0;
      gx[r] = GOUT;
    }
    int up_prev = ANCH && y0 > 0 ? -(gi + (y0 - 1) * gmin) : 0;   // H(x - 1, y0): the diagonal of the first row
    int sh = 0, sf = 0;                                // {H, gap along Q} of the last row at the last step: to lane + 1
    sm->tc[lane] = tcode(lane);
    uint32_t tnext = tcode(32 + lane);
    int2 bpref = above(lane);
    for (int i0 = 0; i0 < nsteps; i0 += 32) {
      // This chunk reads T symbols of columns [i0 - 31, i0 + 31] and the row above for columns [i0, i0 + 32); the
      // rings get the next chunk's entries before the barrier, into slots the previous chunks no longer read.
      sm->tc[(i0 + 32 + lane) & 127] = tnext;
      tnext = tcode(i0 + 64 + lane);
      sm->bin[(i0 + lane) & 63] = bpref;
      // One boundary row per warp, updated in place, is safe.  Column c is loaded into bpref in the chunk that starts at
      // i0 = c - 32 - c % 32, before any step of this band uses it.  Lane 31 makes column c at step c + 31, and the warp
      // stores it with the rest of its 128-byte line [i0 - 64, i0 - 32) in the chunk that starts at i0 = c + 64 - c % 32,
      // once lane 31 has passed the line's last column (at step i0 - 1).  Load and store of a column are made by the
      // same lane (c % 32), so the load always comes first in program order.
      bpref = above(i0 + 32 + lane);
      w.sync();
      if (carry) {
        const int c = i0 - 64 + lane;
        if (c >= 0 && c < LX) bnd[c] = sm->bout[c & 127];
      }
      for (int u = 0; u < 32; ++u) {
        const int k = i0 + u, c = k - lane;            // this lane's column x = c + 1
        const int rh = (int)w.shfl((uint32_t)sh, left), rf = (int)w.shfl((uint32_t)sf, left);
        int hup = rh, fv = rf;
        if (lane == 0) { const int2 b = sm->bin[k & 63]; hup = b.x; fv = b.y; }
        const bool cin = c >= 0 && c < LX;
        const uint32_t tcv = sm->tc[c & 127];
        const int above_h = hup;
        int diag = up_prev;
        uint32_t dword = 0;
#pragma unroll
        for (int r = 0; r < RW; ++r) {
          const int s = ((qc >> (2 * r)) & 3u) == tcv ? ma : mi;
          const int gx_ext = gx[r] - ge, gx_open = hl[r] - gi;
          const int gy_ext = fv - ge, gy_open = hup - gi;
          const int gxv = imax2(gx_ext, gx_open), gyv = imax2(gy_ext, gy_open);
          const int d = diag + s;
          int h = imax2(d, imax2(gxv, gyv));
          if (!ANCH) h = imax2(h, 0);
          if (DIRS) {
            const int e = SWP ? gxv : gyv;                       // E: a base of seq1 against a gap
            const bool e_ext = SWP ? gx_ext > gx_open : gy_ext > gy_open;
            const bool f_ext = SWP ? gy_ext > gy_open : gx_ext > gx_open;
            const uint32_t src = h == d ? 0u : (h == e ? 1u : 2u);
            dword |= (src | (e_ext ? 4u : 0u) | (f_ext ? 8u : 0u)) << (4 * r);
            if (c == LX - 1 && y0 + r + 1 == LY) hlast = h;
          } else if (cin && r < rows_in && h >= best && long_better<SWP>(h, c + 1, y0 + r + 1, best, bxx, byy)) {
            best = h; bxx = c + 1; byy = y0 + r + 1;
          }
          diag = hl[r];
          if (cin) { hl[r] = h; gx[r] = gxv; }
          hup = h; fv = gyv;
        }
        if (cin) up_prev = above_h;
        sh = hup; sf = fv;
        if (DIRS && k < dsteps) dirs[((long long)band * dsteps + k) * 32 + lane] = dword;
        if (carry && lane == 31) sm->bout[c & 127] = make_int2(hup, fv);
        nc += cin ? rows_in : 0;
      }
    }
    w.sync();
    if (carry) {
      // the last lines: lane 31 made its last column, nsteps - 32 >= LX - 1, at step nsteps - 1
      for (int c = nsteps - 64 + lane; c < nsteps - 31; c += 32)
        if (c >= 0 && c < LX) bnd[c] = sm->bout[c & 127];
    }
  }
  *cells += nc;
  if constexpr (DIRS) {
    // H(LX, LY) was made by the lane owning row LY in the last band
    return (int)w.shfl((uint32_t)hlast, ((LY - 1) % kLongBandRows) / RW);
  } else {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int oh = (int)w.shfl((uint32_t)best, lane ^ o), ox = (int)w.shfl((uint32_t)bxx, lane ^ o);
      const int oy = (int)w.shfl((uint32_t)byy, lane ^ o);
      if (long_better<SWP>(oh, ox, oy, best, bxx, byy)) { best = oh; bxx = ox; byy = oy; }
    }
    *bx = bxx; *by = byy;
    return best;
  }
}

// Passes 1 and 2 for pair k: score and span.  Returns this lane's cells.
SWB_HD long long long_span_pair(const AlignBatchParams& P, const WarpCtx& w, long long k, int2* bnd, LongWarpSmem* sm) {
  const int LQ = P.q_len[k], LT = P.t_len[k];
  const bool swp = P.len1[k] != LQ;
  const uint64_t* qw = P.q_words + k * P.q_stride;
  const uint64_t* tw = P.t_words + k * P.t_stride;
  long long nc = 0;
  int xe = 0, ye = 0, rx = 0, ry = 0;
  const AlignSeq X{tw, 0, LT, false}, Y{qw, 0, LQ, false};
  const int s = swp ? long_dp<0, true>(P, w, X, Y, bnd, sm, nullptr, &xe, &ye, &nc)
                    : long_dp<0, false>(P, w, X, Y, bnd, sm, nullptr, &xe, &ye, &nc);
  int s2 = s;
  if (s > 0) {
    const AlignSeq Xr{tw, 0, xe, true}, Yr{qw, 0, ye, true};
    s2 = swp ? long_dp<1, true>(P, w, Xr, Yr, bnd, sm, nullptr, &rx, &ry, &nc)
             : long_dp<1, false>(P, w, Xr, Yr, bnd, sm, nullptr, &rx, &ry, &nc);
  }
  if (w.lane == 0) {
    int* span = P.spans + 4 * k;
    P.scores[k] = s;
    const bool ok = s > 0 && s2 == s;
    const int xs = xe - rx + 1, ys = ye - ry + 1;
    // seq1/seq2 terms: i in seq2, j in seq1
    span[0] = ok ? (swp ? ys : xs) : 0; span[1] = ok ? (swp ? xs : ys) : 0;
    span[2] = ok ? (swp ? ye : xe) : 0; span[3] = ok ? (swp ? xe : ye) : 0;
    if (s2 != s) atomic_or_i32(P.err, kAlignErrStart);
  }
  return nc;
}

// The walk over the direction lines of a span (X / Y as pass 3 saw them) from its last cell back to (0, 0).  Lane 0
// walks; the step index only decreases inside a band, so the warp stages the kLongStageLines lines at and below lane
// 0's step into stage, again whenever the walk leaves them or enters the band above.  Operations come out last-first
// (OpEncoder); returns the count and *total in every lane.
template <bool WRITE>
SWB_HD int long_walk(const AlignBatchParams& P, const WarpCtx& w, const uint32_t* dirs, const AlignSeq& X, const AlignSeq& Y,
                     bool swp, uint32_t* stage, int n, uint32_t* ops, int* total) {
  const int lane = w.lane;
  const long long dsteps = (long long)X.len + 31;
  OpEncoder<WRITE> enc{P.match, P.mismatch, P.gap_init, P.gap_ext, ops, n};
  int x = X.len, y = Y.len, state = 0;
  for (;;) {
    const int band = (int)w.shfl((uint32_t)((y - 1) / kLongBandRows), 0);
    const int top = (int)w.shfl((uint32_t)((x - 1) + ((y - 1) % kLongBandRows) / kLongLaneRows), 0);
    const int base = top - kLongStageLines + 1 > 0 ? top - kLongStageLines + 1 : 0;
    w.sync();
    for (int q = 0; q < kLongStageLines && base + q <= top; ++q)
      stage[q * 32 + lane] = dirs[((long long)band * dsteps + base + q) * 32 + lane];
    w.sync();
    int done = 1;
    if (lane == 0) {
      while (x > 0 && y > 0) {
        const int r0 = (y - 1) % kLongBandRows, ln = r0 / kLongLaneRows, k = (x - 1) + ln;
        if ((y - 1) / kLongBandRows != band || k < base) break;
        const uint32_t d = (stage[(k - base) * 32 + ln] >> (4 * (r0 % kLongLaneRows))) & 0xFu;
        if (state == 0) {
          const uint32_t src = d & 3u;
          if (src == 0) { enc.emit(align_code(X, x - 1) == align_code(Y, y - 1) ? kOpEq : kOpX, 1); --x; --y; }
          else state = (int)src;
        } else if (state == 1) {                   // E: a base of seq1 against a gap
          const bool opened = !(d & 4u);
          enc.emit(kOpIns, 1, opened);
          state = opened ? 0 : 1;
          if (swp) --x; else --y;
        } else {                                   // F: a base of seq2 against a gap
          const bool opened = !(d & 8u);
          enc.emit(kOpDel, 1, opened);
          state = opened ? 0 : 2;
          if (swp) --y; else --x;
        }
      }
      done = !(x > 0 && y > 0);
    }
    if (w.shfl((uint32_t)done, 0)) break;
  }
  int tl = 0;
  if (lane == 0) {
    // the rest runs along row 0 or column 0 of the span: leading gaps
    const int j = swp ? x : y, i = swp ? y : x;
    if (j > 0) enc.emit(kOpIns, j);
    if (i > 0) enc.emit(kOpDel, i);
    enc.flush();
    tl = (int)enc.tot;
  }
  *total = (int)w.shfl((uint32_t)tl, 0);
  return (int)w.shfl((uint32_t)enc.nops, 0);
}

// Pass 3 and the walk for pair k (score and span from long_span_pair); warp: this warp's index in the launch (its
// slot).  Returns this lane's cells, or -1 if the pair must wait for the next round (pool exhausted).
SWB_HD long long long_trace_pair(const AlignBatchParams& P, const WarpCtx& w, long long k, long long warp, int2* bnd,
                                 LongWarpSmem* sm, uint32_t* stage) {
  const int s = P.scores[k];
  if (s <= 0) { if (w.lane == 0) P.ops_count[k] = 0; return 0; }
  const int LQ = P.q_len[k];
  const bool swp = P.len1[k] != LQ;
  const int* span = P.spans + 4 * k;
  // rectangle in Q/T terms: Q rows ys..ye, T columns xs..xe (1-based)
  const int ys = swp ? span[0] : span[1], ye = swp ? span[2] : span[3];
  const int xs = swp ? span[1] : span[0], xe = swp ? span[3] : span[2];
  const int lx = xe - xs + 1, ly = ye - ys + 1;
  const long long words = (long_dir_words(lx, ly) + 1) / 2;          // 64-bit words, the unit of slot and pool
  uint32_t* dirs;
  if (words <= P.slot_words) {
    dirs = reinterpret_cast<uint32_t*>(P.slot + warp * P.slot_words);
  } else {
    unsigned long long at = 0;
    if (w.lane == 0) at = align_atomic_add(P.pool_used, (unsigned long long)words);
    at = (unsigned long long)w.shfl((uint32_t)at, 0) | ((unsigned long long)w.shfl((uint32_t)(at >> 32), 0) << 32);
    if ((long long)at + words > P.pool_words) {
      if (w.lane == 0) P.pending[align_atomic_inc(P.npending)] = (int)k;
      return -1;
    }
    dirs = reinterpret_cast<uint32_t*>(P.pool + at);
  }
  const AlignSeq X{P.t_words + k * P.t_stride, xs - 1, lx, false}, Y{P.q_words + k * P.q_stride, ys - 1, ly, false};
  long long nc = 0;
  int unused0 = 0, unused1 = 0;
  const int h = swp ? long_dp<2, true>(P, w, X, Y, bnd, sm, dirs, &unused0, &unused1, &nc)
                    : long_dp<2, false>(P, w, X, Y, bnd, sm, dirs, &unused0, &unused1, &nc);
  if (h != s) {
    if (w.lane == 0) { atomic_or_i32(P.err, kAlignErrTrace); P.ops_count[k] = 0; }
    return nc;
  }
  w.sync();                                                          // the walk reads lines other lanes stored
  int total = 0;
  const int n = long_walk<false>(P, w, dirs, X, Y, swp, stage, 0, nullptr, &total);
  if (total != s) {
    if (w.lane == 0) { atomic_or_i32(P.err, kAlignErrRescore); P.ops_count[k] = 0; }
    return nc;
  }
  if (n > P.ops_stride) { if (w.lane == 0) P.ops_count[k] = -n; return nc; }
  long_walk<true>(P, w, dirs, X, Y, swp, stage, n, P.ops + k * (long long)P.ops_stride, &total);
  if (w.lane == 0) P.ops_count[k] = n;
  return nc;
}

#if defined(__CUDACC__) && defined(SWB_ALIGN_LONG_KERNELS)      // defined in swb_align_long.cu only: one definition
__global__ void __launch_bounds__(32 * kLongAlignWarps) align_long_span_kernel(const __grid_constant__ AlignBatchParams P) {
  __shared__ LongWarpSmem sm[kLongAlignWarps];
  const WarpCtx w{(int)(threadIdx.x & 31)};
  const int wi = (int)(threadIdx.x / 32);
  const long long warp = (long long)blockIdx.x * kLongAlignWarps + wi;
  int2* bnd = P.col + warp * P.row_stride;
  long long cells = 0;
  for (long long k = long_take(P, w); k < P.npairs; k = long_take(P, w)) cells += long_span_pair(P, w, k, bnd, &sm[wi]);
  if (cells) atomicAdd(P.cells, (unsigned long long)cells);
}
__global__ void __launch_bounds__(32 * kLongAlignWarps) align_long_trace_kernel(const __grid_constant__ AlignBatchParams P) {
  __shared__ LongWarpSmem sm[kLongAlignWarps];
  __shared__ uint32_t stage[kLongAlignWarps][kLongStageLines * 32];
  const WarpCtx w{(int)(threadIdx.x & 31)};
  const int wi = (int)(threadIdx.x / 32);
  const long long warp = (long long)blockIdx.x * kLongAlignWarps + wi;
  int2* bnd = P.col + warp * P.row_stride;
  long long cells = 0;
  for (long long t = long_take(P, w); t < P.ntodo; t = long_take(P, w)) {
    const long long c = long_trace_pair(P, w, P.todo ? P.todo[t] : t, warp, bnd, &sm[wi], stage[wi]);
    cells += c > 0 ? c : 0;
  }
  if (cells) atomicAdd(P.cells, (unsigned long long)cells);
}
#endif

// host launchers (swb_align_long.cu)
void launch_align_long_span(const AlignBatchParams& P, int blocks, cudaStream_t s);
void launch_align_long_trace(const AlignBatchParams& P, int blocks, cudaStream_t s);
const void* align_long_span_kernel_ptr();
const void* align_long_trace_kernel_ptr();

}  // namespace swb
