// swb_traceback.cuh -- the walk of swb200_align through the direction nibbles the mode-10/11 kernels record, and the
// hand-over of a checkpoint row between the launches of a blocked traceback.
//
// Blocked traceback.  When the 4-bit directions of the whole span rectangle do not fit in device memory, the span's rows
// are cut into blocks of K rows (a multiple of the 256-row band).  A forward sweep, one launch per block, keeps only the
// bottom row {H - open, F} of each block but the last (a checkpoint).  The walk then goes back one block at a time: block
// b is recomputed from checkpoint b - 1 over the columns [0, j) left of where the walk entered it (values left of column
// j do not depend on later columns), and walked until the walk leaves it through its top edge.  Every launch starts from
// exact H and F values, so its nibbles are the ones the whole-matrix launch records, and the walk is the same walk.
// Everything here is __host__ __device__ so that tests/emu/align_blocks_emu.cu runs the same source on CPU threads.
#pragma once
#include "swb_engine.cuh"

namespace swb {

constexpr int kDirBandRows = 256;   // rows of one band of the direction kernels: 32 lanes x 8 rows

// A walk between two blocks: the next cell it reads (1-based span row i, column j), its Gotoh state (0 H, 1 E, 2 F),
// and the run-length encoder (current operation, its length, operations written so far).
struct WalkState {
  long long i, j, nops, run;
  unsigned cur;
  int state;
  int done;        // 1 once the walk has reached row 0 or column 0 and flushed its last run
};

SWB_HD WalkState walk_start(long long rows, long long cols) { return WalkState{rows, cols, 0, 0, 0u, 0, 0}; }

SWB_HD void walk_emit(WalkState& ws, unsigned op, long long cnt, unsigned long long* ops, long long ops_cap) {
  if (op == ws.cur) { ws.run += cnt; return; }
  if (ws.run > 0) { if (ws.nops < ops_cap) ops[ws.nops] = ((unsigned long long)ws.cur << 56) | (unsigned long long)ws.run; ++ws.nops; }
  ws.cur = op; ws.run = cnt;
}

// Follows the directions of ONE launch back from cell (ws.i, ws.j) in state ws.state.  The launch covered the span rows
// (row0, row0 + its bands * 256] (row0 a multiple of 256; dirs holds its bands from row0 / 256 on, nsteps steps each; lane l
// processed column j at step j - 1 + sk * l).  Operations come out last-first, run-length encoded: ops[k] = op << 56 |
// count, op 'M' (a column of seq1 against a row of seq2), 'I' (a column of seq1 against a gap), 'D' (a row of seq2
// against a gap).  In H the cell says diagonal / E / F; in E (F) it says whether the gap was extended or opened.
// Returns when the walk leaves these rows through their top edge (ws.i == row0 > 0: the caller continues in the block
// above, same column, same state), or when it reaches row 0 or column 0: the rest is one gap, and the last run is flushed.
// row0 = 0 over the whole span's directions is the one-block walk.
SWB_HD void walk_block(const uint32_t* dirs, long long nsteps, int sk, long long row0, WalkState& ws,
                       unsigned long long* ops, long long ops_cap) {
  long long i = ws.i, j = ws.j;
  int state = ws.state;
  while (i > row0 && j > 0) {
    const long long r0 = i - 1 - row0;
    const long long band = r0 >> 8;                       // 32 lanes x 8 rows per band
    const int lane = (int)((r0 & 255) >> 3), r = (int)(r0 & 7);
    const long long k = (j - 1) + (long long)sk * lane;   // the step at which this lane processed column j
    const uint32_t d = (dirs[(size_t)(band * nsteps + k) * 32 + lane] >> (4 * r)) & 0xFu;
    if (state == 0) {
      const uint32_t src = d & 3u;
      if (src == 0) { walk_emit(ws, 'M', 1, ops, ops_cap); --i; --j; } else state = (int)src;
    } else if (state == 1) {
      walk_emit(ws, 'I', 1, ops, ops_cap); state = (d & 4u) ? 1 : 0; --j;
    } else {
      walk_emit(ws, 'D', 1, ops, ops_cap); state = (d & 8u) ? 2 : 0; --i;
    }
  }
  ws.i = i; ws.j = j; ws.state = state;
  if (i == 0 || j == 0) {
    if (j > 0) walk_emit(ws, 'I', j, ops, ops_cap);
    if (i > 0) walk_emit(ws, 'D', i, ops, ops_cap);
    walk_emit(ws, 0, 0, ops, ops_cap);                    // flush the last run
    ws.done = 1;
  }
}

// Checkpoint hand-over.  The last band of a forward block launch writes its bottom row through final_out: slot s holds
// {H - open, F} of T position s - SKEW at entries 2s, 2s + 1, tagged with that launch's epoch.  The first band of a later
// launch waits for tag ext_tag_base | first_band << 8 (producer step s < ext_len: lap 0), so the values are copied into
// that launch's ext_in stream under its own tag.  A fresh epoch per launch keeps stale link entries of a recomputed band
// from validating.
SWB_HD void retag_slot(const uint2* ckpt, uint2* ext, long long s, uint32_t tag) {
  ext[2 * s] = make_uint2(ckpt[2 * s].x, tag);
  ext[2 * s + 1] = make_uint2(ckpt[2 * s + 1].x, tag);
}

}  // namespace swb
