// swb_engine.cuh -- the wavefront DP engine: score-only Gotoh local alignment of one pair.
//
// Replaces the reference's per-anti-diagonal kernels (simpleGPU.cu:78-107 DPMatrices,
// cudaLazy.cu:21-56 sw_kernel_diag, cudaSmithM.cu:87-126 kernel_compute_diagonal,
// SmithDiagonalGPU.cu:40-67 smithWatermanDiagonal) and their host loops.  Same recurrence as
// main.cpp:57-63, nothing else in common.
//
// Geometry.  One sequence ("Q") is striped across lanes, the other ("T") is streamed.  A *band* is
// the block of Q rows one warp owns while it sweeps all of T.  With packed 16-bit lanes a thread
// carries two *sub-lanes* (lo/hi half of every register) that own R consecutive Q rows each, so a
// band is 64*R rows; with 32-bit lanes a thread is one sub-lane and a band is 32*R rows.  Sub-lane
// v+1 runs one T position behind sub-lane v, so the anti-diagonal dependency of the recurrence
// moves between lanes through one __shfl_sync per step and never touches memory.  H/E stay in
// registers for the whole sweep; the only state that leaves a warp is the band's bottom boundary
// row (H-open and F per T position), handed to the warp that owns the next band through 8-byte
// {value,tag} words in L2 (or in a peer GPU's memory for the last warp of a GPU).  All warps of
// all GPUs form one ring; band b is processed by ring slot b mod ring_total, so consecutive bands
// run concurrently, one boundary-latency apart: a pipelined wavefront with no host involvement.
//
// Arithmetic per cell vector (s16x2: two cells): PRMT (substitution score from a 4-byte table of
// the streamed symbol), VIADD.16x2 (diag+s), VIADDMNMX.S16x2 (E), VIADDMNMX.S16x2 (F),
// VIMNMX3.S16x2.RELU (H), VIADD.16x2 (H-open), 1/2 VIMNMX (running best).  When gap_init ==
// gap_ext the E/F registers are provably redundant (E = H_left-g, F = H_up-g) and MODE 1 drops them.
#pragma once
#include "swb_device.cuh"
#include <type_traits>

namespace swb {

// Step-loop unroll factor.  8 measured 10 % faster than 4 on cfg2 (4.72 -> 4.28 ms; 16 and 2 are slower) -- as long as
// the unrolled loop stays below ~800 instructions: with 12 or more affine rows per lane it got 15-30 % SLOWER
// (instruction cache), so the factor follows the size of one step.
#ifndef SWB_STEP_UNROLL
#define SWB_STEP_UNROLL 8
#endif
constexpr int kStepUnroll = SWB_STEP_UNROLL;
SWB_HD constexpr int step_unroll(double instr_per_row, int rows, int big) { return instr_per_row * rows + 10.0 <= 100.0 ? big : 4; }
#ifndef SWB_STEP_UNROLL32
#define SWB_STEP_UNROLL32 8
#endif
constexpr int kStepUnroll32 = SWB_STEP_UNROLL32;   // 32-bit engine
constexpr int kChunk = 32;     // steps between boundary polls / table refills
constexpr int kTabRing = 256;  // per-warp ring of substitution tables (one per T position), kept twice
constexpr int kInbox = 64;     // per-warp ring of validated top-boundary values

enum : int { STATUS_S16_OVERFLOW = 1, STATUS_SPIN_TIMEOUT = 2, STATUS_BAD_SYMBOL = 4, STATUS_REBASE_RANGE = 8 };

constexpr int kRebaseBlock = 256;     // steps between re-base decisions (re-based 16-bit mode)
constexpr int kRebaseTrigger = 8000;  // re-centre when a live H-open leaves [-8000, 8000] relative to the base

struct EngineParams {
  const uint8_t* q_codes;       // LQ codes in {0,1,2,3}; >= 4 never matches (generic-byte mode: the raw bytes)
  const uint64_t* t_packed;     // LT 2-bit codes, 32 per 64-bit word, position p at bits 2*(p%32)
  const uint8_t* t_bytes;       // generic-byte mode only: the raw bytes of T
  long long LQ, LT;
  int NB;                       // bands = ceil(LQ / rows_per_band)
  int ring_total;               // warps in the whole ring (all GPUs)
  int ring_offset;              // global index of this GPU's first warp
  int warps_local;              // warps launched on this GPU
  uint2* links;                 // (warps_local-1) rings, 2*link_len entries each
  unsigned link_mask;           // link_len-1 (link_len is a power of two, >= 4096)
  int link_shift;               // log2(link_len)
  unsigned long long* progress; // [warps_local] consumer progress words for ring back-pressure
  const uint2* ext_in;          // stream consumed by local warp 0 (full length: 2*ext_len entries)
  uint2* ext_out;               // stream produced by the last local warp (peer memory on multi-GPU)
  unsigned ext_mask;
  int ext_shift;
  uint2* final_out;             // optional: the LAST band's bottom boundary row goes here, slot = its step (two-sided sweep)
  unsigned final_mask;
  uint32_t tag_base;            // local rings: epoch << 26
  uint32_t ext_tag_base;        // ext streams: 14-bit call epoch, high 6 bits << 26 | low 8 bits (ext lap bits are always 0)
  int* result;                  // [0] best score (atomicMax), [1] status bits (atomicOr)
  int match, mismatch, gap_init, gap_ext;
  long long spin_limit;         // polls before a waiting warp gives up (sets STATUS_SPIN_TIMEOUT)
  int dbg;                      // timing experiments only: 1 = no boundary stores, 2 = no boundary polls
  long long* prof;              // optional [warps_local][8]: cycles in prologue, cycles in steps, failed polls, chunks,
                                //   globaltimer at the first band's first chunk / at its end, SM id
  int* cand;                    // TRACK kernels: per band {best H, its T position, its Q row} (first in column-major order)
  uint32_t* dirs;               // DIRS kernels: traceback directions, 4 bits per cell, word (band * nsteps + step) * 32 + lane,
                                //   nibble r = row r of the lane: bits 0-1 where H came from (0 diagonal, 1 E, 2 F), bit 2 E extended, bit 3 F extended
};

constexpr int kRawEntries = kChunk + 4;   // TMA flavour: 32 entries, one more when the first is odd, rounded to 16 bytes
struct WarpSmem {
  uint32_t tab[2 * kTabRing];
  uint32_t inbox[4 * kInbox];   // plane 0: H-open (or packed H-open|F), plane 1: F (s32); each ring kept twice
};
struct WarpSmemTma : WarpSmem {            // launch config 5 only
  alignas(16) uint2 raw[2][kRawEntries];   // boundary entries as the bulk copy delivered them, double buffered
  alignas(8) unsigned long long mbar[2];   // one mbarrier per raw buffer
};

SWB_HD uint32_t pack2(int v) { return ((uint32_t)v & 0xFFFFu) * 0x10001u; }

// PRMT selector producing the packed s16x2 substitution word of one row vector: low half from table
// register A (codes of the lo sub-lane's T symbol), high half from table register B.
SWB_HD uint32_t mk_sel16(uint32_t code_lo, uint32_t code_hi) {
  const uint32_t lo = code_lo < 4 ? (code_lo | ((code_lo | 8u) << 4)) : 0x88u;           // byte, then its sign
  const uint32_t hi = code_hi < 4 ? ((code_hi + 4u) | ((code_hi + 12u) << 4)) : 0xCCu;
  return lo | (hi << 8);
}
SWB_HD uint32_t mk_sel32(uint32_t code) {
  return code < 4 ? (code | ((code | 8u) * 0x1110u)) : 0x8888u;
}

// 4-byte table of (substitution score + gap_init) against T symbol c; c >= 4 = matches nothing.
SWB_HD uint32_t table_word(uint32_t c, uint32_t padw, uint32_t flip) { return c < 4 ? (padw ^ (flip << (8 * c))) : padw; }

struct Waiter {
  long long budget;
  bool aborted;
};

// First lane that gives up leaves a post-mortem in result[3..]: who waited for what.
SWB_HD void record_timeout(const EngineParams& P, int kind, long long a, long long b, long long c, long long d) {
#if SWB_DEVICE_CODE
  if (atomicCAS(P.result + 3, 0, kind) == 0) {
    P.result[4] = (int)a; P.result[5] = (int)b; P.result[6] = (int)c; P.result[7] = (int)d;
    P.result[8] = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  }
#else
  (void)P; (void)kind; (void)a; (void)b; (void)c; (void)d;
#endif
}

// Wait until the entry for producer step j of band `tagband` is present; returns its value.
// Warp-uniform wait: every lane polls its own slot, the warp leaves the loop together.  (A per-lane
// spin loop leaves the warp diverged under independent thread scheduling; every later __shfl_sync
// then takes the divergent slow path -- measured 5x slower steps on B200.)
// need: this lane has a slot to wait for.  Returns the entry value (undefined if !need).
template <class Ctx>
SWB_HD uint32_t wait_entry(const EngineParams& P, const Ctx& w, bool need, const uint2* slot, uint32_t want_tag, uint2 e,
                           Waiter& wt) {
  // e: what a speculative load of *slot returned one chunk ago (usually already the wanted entry)
  for (;;) {
    const bool ok = !need || e.y == want_tag;
    if (w.all(ok) || wt.aborted) break;
    bool give_up = --wt.budget < 0;
    if ((wt.budget & 255) == 0) give_up = give_up || (ld_flag(P.result + 1) & STATUS_SPIN_TIMEOUT);
    if (w.any(give_up)) {
      if (!ok) record_timeout(P, 1, (long long)want_tag, (long long)e.y, (long long)e.x, wt.budget);
      atomic_or_i32(P.result + 1, STATUS_SPIN_TIMEOUT);
      wt.aborted = true;
      break;
    }
    spin_pause();
    if (!ok) e = ld_entry(slot);
  }
  return e.x;
}

// Warp-uniform back-pressure wait on a monotonic progress word.
template <class Ctx>
SWB_HD void wait_progress(const EngineParams& P, const Ctx& w, const unsigned long long* word, unsigned long long need,
                          long long band, long long i0, Waiter& wt) {
  for (;;) {
    const unsigned long long have = ld_progress(word);
    if (w.any(have >= need) || wt.aborted) break;
    if (w.any(--wt.budget < 0)) {
      record_timeout(P, 2, band, i0, (long long)need, (long long)have);
      atomic_or_i32(P.result + 1, STATUS_SPIN_TIMEOUT);
      wt.aborted = true;
      break;
    }
    spin_pause();
  }
}

// Rare path of the chunk prologue, kept out of line so that the common path is straight-line code: the boundary
// entry (and, re-based lanes, the producer's base entry) this lane needs has not arrived yet.  Polls until every
// lane of the warp has what it needs (warp-uniform exit: a per-lane spin loop leaves the warp diverged, and every
// later __shfl_sync then takes the divergent slow path -- measured 5x slower steps on B200), or until the wait
// budget is spent; then STATUS_SPIN_TIMEOUT is set, the caller stops expecting entries and the host reports
// SWB200_ERR_TIMEOUT.
template <class Ctx>
__host__ __device__ __noinline__ long long poll_boundary(const EngineParams& P, const Ctx& w, bool need, const uint2* slot,
                                                         uint32_t want, const uint2* bslot, uint32_t bwant, bool with_base,
                                                         long long budget) {
  // Everything goes in and out BY VALUE (the remaining budget is the result, -1 = gave up): a reference parameter
  // would force the caller's registers into local memory on the hot path.
  for (;;) {
    bool ok = true;
    uint2 e = make_uint2(0u, 0u), be = make_uint2(0u, 0u);
    if (need) {
      e = ld_entry(slot);
      ok = e.y == want;
      if (with_base) { be = ld_entry(bslot); ok = ok && be.y == bwant; }
    }
    if (w.all(ok)) return budget < 0 ? 0 : budget;
    bool give_up = --budget < 0;
    if ((budget & 255) == 0) give_up = give_up || (ld_flag(P.result + 1) & STATUS_SPIN_TIMEOUT);
    if (w.any(give_up)) {
      if (!ok) record_timeout(P, 1, (long long)want, (long long)e.y, (long long)e.x, budget);
      atomic_or_i32(P.result + 1, STATUS_SPIN_TIMEOUT);
      return -1;
    }
    spin_pause();
  }
}

// =================================================================================================
//  Packed 16-bit engine.  MODE 0: affine gaps.  MODE 1: gap_init == gap_ext (E/F eliminated).
//  SLACK 1: a shuffled boundary value is consumed one step after it was sent (hides SHFL latency
//  when a scheduler has a single warp); SLACK 0: consumed in the same step (shorter pipeline).
//  RB (re-based lanes): every register holds value - base, base a warp-uniform int32 that follows the
//  score level, so pairs whose score leaves the s16 range keep two cells per instruction.  Exact:
//  the values a warp holds at one time differ by a bounded amount (|dH| <= max(match, gap) per cell),
//  so they always fit 16 bits around a common base; the zero floor becomes max(.., -base); every 256
//  steps the warp re-centres (adds a constant to all its registers) and publishes its base next to
//  the boundary entries so the band below can translate what it receives.
//
//  Loop structure (round 2).  With one warp per scheduler nothing hides a branch: ncu's source page showed the
//  32-step chunk prologue of round 1 at ~500 cycles (a quarter of the sweep) although it issues only ~150
//  instructions -- a dozen small branches at 15-30 cycles each (predicate -> branch latency, refetch after a taken
//  branch), three clock reads of the profiling hook, 64-bit index arithmetic.  So: blocks of 256 steps carry
//  everything that happens less often than once per chunk (re-basing, progress word, ring back-pressure); the chunk
//  prologue is straight-line code with ONE vote and one never-taken branch to the out-of-line poll loop; the
//  profiling hook is compiled in only with -DSWB_ENABLE_PROF (bench/diag.py builds).
// =================================================================================================
SWB_HD int hi_half_max(uint32_t v) { const int a = (short)(v & 0xFFFFu), b = (short)(v >> 16); return a > b ? a : b; }
SWB_HD int lo_half_min(uint32_t v) { const int a = (short)(v & 0xFFFFu), b = (short)(v >> 16); return a < b ? a : b; }

constexpr int kBlock = kRebaseBlock;   // steps per block; nsteps of the 16-bit engine is a multiple of it (host: run_once)

//  HS (round 2): the same slack for the hand-off INSIDE a thread.  The hi sub-lane's top neighbour is the lo
//  sub-lane's bottom row, so with HS 0 a step cannot start before the previous step's whole row chain has finished:
//  PRMT -> R dependent max ops -> VIADD -> PRMT, a loop-carried recurrence of 4R+10 cycles that one warp per scheduler
//  cannot hide (measured: the step time did not move when every memory instruction and the shuffle were taken out).
//  With HS 1 the hi sub-lane runs two T positions behind the lo sub-lane and consumes the lo bottom row of the step
//  BEFORE the previous one: the recurrence spans two steps.  Costs one register and 31 more positions of lane skew.
//  TMA (launch config 5): the next chunk's 32 boundary entries are fetched by ONE cp.async.bulk (272 bytes, global ->
//  shared, completion on an mbarrier) issued by lane 0 half a chunk ahead, instead of 32 lanes' speculative loads; at
//  the chunk start the warp waits on the mbarrier and every lane takes its {value, tag} from shared memory.  Tag
//  validation, the out-of-line poll and everything after it are unchanged.  Device only (the emulator runs TMA = false).
template <int R, int MODE, int SLACK, bool RB = false, bool SHORT = true, int HS = 0, bool TMA = false>
SWB_HD void engine_warp_s16(const EngineParams& P, const WarpCtx& w, int lw, WarpSmem* sm_base) {
  typedef typename std::conditional<TMA, WarpSmemTma, WarpSmem>::type Smem;
  Smem* sm = static_cast<Smem*>(sm_base);
  static_assert(SLACK == 0 || SLACK == 1, "a shuffled boundary value is consumed in the same step or one step later");
  static_assert(HS == 0 || HS == 1, "the hi sub-lane trails the lo sub-lane by one or two positions");
  constexpr int SK = 2 + SLACK + HS;   // T positions between neighbouring lanes
  constexpr int SKEW = 31 * SK + 1 + HS;   // lane 31's hi sub-lane trails lane 0's lo sub-lane by this
  constexpr int kU = step_unroll(MODE == 0 ? (RB ? 8.5 : 7.5) : (RB ? 5.5 : 4.5), R, kStepUnroll);
  const int lane = w.lane;
  const bool last_lane = lane == 31;
  const int src_lane = (lane + 31) & 31;
  const uint32_t nopen = pack2(-P.gap_init), next = pack2(-P.gap_ext);
  const uint32_t fnext = pack2(-(P.gap_ext < P.gap_init ? P.gap_ext : P.gap_init));   // F carried down inside a lane
  const uint32_t padb = (uint32_t)(P.mismatch + P.gap_init) & 0xFFu;
  const uint32_t padw = padb * 0x01010101u;
  const uint32_t flip = padb ^ ((uint32_t)(P.match + P.gap_init) & 0xFFu);
  const int LT = (int)P.LT;            // step arithmetic is 32-bit (the host refuses LT >= 2^30); only ring indices,
                                       // which count steps over all rounds, are 64-bit
  const int nsteps = ((LT + SKEW + kBlock - 1) / kBlock) * kBlock;
  uint32_t best0 = 0, best1 = 0;
  int base = 0, best_abs = 0;          // RB only
  uint32_t floorw = 0;                 // RB only: packed max(-base, -30000)
  Waiter wt{P.spin_limit, false};
#if SWB_DEVICE_CODE
  uint32_t tma_phase0 = 0, tma_phase1 = 0;      // parity of the next completion of mbar[0] / mbar[1]
  if constexpr (TMA) {
    if (lane == 0) { mbar_init(&sm->mbar[0], 1); mbar_init(&sm->mbar[1], 1); }
    mbar_init_fence();
    w.sync();
  }
#endif
  // P is picked at run time between the two halves of a launch, so every P.field inside a loop is a constant load
  // through a register index; the one the chunk loop needs is kept in a register.
  // (measured: +4.8 % on cfg2 with one warp per scheduler, -2.5 % with two warps per scheduler: only the former do it)
  const uint64_t* t_packed_reg = P.t_packed;
#if SWB_DEVICE_CODE
  if (SHORT) asm volatile("" : "+l"(t_packed_reg));
#endif
#define SWB_T_PACKED (SHORT ? t_packed_reg : P.t_packed)

  for (long long band = P.ring_offset + lw; band < P.NB; band += P.ring_total) {
    const bool zero_src = band == 0 || (P.dbg & 2);
    const bool is_final = band == P.NB - 1 && P.final_out != nullptr;   // its bottom row is wanted by the caller
    const bool has_sink = band + 1 < P.NB || is_final;
    const bool emit = has_sink && last_lane && !(P.dbg & 1);
    const bool first_local = lw == 0, last_local = lw == P.warps_local - 1 || is_final;   // "last": full-length stream, no back-pressure
    const uint2* in = first_local ? P.ext_in : P.links + (size_t)(lw - 1) * 2 * ((size_t)P.link_mask + 1);
    const unsigned in_mask = first_local ? P.ext_mask : P.link_mask;
    const int in_shift = first_local ? P.ext_shift : P.link_shift;
    uint2* out = is_final ? P.final_out : (last_local ? P.ext_out : P.links + (size_t)lw * 2 * ((size_t)P.link_mask + 1));
    const unsigned out_mask = is_final ? P.final_mask : (last_local ? P.ext_mask : P.link_mask);
    const int out_shift = last_local ? P.ext_shift : P.link_shift;
    const uint32_t in_tag = (first_local ? P.ext_tag_base : P.tag_base) | ((uint32_t)band << 8);   // written by band-1 as (band-1)+1
    const uint32_t out_tag = (last_local ? P.ext_tag_base : P.tag_base) | ((uint32_t)(band + 1) << 8);
    unsigned long long* my_progress = P.progress + lw;
    const unsigned long long* sink_progress = P.progress + lw + 1;       // only read when !last_local
    // Inner rings are indexed by the CUMULATIVE producer step over all rounds (sbase + step), so a
    // ring is one continuous stream and back-pressure spans band boundaries; the full-length ext
    // stream restarts at 0 every band (safe: see DESIGN.md, hand-off protocol).
    const long long sbase = (band / P.ring_total) * (long long)nsteps;
    const long long in_base = first_local ? 0 : sbase, out_base = last_local ? 0 : sbase;
    const bool check_sink = has_sink && !last_local;                     // ring back-pressure applies

    // ---- per-band constants: PRMT selectors of this thread's 2*R rows
    uint32_t sel[R];
    {
      const long long row_lo = band * (64LL * R) + (long long)(2 * lane) * R;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const long long a = row_lo + r, b = row_lo + R + r;
        const uint32_t ca = a < P.LQ ? P.q_codes[a] : 4u;
        const uint32_t cb = b < P.LQ ? P.q_codes[b] : 4u;
        sel[r] = mk_sel16(ca, cb);
      }
    }
    // ---- state: H-open, E per row vector; zero boundary = H 0, E/F any value <= 0
    uint32_t Ho[R], E[R];
#pragma unroll
    for (int r = 0; r < R; ++r) { Ho[r] = nopen; E[r] = nopen; }
    uint32_t Fbot = nopen, up_prev = nopen, xsend = nopen, yold = nopen, Thi = padw;
    uint32_t HoLast_d = nopen, Fbot_d = nopen, Thi_d = padw;   // HS: the lo sub-lane's bottom row / table word, one step older
    if (RB) { base = 0; floorw = 0; best0 = 0; best1 = 0; }   // every band starts at T position 0, where all scores are small
    // base entries live in the second half of a link ring: one {base, tag} per kRebaseBlock producer steps
    // (on the full-length ext stream, which restarts every band, four bands' worth of base entries rotate, so a
    //  band's bases are not overwritten while the previous band's are still being read)
    const uint2* in_bases = in + ((size_t)in_mask + 1) + (first_local ? (size_t)((band - 1) & 3) << (in_shift - 2) : 0);
    uint2* out_bases = out + ((size_t)out_mask + 1) + (last_local ? (size_t)(band & 3) << (out_shift - 2) : 0);
    const unsigned inb_mask = first_local ? (in_mask >> 2) : in_mask, outb_mask = last_local ? (out_mask >> 2) : out_mask;

    // ---- table ring: everything pad, then T positions [0, 32)
    w.sync();
#pragma unroll
    for (int k = 0; k < 2 * kTabRing / 32; ++k) sm->tab[k * 32 + lane] = padw;
    w.sync();
    {
      const int q = lane;
      uint32_t c = 4;
      if (q < LT) c = (uint32_t)(SWB_T_PACKED[q >> 5] >> (2 * (q & 31))) & 3u;
      const uint32_t tw = table_word(c, padw, flip);
      sm->tab[q & (kTabRing - 1)] = tw;
      sm->tab[(q & (kTabRing - 1)) + kTabRing] = tw;
    }
    // ---- loads issued one chunk ahead of their use: the packed T word of positions [32,64) and a
    //      speculative read of this lane's first boundary entry (and, re-based mode, of its producer's base)
    uint64_t twpref = (kChunk + lane < LT) ? ld_early_u64(SWB_T_PACKED + ((kChunk + lane) >> 5)) : 0ull;
    uint2 epref = make_uint2(0u, 0u), bpref = make_uint2(0u, 0u);
    bool live = !zero_src;             // warp-uniform: top boundary entries are expected (false: zero border, or after a timeout)
    bool tma_inflight = false;         // TMA flavour: a bulk copy for the next chunk has been issued
    if (live && SLACK + lane < LT) {
      const long long j = in_base + SLACK + lane + SKEW;
      epref = ld_entry(in + (j & in_mask));
      if (RB) bpref = ld_entry(in_bases + ((j >> 8) & inb_mask));
    }
    if (SLACK && live) {
      // With the slack step lane 0 consumes at step i what was shuffled at step i-1; nothing is shuffled before
      // step 0, so the boundary value of T position 0 is handed to lane 0 here.  (Every band starts with base 0,
      // so no translation is needed in re-based mode.)
      const long long j0 = in_base + SKEW;
      const uint32_t v0 = wait_entry(P, w, true, in + (j0 & in_mask), in_tag | ((uint32_t)(j0 >> in_shift) & 0xFFu),
                                     ld_entry(in + (j0 & in_mask)), wt);
      if (lane == 0) yold = v0;
      live = !wt.aborted;
    }
#ifdef SWB_ENABLE_PROF
    long long prof_pro = 0, prof_steps = 0, prof_polls = 0, prof_chunks = 0;
#if SWB_DEVICE_CODE
    if (P.prof && lane == 31 && P.prof[8 * lw + 4] == 0) {
      unsigned long long gt; unsigned smid;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      P.prof[8 * lw + 4] = (long long)gt; P.prof[8 * lw + 6] = (long long)smid;
    }
#endif
#endif

    for (int i8 = 0; i8 < nsteps; i8 += kBlock) {
      // ================= once per block of 256 steps =================
      // (a') re-based mode: re-centre the registers around the live score level
      if (RB) {
        if (i8 > 0) {
          uint32_t mxw = Ho[0], mnw = Ho[0];
#pragma unroll
          for (int r = 1; r < R; ++r) { mxw = max16x2(mxw, Ho[r]); mnw = min16x2(mnw, Ho[r]); }
          const int mx = w.reduce_max(hi_half_max(mxw));
          const int mn = -w.reduce_max(-lo_half_min(mnw));
          if (mx - mn > 20000) atomic_or_i32(P.result + 1, STATUS_REBASE_RANGE);   // never seen; host repeats in 32 bit
          int delta = (mx > kRebaseTrigger || mn < -kRebaseTrigger) ? (mx + mn) / 2 : 0;
          if (base + delta < 0) delta = -base;
          if (delta != 0) {                                               // warp-uniform
            const int b = hi_half_max(max16x2(best0, best1)) + base;
            best_abs = best_abs > b ? best_abs : b;
            best0 = best1 = pack2(-32768);
            const uint32_t dw = pack2(-delta);
#pragma unroll
            for (int r = 0; r < R; ++r) { Ho[r] = add16x2(Ho[r], dw); E[r] = add16x2(E[r], dw); }
            // up_prev / yold may hold the stand-in for a boundary value that does not exist (T positions beyond LT,
            // -30000 - open once the base is high): clamp before shifting, or a rising base wraps it around to a huge
            // positive value (seen on a 4 M x 4 M pair whose LT is a multiple of the block: score 483 137 for 456 586)
            const uint32_t lowc = pack2(delta > 2768 ? -30000 + delta : -32768);
            Fbot = add16x2(Fbot, dw); xsend = add16x2(xsend, dw);
            up_prev = add16x2(max16x2(up_prev, lowc), dw); yold = add16x2(max16x2(yold, lowc), dw);
            if (HS) { HoLast_d = add16x2(HoLast_d, dw); Fbot_d = add16x2(Fbot_d, dw); }
            base += delta;
            floorw = pack2(-base > -30000 ? -base : -30000);
          }
        }
        // tell the band below which base the entries of this block are relative to
        if (emit) st_entry(out_bases + (((out_base + i8) >> 8) & outb_mask), (uint32_t)base,
                           out_tag | ((uint32_t)(((out_base + i8) >> 8) >> out_shift) & 0xFFu));
      }
      // Re-based lanes far above zero: the clamp at the zero floor cannot bind (floorw is then the stand-in -30000, and
      // every live value is within +-20000 of the base or the range check above fires and the host repeats in 32 bit),
      // so this block's steps run without it.  Every band starts at base 0, i.e. with the clamp.
      // (linear-gap kernels only: measured -3.6 % on cfg3; the affine kernel got 3 % SLOWER with a second copy of its larger loop.
      //  And only in the fewest-instructions row loop of two warps per scheduler: in the short-chain loop the clamp rides on a
      //  VIMNMX3 and dropping it saves a VIADD on the idle pipe, while the second copy of the loop costs a single warp its
      //  instruction cache -- the 8-GPU ring, one warp per scheduler, went from 375 to 448 ms on the ranks whose bands sit above 30000)
      const bool nofloor = RB && MODE == 1 && !SHORT && base > 30000 && !(P.dbg & 4);
      // every boundary entry of the steps before this block has been read: tell the producer (ring back-pressure)
      if (lane == 0) st_progress(my_progress, (unsigned long long)(sbase + i8 + SLACK));
      // (c) ring back-pressure: never overwrite an entry the consumer has not read yet
      if (check_sink && ((sbase + i8) & 1023) == 0 && sbase + i8 + 1024 > (long long)out_mask + 1) {
        const unsigned long long need = (unsigned long long)(sbase + i8 + 1024 - ((long long)out_mask + 1));
        wait_progress(P, w, sink_progress, need, band, i8, wt);
      }

      for (int i0 = i8; i0 < i8 + kBlock; i0 += kChunk) {
        // ================= once per chunk of 32 steps: straight-line code =================
#if defined(SWB_ENABLE_PROF) && SWB_DEVICE_CODE
        const long long tp0 = clock64();
        const long long bud0 = wt.budget;
#endif
        // this chunk's tables were stored a chunk ago: start the first table load now, its latency hides behind the
        // prologue instead of standing in front of the first step
        const uint32_t* tabp = sm->tab + ((i0 - SK * lane) & (kTabRing - 1));
        uint32_t Tnext = tabp[0];
        // (a) substitution tables for T positions [i0+32, i0+64); fetch the word after that
        {
          const int q = i0 + kChunk + lane;
          uint32_t c = 4;
          if (q < LT) c = (uint32_t)(twpref >> (2 * (q & 31))) & 3u;
          const uint32_t tw = table_word(c, padw, flip);
          sm->tab[q & (kTabRing - 1)] = tw;
          sm->tab[(q & (kTabRing - 1)) + kTabRing] = tw;
          twpref = (q + kChunk < LT) ? ld_early_u64(SWB_T_PACKED + ((q + kChunk) >> 5)) : 0ull;
        }
        // (b) top boundary for lane 0's positions [i0+SLACK, i0+SLACK+32): normally already here (loaded half a
        //     chunk ago); one vote decides whether the out-of-line poll loop is needed
        const int q = i0 + SLACK + lane;
        const long long j = in_base + q + SKEW;                           // producer step that emitted q
        const bool need = live && q < LT;
#if SWB_DEVICE_CODE
        if constexpr (TMA) if (tma_inflight) {                            // warp-uniform
          const int b = (i0 / kChunk) & 1;
          unsigned long long* bar = &sm->mbar[b];
          const uint32_t ph = b ? tma_phase1 : tma_phase0;
          while (!mbar_try_wait(bar, ph)) {}
          if (b) tma_phase1 ^= 1u; else tma_phase0 ^= 1u;
          const uint32_t s0 = (uint32_t)((in_base + i0 + SLACK + SKEW) & in_mask);
          epref = sm->raw[b][lane + (s0 & 1u)];
          tma_inflight = false;
        }
#endif
        {
          const uint32_t want = in_tag | ((uint32_t)(j >> in_shift) & 0xFFu);
          const long long bj = j >> 8;
          const uint32_t bwant = in_tag | ((uint32_t)(bj >> in_shift) & 0xFFu);
          const bool ok = !need || (epref.y == want && (!RB || bpref.y == bwant));
          if (!w.all(ok)) {                       // rare: out of line; the entries are re-read here once they are valid
            wt.budget = poll_boundary(P, w, need, in + (j & in_mask), want, in_bases + (bj & inb_mask), bwant, RB, wt.budget);
            if (wt.budget < 0) { wt.aborted = true; live = false; }
            else if (need) { epref = ld_entry(in + (j & in_mask)); if (RB) bpref = ld_entry(in_bases + (bj & inb_mask)); }
          }
          uint32_t v = RB ? add16x2(nopen, floorw) : nopen;
          if (need && live) {
            v = epref.x;
            if (RB) {                  // translate from the producer's base (published once per block) into ours
              const int diff = (int)bpref.x - base;
              if (diff > 30000 || diff < -30000) atomic_or_i32(P.result + 1, STATUS_REBASE_RANGE);
              v = add16x2(v, pack2(diff));
            }
          }
          sm->inbox[q & (kInbox - 1)] = v;
          sm->inbox[(q & (kInbox - 1)) + kInbox] = v;
        }
        // next chunk's entry: loaded speculatively half a chunk from now (between the two step loops)
        const bool spec = live && q + kChunk < LT;
        const uint2* spec_e = in + ((j + kChunk) & in_mask);
        const uint2* spec_b = in_bases + (((j + kChunk) >> 8) & inb_mask);
        w.sync();
#if defined(SWB_ENABLE_PROF) && SWB_DEVICE_CODE
        const long long tp1 = clock64();
#endif

        const uint32_t* inbp = sm->inbox + ((i0 + SLACK) & (kInbox - 1));
        uint2* outp = out + ((out_base + i0) & out_mask);
        const uint32_t otag = out_tag | ((uint32_t)((out_base + i0) >> out_shift) & 0xFFu);

        uint32_t xnext = inbp[0];                        // loaded one step ahead of use (like Tnext)
        // FLOORC: std::true_type = clamp at the zero floor (-base in re-based lanes), std::false_type = re-based lanes
        // whose base is so high that the floor cannot bind (see `nofloor` above): one instruction less per row
        auto step = [&](const int k, auto FLOORC) {
          constexpr bool FL = decltype(FLOORC)::value;
          const uint32_t Tlo = Tnext;
          const uint32_t xin = xnext;
          Tnext = tabp[k + 1];
          xnext = inbp[k + 1];
          const uint32_t xs = last_lane ? xin : xsend;
          const uint32_t ynew = w.shfl(xs, src_lane);
          const uint32_t yuse = SLACK ? yold : ynew;
          yold = ynew;
          // what the hi sub-lane sees above it: the lo sub-lane's bottom row after the previous step (HS 0) or after
          // the step before that (HS 1); likewise its table word
          const uint32_t lo_bottom = HS ? HoLast_d : Ho[R - 1];
          const uint32_t lo_bottom_f = HS ? Fbot_d : Fbot;
          const uint32_t Thi_use = HS ? Thi_d : Thi;
          if (HS) { HoLast_d = Ho[R - 1]; Fbot_d = Fbot; Thi_d = Thi; }
          uint32_t upHo, F;
          if (MODE == 0) {
            upHo = prmt(yuse, lo_bottom, 0x5410u);   // lo <- neighbour's bottom (H-open), hi <- own lo bottom
            F = prmt(yuse, lo_bottom_f, 0x5432u);    // lo <- neighbour's bottom F,      hi <- own lo bottom F
          } else {
            upHo = prmt(yuse, lo_bottom, 0x5432u);   // linear mode ships the whole H-open word
            F = 0;
          }
          uint32_t diag = up_prev;
          up_prev = upHo;
          if (SHORT) {
            // Row loop with ONE dependent instruction per row (used with one warp per scheduler, where the
            // dependency chain and not the issue rate limits a step).  With m = max(diag + s, E, 0):
            //   F[r]  = max(F[r-1] - min(ext, open), m[r-1] - open)   because H[r-1] = max(m[r-1], F[r-1]);
            //   Ho[r] = H[r] - open = max(m[r], F[r]) - open.
            // Only F (affine) or H (linear) is carried from row to row; everything else depends on the previous
            // column alone.  Row 0 takes the true neighbour values (upHo, F) and the plain recurrence.
            uint32_t X = upHo, hprev = 0;
#pragma unroll
            for (int r = 0; r < R; ++r) {
              const uint32_t s = prmt(Tlo, Thi_use, sel[r]);
              const uint32_t old = Ho[r];
              uint32_t h;
              if (MODE == 0) {
                E[r] = addmax16x2(E[r], next, old);
                const uint32_t m = RB ? (FL ? max16x2(addmax16x2(diag, s, E[r]), floorw) : addmax16x2(diag, s, E[r])) : addmaxrelu16x2(diag, s, E[r]);
                F = addmax16x2(F, r == 0 ? next : fnext, X);
                X = add16x2(m, nopen);
                h = max16x2(m, F);
              } else if (RB) {
                const uint32_t t = FL ? max3_16x2(add16x2(diag, s), old, floorw) : addmax16x2(diag, s, old);
                h = r == 0 ? max16x2(t, X) : addmax16x2(hprev, nopen, t);
              } else {
                const uint32_t t = addmax16x2(diag, s, old);
                h = r == 0 ? maxrelu16x2(t, X) : addmaxrelu16x2(hprev, nopen, t);
              }
              hprev = h;
              Ho[r] = add16x2(h, nopen);
              diag = old;
              if (r & 1) best1 = max16x2(best1, h); else best0 = max16x2(best0, h);
            }
          } else {
            // Fewest instructions per row (used with two warps per scheduler, where the issue rate is the limit).
            uint32_t Hup = upHo;
#pragma unroll
            for (int r = 0; r < R; ++r) {
              const uint32_t s = prmt(Tlo, Thi_use, sel[r]);
              const uint32_t d = add16x2(diag, s);
              const uint32_t old = Ho[r];
              uint32_t h;
              if (MODE == 0) {
                E[r] = addmax16x2(E[r], next, old);
                F = addmax16x2(F, next, Hup);
                h = RB ? (FL ? max16x2(max3_16x2(d, E[r], F), floorw) : max3_16x2(d, E[r], F)) : max3relu16x2(d, E[r], F);
              } else {
                // non-RB: the clamp at 0 rides on the fused add-max, the second max is the plain full-rate VIMNMX
                h = RB ? (FL ? max16x2(max3_16x2(d, old, Hup), floorw) : max16x2(addmax16x2(diag, s, old), Hup)) : max16x2(addmaxrelu16x2(diag, s, old), Hup);
              }
              Ho[r] = add16x2(h, nopen);
              Hup = Ho[r];
              diag = old;
              if (r & 1) best1 = max16x2(best1, h); else best0 = max16x2(best0, h);
            }
          }
          Fbot = F;
          xsend = (MODE == 0) ? prmt(Ho[R - 1], Fbot, 0x7632u) : Ho[R - 1];
          Thi = Tlo;
          // slot = producer step (always in range); steps whose T position is outside [0,LT) are never read
          if (emit) st_entry(outp + k, xsend, otag);
        };
        // Two sequential half-chunk loops (not a nested one: that cost more in code generation than it saved) with
        // the speculative boundary loads of the next chunk in between: the band above only has to be
        // SKEW + 1.5 chunks ahead instead of SKEW + 2 chunks.
        auto mid_chunk = [&]() {
#if SWB_DEVICE_CODE
        if constexpr (TMA) {
          // one bulk copy for the whole next chunk: entries a0 .. a0+33 of the ring (a0 even: 16-byte aligned), split in
          // two when the 34 entries run over the end of the ring (ring lengths are even, so both parts stay 16-byte multiples)
          if (live && i0 + kChunk + SLACK < LT) {                         // warp-uniform: lane 0's next entry exists
            const int b = ((i0 / kChunk) + 1) & 1;
            if (lane == 0) {
              const uint32_t s0 = (uint32_t)((in_base + i0 + kChunk + SLACK + SKEW) & in_mask);
              const uint32_t a0 = s0 & ~1u;
              const uint32_t ring_len = in_mask + 1u;
              const uint32_t n1 = (a0 + (kChunk + 2) <= ring_len) ? (uint32_t)(kChunk + 2) : ring_len - a0;
              mbar_expect_tx(&sm->mbar[b], (kChunk + 2) * 8u);
              bulk_g2s(&sm->raw[b][0], in + a0, n1 * 8u, &sm->mbar[b]);
              if (n1 < (uint32_t)(kChunk + 2)) bulk_g2s(&sm->raw[b][n1], in, ((kChunk + 2) - n1) * 8u, &sm->mbar[b]);
            }
            tma_inflight = true;
          }
        } else
#endif
        if (spec) epref = ld_entry(spec_e);
        if (RB && spec) bpref = ld_entry(spec_b);
        };
        if (RB && MODE == 1 && !SHORT && nofloor) {   // warp-uniform, constant over a block of 256 steps
#pragma unroll (kU)
          for (int k = 0; k < kChunk / 2; ++k) step(k, std::false_type{});
          mid_chunk();
#pragma unroll (kU)
          for (int k = kChunk / 2; k < kChunk; ++k) step(k, std::false_type{});
        } else {
#pragma unroll (kU)
          for (int k = 0; k < kChunk / 2; ++k) step(k, std::true_type{});
          mid_chunk();
#pragma unroll (kU)
          for (int k = kChunk / 2; k < kChunk; ++k) step(k, std::true_type{});
        }
#if defined(SWB_ENABLE_PROF) && SWB_DEVICE_CODE
        { const long long tp2 = clock64(); prof_pro += tp1 - tp0; prof_steps += tp2 - tp1; prof_polls += bud0 - wt.budget; prof_chunks += 1; }
#endif
      }
    }
#if defined(SWB_ENABLE_PROF) && SWB_DEVICE_CODE
    if (P.prof && lane == 31) {
      long long* pr = P.prof + 8 * lw;
      pr[0] += prof_pro; pr[1] += prof_steps; pr[2] += prof_polls; pr[3] += prof_chunks;
      if (pr[5] == 0) { unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); pr[5] = (long long)gt; }
    }
#endif
    if (RB) {
      const int b = hi_half_max(max16x2(best0, best1)) + base;
      best_abs = best_abs > b ? best_abs : b;
    }
    if (lane == 0) st_progress(my_progress, (unsigned long long)(sbase + nsteps));
  }

  // ---- running best: halves -> int, warp max, one atomic
  const int m = w.reduce_max(RB ? best_abs : hi_half_max(max16x2(best0, best1)));
  if (lane == 0) {
    atomic_max_i32(P.result, m);
    if (!RB && m > 32767 - P.match - 1) atomic_or_i32(P.result + 1, STATUS_S16_OVERFLOW);
  }
}

#undef SWB_T_PACKED

// =================================================================================================
//  32-bit engine (scores beyond the s16 range): one sub-lane per thread, band = 32*R rows.
//  Boundary entries come in pairs: slot 2j = H-open, slot 2j+1 = F.
// =================================================================================================
//  GEN: any byte alphabet (the reference compares raw bytes, main.cpp:28-33): the table ring holds the raw T byte
//  and the substitution score is a compare + select instead of a PRMT table look-up.
//  TRACK: also report WHERE the maximum is (SURVEY.md 8(f) row 4; the reference is score-only).  The running best
//  becomes a key  H << 11 | (127 - step mod 128) << 4 | (15 - row in lane):  one max keeps the highest H and,
//  among equals, the earliest step (= smallest T position for a lane) and then the smallest row; which 128-step
//  window the key belongs to is noted once per chunk, when the lane's best H has grown.  Per band the warp
//  reduces (max H, min T position, min Q row) into P.cand; the host reduces the bands by the same rule.
//  Needs H < 2^20 and R <= 16.
//  ANCH (with TRACK): the ANCHORED recurrence -- every alignment starts at cell (0,0), H is not clamped at 0, the
//  borders carry the gap costs (row 0: H(0,j) = -(open + (j-1)*min(ext, open)), column 0 likewise, E/F = -inf
//  there).  Run on the reversed prefixes that end at the best alignment's end cell, the position of the maximum
//  is that alignment's START cell.  Only lane 0 of a band starts with the column-0 border in its registers; the
//  other lanes start at -inf (they are still left of column 0) and build column 0 from the F values arriving from
//  above, which is exactly the recurrence of that column.
//  DIRS (with ANCH, round 2): also record, for every cell, where its H, E and F came from (4 bits per cell, one 32-bit
//  word per lane and step for R = 8) -- the traceback matrix of the GLOBAL alignment between the start and the end
//  cell that swb200_score_span found; walk_block (swb_traceback.cuh) follows it back.  Uses the plain row loop
//  (E and F exactly as in main.cpp:57-58, no short-chain rewriting), so the flags mean what they say.
template <int R, int SLACK, bool GEN = false, bool SHORT = true, bool TRACK = false, bool ANCH = false, bool DIRS = false>
SWB_HD void engine_warp_s32(const EngineParams& P, const WarpCtx& w, int lw, WarpSmem* sm) {
  static_assert(!DIRS || (ANCH && !SHORT && !TRACK && R <= 8), "direction recording: anchored recurrence, plain row loop, 8 rows per lane");
  constexpr int SK = 1 + SLACK;
  constexpr int SKEW = 31 * SK;
  constexpr int kU = step_unroll(8.0, R, kStepUnroll32);
  const int lane = w.lane;
  const bool last_lane = lane == 31;
  const int src_lane = (lane + 31) & 31;
  const int nopen = -P.gap_init, next = -P.gap_ext;
  const int fnext = -(P.gap_ext < P.gap_init ? P.gap_ext : P.gap_init);   // F carried down inside a lane
  constexpr int NEG = -(1 << 29);                                         // ANCH: "minus infinity" (no s32 overflow within 2^21 steps)
  const uint32_t padb = (uint32_t)(P.mismatch + P.gap_init) & 0xFFu;
  const uint32_t padw = GEN ? 0x200u : padb * 0x01010101u;       // GEN: 0x200 equals no byte and no pad row (0x100)
  const uint32_t flip = padb ^ ((uint32_t)(P.match + P.gap_init) & 0xFFu);
  const int s_match = P.match + P.gap_init, s_mismatch = P.mismatch + P.gap_init;
  const int LT = (int)P.LT;            // step arithmetic is 32-bit (the host refuses LT >= 2^30); only ring indices,
                                       // which count steps over all rounds, are 64-bit
  const int nsteps = ((LT + SKEW + kChunk - 1) / kChunk) * kChunk;
  int best0 = 0, best1 = 0;
  Waiter wt{P.spin_limit, false};

  for (long long band = P.ring_offset + lw; band < P.NB; band += P.ring_total) {
    const bool zero_src = band == 0 || (P.dbg & 2);
    const bool is_final = band == P.NB - 1 && P.final_out != nullptr;   // its bottom row is wanted by the caller
    const bool has_sink = band + 1 < P.NB || is_final;
    const bool emit = has_sink && last_lane && !(P.dbg & 1);
    const bool first_local = lw == 0, last_local = lw == P.warps_local - 1 || is_final;   // "last": full-length stream, no back-pressure
    const uint2* in = first_local ? P.ext_in : P.links + (size_t)(lw - 1) * 2 * ((size_t)P.link_mask + 1);
    const unsigned in_mask = first_local ? P.ext_mask : P.link_mask;
    const int in_shift = first_local ? P.ext_shift : P.link_shift;
    uint2* out = is_final ? P.final_out : (last_local ? P.ext_out : P.links + (size_t)lw * 2 * ((size_t)P.link_mask + 1));
    const unsigned out_mask = is_final ? P.final_mask : (last_local ? P.ext_mask : P.link_mask);
    const int out_shift = last_local ? P.ext_shift : P.link_shift;
    const uint32_t in_tag = (first_local ? P.ext_tag_base : P.tag_base) | ((uint32_t)band << 8);
    const uint32_t out_tag = (last_local ? P.ext_tag_base : P.tag_base) | ((uint32_t)(band + 1) << 8);
    unsigned long long* my_progress = P.progress + lw;
    const unsigned long long* sink_progress = P.progress + lw + 1;
    // Inner rings are indexed by the CUMULATIVE producer step over all rounds (sbase + step), so a
    // ring is one continuous stream and back-pressure spans band boundaries; the full-length ext
    // stream restarts at 0 every band (safe: see DESIGN.md, hand-off protocol).  Rounds count from
    // ring_offset: a blocked traceback launch (swb200_align) runs the band window [ring_offset, NB) on
    // one GPU, and a producer and its consumer must agree on the round whatever the window's first band.
    // (Every other launch has ring_offset + lw < ring_total, where this is band / ring_total.)
    const long long sbase = ((band - P.ring_offset) / P.ring_total) * (long long)nsteps;
    const long long in_base = first_local ? 0 : sbase, out_base = last_local ? 0 : sbase;

    uint32_t sel[R];
    {
      const long long row0 = band * (32LL * R) + (long long)lane * R;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const long long a = row0 + r;
        sel[r] = GEN ? (a < P.LQ ? (uint32_t)P.q_codes[a] : 0x100u) : mk_sel32(a < P.LQ ? P.q_codes[a] : 4u);
      }
    }
    int Ho[R], E[R];
#pragma unroll
    for (int r = 0; r < R; ++r) { Ho[r] = nopen; E[r] = nopen; }
    int up_prev = nopen, xsH = nopen, xsF = nopen, yoldH = nopen, yoldF = nopen;
    if (ANCH) {
      // column 0 of the anchored matrix: H(i,0) = -(open + (i-1)*gmin) for i >= 1, H(0,0) = 0, E = -inf
      const long long i_first = band * (32LL * R) + 1;            // 1-based row of lane 0's first row
#pragma unroll
      for (int r = 0; r < R; ++r) {
        Ho[r] = lane == 0 ? (int)(nopen + (i_first + r - 1) * fnext) + nopen : NEG;
        E[r] = NEG;
      }
      const int h_above = i_first == 1 ? 0 : (int)(nopen + (i_first - 2) * fnext);     // H(i_first - 1, 0)
      up_prev = lane == 0 ? h_above + nopen : NEG;
      xsH = lane == 0 ? Ho[R - 1] : NEG;
      xsF = lane == 0 ? Ho[R - 1] - nopen : NEG;                  // F(i,0) = H(i,0) in column 0
      yoldH = (lane == 0 && zero_src) ? nopen + nopen : NEG;      // band 0: H(0,1) - open; later bands: set by the wait below
      yoldF = NEG;
    }
    int bestkey = 0, rec_h = 0, rec_key = 0;         // TRACK only
    int rec_win = 0;

    w.sync();
#pragma unroll
    for (int k = 0; k < 2 * kTabRing / 32; ++k) sm->tab[k * 32 + lane] = padw;
    w.sync();
    {
      const int q = lane;
      uint32_t tw;
      if (GEN) tw = q < LT ? (uint32_t)P.t_bytes[q] : padw;
      else {
        uint32_t c = 4;
        if (q < LT) c = (uint32_t)(P.t_packed[q >> 5] >> (2 * (q & 31))) & 3u;
        tw = table_word(c, padw, flip);
      }
      sm->tab[q & (kTabRing - 1)] = tw;
      sm->tab[(q & (kTabRing - 1)) + kTabRing] = tw;
    }
    uint64_t twpref = GEN ? (kChunk + lane < LT ? (uint64_t)P.t_bytes[kChunk + lane] : (uint64_t)padw)
                          : ((kChunk + lane < LT) ? ld_early_u64(P.t_packed + ((kChunk + lane) >> 5)) : 0ull);
    uint2 eprefH = make_uint2(0u, 0u), eprefF = make_uint2(0u, 0u);
    if (!zero_src && SLACK + lane < LT) {
      eprefH = ld_entry(in + 2 * ((in_base + SLACK + lane + SKEW) & in_mask));
      eprefF = ld_entry(in + 2 * ((in_base + SLACK + lane + SKEW) & in_mask) + 1);
    }
    if (SLACK && !zero_src) {      // boundary value of T position 0 for lane 0 (see the 16-bit engine)
      const long long j0 = in_base + SKEW;
      const uint32_t tg0 = in_tag | ((uint32_t)(j0 >> in_shift) & 0xFFu);
      const uint32_t h0 = wait_entry(P, w, true, in + 2 * (j0 & in_mask), tg0, ld_entry(in + 2 * (j0 & in_mask)), wt);
      const uint32_t f0 = wait_entry(P, w, true, in + 2 * (j0 & in_mask) + 1, tg0, ld_entry(in + 2 * (j0 & in_mask) + 1), wt);
      if (lane == 0) { yoldH = (int)h0; yoldF = (int)f0; }
    }

    for (int i0 = 0; i0 < nsteps; i0 += kChunk) {
      {
        const int q = i0 + kChunk + lane;
        uint32_t tw;
        if (GEN) tw = (uint32_t)twpref;
        else {
          uint32_t c = 4;
          if (q < LT) c = (uint32_t)(twpref >> (2 * (q & 31))) & 3u;
          tw = table_word(c, padw, flip);
        }
        sm->tab[q & (kTabRing - 1)] = tw;
        sm->tab[(q & (kTabRing - 1)) + kTabRing] = tw;
        if (GEN) twpref = q + kChunk < LT ? (uint64_t)P.t_bytes[q + kChunk] : (uint64_t)padw;
        else twpref = (q + kChunk < LT) ? ld_early_u64(P.t_packed + ((q + kChunk) >> 5)) : 0ull;
      }
      {
        const int q = i0 + SLACK + lane;
        uint32_t vH = (uint32_t)nopen, vF = (uint32_t)nopen;
        if (ANCH) {              // row 0 of the anchored matrix: H(0, q+1) - open, F = -inf (also beyond LT: harmless)
          vH = (uint32_t)((int)(nopen + (long long)q * fnext) + nopen);
          vF = (uint32_t)NEG;
        }
        if (!zero_src) {
          const bool need = q < LT;
          const long long j = in_base + q + SKEW;
          const uint32_t tg = in_tag | ((uint32_t)(j >> in_shift) & 0xFFu);
          const uint32_t gH = wait_entry(P, w, need, in + 2 * (j & in_mask), tg, eprefH, wt);
          const uint32_t gF = wait_entry(P, w, need, in + 2 * (j & in_mask) + 1, tg, eprefF, wt);
          if (need) { vH = gH; vF = gF; }
          if (q + kChunk < LT) {
            eprefH = ld_entry(in + 2 * ((j + kChunk) & in_mask));
            eprefF = ld_entry(in + 2 * ((j + kChunk) & in_mask) + 1);
          }
        }
        sm->inbox[q & (kInbox - 1)] = vH;
        sm->inbox[(q & (kInbox - 1)) + kInbox] = vH;
        sm->inbox[(q & (kInbox - 1)) + 2 * kInbox] = vF;
        sm->inbox[(q & (kInbox - 1)) + 3 * kInbox] = vF;
        if (lane == 0 && (i0 & 255) == 0)
          st_progress(my_progress, (unsigned long long)(sbase + i0 + SLACK + kChunk));
      }
      if (has_sink && !last_local && ((sbase + i0) & 1023) == 0 && sbase + i0 + 1024 > (long long)out_mask + 1) {
        const unsigned long long need = (unsigned long long)(sbase + i0 + 1024 - ((long long)out_mask + 1));
        wait_progress(P, w, sink_progress, need, band, i0, wt);
      }
      w.sync();

      const uint32_t* tabp = sm->tab + ((i0 - SK * lane) & (kTabRing - 1));
      const uint32_t* inbp = sm->inbox + ((i0 + SLACK) & (kInbox - 1));
      uint2* outp = out + 2 * ((out_base + i0) & out_mask);
      const uint32_t otag = out_tag | ((uint32_t)((out_base + i0) >> out_shift) & 0xFFu);

      uint32_t Tnext = tabp[0];
      int xnH = (int)inbp[0], xnF = (int)inbp[2 * kInbox];
      int cstep = ((127 - (int)(i0 & 127)) << 4) + 15;      // TRACK: low key bits of row 0 at the chunk's first step
#pragma unroll (kU)
      for (int k = 0; k < kChunk; ++k) {
        const uint32_t Tw = Tnext;
        const int xinH = xnH, xinF = xnF;
        Tnext = tabp[k + 1];
        xnH = (int)inbp[k + 1];
        xnF = (int)inbp[k + 1 + 2 * kInbox];
        const int ynewH = (int)w.shfl((uint32_t)(last_lane ? xinH : xsH), src_lane);
        const int ynewF = (int)w.shfl((uint32_t)(last_lane ? xinF : xsF), src_lane);
        const int upHo = SLACK ? yoldH : ynewH;
        int F = SLACK ? yoldF : ynewF;
        yoldH = ynewH; yoldF = ynewF;
        int diag = up_prev;
        up_prev = upHo;
        if (SHORT) {     // one dependent instruction per row (F only), as in engine_warp_s16
          int X = upHo;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const int s = GEN ? (sel[r] == Tw ? s_match : s_mismatch) : (int)prmt(Tw, 0u, sel[r]);
            const int old = Ho[r];
            E[r] = addmax32(E[r], next, old);
            const int m = ANCH ? addmax32(diag, s, E[r]) : addmaxrelu32(diag, s, E[r]);
            F = addmax32(F, r == 0 ? next : fnext, X);
            X = m + nopen;
            const int h = m > F ? m : F;
            Ho[r] = h + nopen;
            diag = old;
            if (TRACK) { const int key = (ANCH ? (h > 0 ? h : 0) : h) * 2048 + (cstep - r); bestkey = bestkey > key ? bestkey : key; }
            else if (r & 1) best1 = best1 > h ? best1 : h; else best0 = best0 > h ? best0 : h;
          }
        } else {
          int Hup = upHo;
          uint32_t dword = 0;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const int s = GEN ? (sel[r] == Tw ? s_match : s_mismatch) : (int)prmt(Tw, 0u, sel[r]);
            const int d = diag + s;
            const int old = Ho[r];
            const int e_ext = E[r] + next, f_ext = F + next;
            E[r] = addmax32(E[r], next, old);
            F = addmax32(F, next, Hup);
            const int h = ANCH ? max3_32(d, E[r], F) : max3relu32(d, E[r], F);
            if (DIRS) {
              // ties: diagonal before E before F; a gap counts as extended only if extending is strictly better
              const uint32_t src = h == d ? 0u : (h == E[r] ? 1u : 2u);
              dword |= (src | (e_ext > old ? 4u : 0u) | (f_ext > Hup ? 8u : 0u)) << (4 * r);
            }
            Ho[r] = h + nopen;
            Hup = Ho[r];
            diag = old;
            if (TRACK) { const int key = (ANCH ? (h > 0 ? h : 0) : h) * 2048 + (cstep - r); bestkey = bestkey > key ? bestkey : key; }
            else if (r & 1) best1 = best1 > h ? best1 : h; else best0 = best0 > h ? best0 : h;
          }
          if (DIRS) P.dirs[((size_t)(band - P.ring_offset) * (size_t)nsteps + (size_t)(i0 + k)) * 32 + lane] = dword;   // window-relative band
        }
        if (TRACK) cstep -= 16;
        xsH = Ho[R - 1];
        xsF = F;
        if (emit) {
          st_entry(outp + 2 * k, (uint32_t)xsH, otag);
          st_entry(outp + 2 * k + 1, (uint32_t)xsF, otag);
        }
      }
      if (TRACK) {                                     // once per chunk: has this lane's best H grown?
        const int hb = bestkey >> 11;
        const bool upd = hb > rec_h;
        rec_h = upd ? hb : rec_h;
        rec_key = upd ? bestkey : rec_key;
        rec_win = upd ? (i0 & ~127) : rec_win;
      }
    }
    if (TRACK) {
      // this lane's first best cell: step -> T position (lane l is SK*l positions behind lane 0), row in Q
      const int step = rec_win + 127 - ((rec_key >> 4) & 127);
      const int pos = step - SK * lane;
      const int row = (int)(band * (32LL * R) + (long long)lane * R + (15 - (rec_key & 15)));
      const int hmax = w.reduce_max(rec_h);
      const int pmin = -w.reduce_max(rec_h == hmax ? -pos : -0x7fffffff);
      const int rmin = -w.reduce_max((rec_h == hmax && pos == pmin) ? -row : -0x7fffffff);
      if (lane == 0) { P.cand[3 * band] = hmax; P.cand[3 * band + 1] = pmin; P.cand[3 * band + 2] = rmin; }
      best0 = best0 > hmax ? best0 : hmax;
      bestkey = 0; rec_h = 0; rec_key = 0; rec_win = 0;
    }
    if (lane == 0) st_progress(my_progress, (unsigned long long)(sbase + nsteps));
  }
  int m = w.reduce_max(best0 > best1 ? best0 : best1);
  if (lane == 0) atomic_max_i32(P.result, m);
}

// rows of Q one band covers
// modes 2, 5, 6, 7 run 32-bit lanes (6, 7 = 2, 5 with end-cell tracking)
SWB_HD bool mode_is_s32(int mode) { return mode == 2 || mode >= 5; }      // 8, 9 = 6, 7 with the anchored recurrence; 10, 11 = anchored + traceback directions
SWB_HD int rows_per_band(int R, int mode) { return (mode_is_s32(mode) ? 32 : 64) * R; }

}  // namespace swb
