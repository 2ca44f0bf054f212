// align_blocks_emu.cu -- runs the product's blocked traceback (swb200_align, csrc/swb_traceback.cuh) on CPU threads.
//
// TEST TOOL ONLY.  The mode-10 direction kernel body (engine_warp_s32 with the anchored recurrence and direction
// recording), the checkpoint hand-over (retag_slot) and the walk (walk_block) are __host__ __device__; this program runs
// them the way the host code of swb200_align does, with one pthread per lane as tests/emu/engine_emu.cu does:
//   1. the whole span in one launch, then the one-block walk;
//   2. the span in blocks of K rows: a forward sweep, one launch per block over the band window of the block, each
//      block's last band leaving its bottom row in a checkpoint that the next launch reads; then the walk from the last
//      block up, every block but the last recomputed from its checkpoint over the columns left of the walk.
// It prints the score of both, how many direction nibbles of the blocked launches differ from the one-launch nibble of
// the same cell, whether both walks wrote the same operations, and the blocked walk's operations (first operation
// first).  tests/test_align_blocks_emu.py checks them against the oracle.  Nothing here is linked into libswb200.so.
//
// usage: align_blocks_emu qfile tfile slack warps block_rows match mismatch gap_init gap_ext
//        qfile: seq2's span (rows, striped), tfile: seq1's span (columns, streamed), raw ASCII bytes over {A,C,G,T}
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <string>
#include <thread>
#include <vector>
#include "../../concurrentproject_b200/csrc/swb_traceback.cuh"

using namespace swb;

#if !SWB_DEVICE_CODE   // host pass only; the device pass of nvcc sees an empty translation unit

static std::vector<uint8_t> read_file(const char* path) {
  std::vector<uint8_t> v;
  FILE* f = fopen(path, "rb");
  if (!f) { fprintf(stderr, "cannot open %s\n", path); exit(2); }
  uint8_t buf[65536]; size_t n;
  while ((n = fread(buf, 1, sizeof buf, f)) > 0) v.insert(v.end(), buf, buf + n);
  fclose(f);
  return v;
}

template <int SLACK>
static void run_lane(const EngineParams* P, WarpShared* ws, int lane, int lw, WarpSmem* sm) {
  WarpCtx w{lane, ws};
  engine_warp_s32<8, SLACK, false, false, false, true, true>(*P, w, lw, sm);   // mode 10 (swb_kernels.cuh)
}

struct Geometry {
  long long LQ, LT, NB, nsteps, ext_len;
  int slack, skew, ext_shift;
};

static Geometry geometry(long long LQ, long long LT, int slack) {
  Geometry g{};
  g.LQ = LQ; g.LT = LT; g.slack = slack; g.skew = 31 * (1 + slack);
  g.NB = (LQ + kDirBandRows - 1) / kDirBandRows;
  g.nsteps = ((LT + g.skew + kChunk - 1) / kChunk) * kChunk;
  g.ext_len = 1; g.ext_shift = 0;
  while (g.ext_len < g.nsteps + kChunk || g.ext_shift < 4) { g.ext_len <<= 1; ++g.ext_shift; }
  return g;
}

struct Launch {
  std::vector<uint32_t> dirs;   // window-relative bands, nsteps steps each
  long long band0, nsteps;
  int score, status;
};

// One launch over the bands [band0, band1) and the T positions [0, LT), as run_once does it for a DirBlock:
// `warps` warps, ring_offset = band0, NB = band1, a fresh epoch; top: checkpoint row above band0, bottom: where band1 - 1
// leaves its bottom row.
static Launch launch(const uint8_t* q, const uint64_t* t, long long LQ, long long LT, int slack, int warps, long long band0,
                     long long band1, const uint2* top, uint2* bottom, unsigned epoch, const int prm[4]) {
  const Geometry g = geometry(LQ, LT, slack);
  const long long link_len = 4096;
  std::vector<uint2> links((size_t)(warps > 1 ? warps - 1 : 1) * 2 * link_len, make_uint2(0, 0));
  std::vector<uint2> ext((size_t)2 * g.ext_len, make_uint2(0, 0));
  std::vector<unsigned long long> progress((size_t)warps + 4, 0);
  int result[12] = {0};
  Launch L;
  L.band0 = band0; L.nsteps = g.nsteps;
  L.dirs.assign((size_t)(band1 - band0) * (size_t)g.nsteps * 32, 0u);
  EngineParams P{};
  P.q_codes = q; P.t_packed = t; P.LQ = LQ; P.LT = LT; P.NB = (int)band1;
  P.ring_total = warps; P.ring_offset = (int)band0; P.warps_local = warps;
  P.links = links.data(); P.link_mask = (unsigned)(link_len - 1); P.link_shift = 12;
  P.progress = progress.data();
  P.ext_in = ext.data(); P.ext_out = ext.data();
  P.ext_mask = (unsigned)(g.ext_len - 1); P.ext_shift = g.ext_shift;
  P.tag_base = epoch << 26; P.ext_tag_base = P.tag_base; P.result = result;
  P.match = prm[0]; P.mismatch = prm[1]; P.gap_init = prm[2]; P.gap_ext = prm[3];
  P.spin_limit = 200000000LL;
  P.dirs = L.dirs.data();
  if (bottom) { P.final_out = bottom; P.final_mask = (unsigned)(g.ext_len - 1); }
  if (top)
    for (long long s = g.skew; s < g.skew + LT; ++s) retag_slot(top, ext.data(), s, P.tag_base | ((uint32_t)band0 << 8));
  std::vector<WarpShared> ws((size_t)warps);
  std::vector<WarpSmem> sm((size_t)warps);
  for (auto& x : ws) pthread_barrier_init(&x.bar, nullptr, 32);
  std::vector<std::thread> th;
  for (int w = 0; w < warps; ++w)
    for (int l = 0; l < 32; ++l)
      th.emplace_back(slack ? run_lane<1> : run_lane<0>, &P, &ws[(size_t)w], l, w, &sm[(size_t)w]);
  for (auto& x : th) x.join();
  for (auto& x : ws) pthread_barrier_destroy(&x.bar);
  L.score = result[0]; L.status = result[1];
  return L;
}

static unsigned nibble(const Launch& L, long long row, long long col, int sk) {
  const long long band = row / kDirBandRows - L.band0;
  const int lane = (int)((row % kDirBandRows) / 8), r = (int)(row % 8);
  const long long step = col + (long long)sk * lane;
  return (L.dirs[(size_t)(band * L.nsteps + step) * 32 + lane] >> (4 * r)) & 0xFu;
}

// cells of the blocked launch (its bands, columns [0, ncols)) whose nibble differs from the one-launch run's
static long long differing(const Launch& whole, const Launch& blk, long long band1, long long LQ, long long ncols, int sk) {
  long long bad = 0;
  for (long long row = blk.band0 * kDirBandRows; row < band1 * kDirBandRows && row < LQ; ++row)
    for (long long col = 0; col < ncols; ++col) bad += nibble(whole, row, col, sk) != nibble(blk, row, col, sk);
  return bad;
}

int main(int argc, char** argv) {
  if (argc < 10) { fprintf(stderr, "usage: align_blocks_emu qfile tfile slack warps block_rows ma mi gi ge\n"); return 2; }
  std::vector<uint8_t> qa = read_file(argv[1]), ta = read_file(argv[2]);
  const long long LQ = (long long)qa.size(), LT = (long long)ta.size();
  const int slack = atoi(argv[3]), W = atoi(argv[4]);
  const long long K = atoll(argv[5]);
  const int prm[4] = {atoi(argv[6]), atoi(argv[7]), atoi(argv[8]), atoi(argv[9])};
  if (LQ < 1 || LT < 1 || K < kDirBandRows || K % kDirBandRows || (slack != 0 && slack != 1) || W < 1) { fprintf(stderr, "bad arguments\n"); return 2; }
  const int sk = 1 + slack;

  // ACGT -> 2-bit codes exactly as the product's encode kernels do: (c >> 1) & 3
  std::vector<uint8_t> q((size_t)LQ + 64, 4);
  for (long long k = 0; k < LQ; ++k) q[(size_t)k] = (uint8_t)((qa[(size_t)k] >> 1) & 3);
  std::vector<uint64_t> t((size_t)(LT / 32 + 8), 0);
  for (long long k = 0; k < LT; ++k) t[(size_t)(k >> 5)] |= (uint64_t)((ta[(size_t)k] >> 1) & 3) << (2 * (k & 31));
  const Geometry g = geometry(LQ, LT, slack);
  const size_t cap = (size_t)(LQ + LT + 4);
  unsigned epoch = 0;
  auto next_epoch = [&]() { epoch = epoch % 63 + 1; return epoch; };

  // 1. one launch, one-block walk
  const Launch whole = launch(q.data(), t.data(), LQ, LT, slack, W, 0, g.NB, nullptr, nullptr, next_epoch(), prm);
  std::vector<unsigned long long> ops1(cap);
  WalkState w1 = walk_start(LQ, LT);
  walk_block(whole.dirs.data(), whole.nsteps, sk, 0, w1, ops1.data(), (long long)cap);

  // 2. blocks of K rows
  const long long kb = K / kDirBandRows, B = (g.NB + kb - 1) / kb;
  std::vector<uint2> ckpt((size_t)(B > 1 ? B - 1 : 1) * 2 * (size_t)g.ext_len, make_uint2(0, 0));
  auto top_of = [&](long long b) -> const uint2* { return b > 0 ? ckpt.data() + (size_t)(b - 1) * 2 * (size_t)g.ext_len : nullptr; };
  long long bad = 0, launches = 0;
  int best = 0, status = whole.status;
  Launch last;
  for (long long b = 0; b < B; ++b) {          // forward sweep
    const long long b1 = std::min(g.NB, (b + 1) * kb);
    uint2* bottom = b + 1 < B ? ckpt.data() + (size_t)b * 2 * (size_t)g.ext_len : nullptr;
    Launch L = launch(q.data(), t.data(), LQ, LT, slack, W, b * kb, b1, top_of(b), bottom, next_epoch(), prm);
    ++launches;
    bad += differing(whole, L, b1, LQ, LT, sk);
    best = std::max(best, L.score);
    status |= L.status;
    if (b == B - 1) last = std::move(L);
  }
  std::vector<unsigned long long> ops2(cap);
  WalkState w2 = walk_start(LQ, LT);
  walk_block(last.dirs.data(), last.nsteps, sk, (B - 1) * K, w2, ops2.data(), (long long)cap);
  long long min_edge_col = LT + 1;               // smallest column at which the walk crossed a block edge
  for (long long b = B - 2; b >= 0 && !w2.done; --b) {
    min_edge_col = std::min(min_edge_col, w2.j);
    const long long b1 = std::min(g.NB, (b + 1) * kb);
    const Launch L = launch(q.data(), t.data(), LQ, w2.j, slack, W, b * kb, b1, top_of(b), nullptr, next_epoch(), prm);
    ++launches;
    bad += differing(whole, L, b1, LQ, w2.j, sk);
    status |= L.status;
    walk_block(L.dirs.data(), L.nsteps, sk, b * K, w2, ops2.data(), (long long)cap);
  }
  bool same = w1.done && w2.done && w1.nops == w2.nops;
  for (long long k = 0; same && k < w1.nops; ++k) same = ops1[(size_t)k] == ops2[(size_t)k];
  std::string cig;
  for (long long k = w2.nops - 1; k >= 0; --k)
    cig += std::to_string(ops2[(size_t)k] & 0x00FFFFFFFFFFFFFFull) + (char)(ops2[(size_t)k] >> 56);
  printf("score=%d blocked=%d status=%d blocks=%lld launches=%lld differing=%lld same_ops=%d edge_col=%lld cigar=%s\n",
         whole.score, best, status, B, launches, bad, (int)same, min_edge_col, cig.empty() ? "-" : cig.c_str());
  return 0;
}
#endif
