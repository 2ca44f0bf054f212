// align_long_emu.cu -- runs the product's long-pair batch alignment bodies (csrc/swb_align_long.cuh: long_span_pair,
// long_trace_pair) on CPU threads, two emulated warps of one pthread per lane drawing pairs from a counter, with the host
// driver's round structure (trace, then the pending pairs again with the pool emptied).  TEST TOOL ONLY.
//
// usage: align_long_emu pairs.bin ma mi gi ge slot_words pool_words ops_stride
//   pairs.bin: int32 npairs, then per pair int32 len1, int32 len2, len1 bytes, len2 bytes (A, C, G, T only).
//   Packed as the batch packer does with keep_order = 0: the shorter sequence is Q (seq1 on a tie), len1 kept.
//   slot_words / pool_words: 64-bit words (the pool gets at least the largest rectangle, as the host sizes it).
//   prints one line per pair: "score i_start j_start i_end j_end n_ops op op ..." (ops as count << 4 | op), then
//   "rounds R err E cells C"
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <thread>
#include <algorithm>
#include "../../concurrentproject_b200/csrc/swb_align_long.cuh"

using namespace swb;

#if !SWB_DEVICE_CODE

static void pack(const std::vector<uint8_t>& s, uint64_t* words) {
  for (size_t k = 0; k < s.size(); ++k) words[k >> 5] |= (uint64_t)((s[k] >> 1) & 3) << (2 * (k & 31));
}

int main(int argc, char** argv) {
  if (argc < 9) { fprintf(stderr, "usage: align_long_emu pairs.bin ma mi gi ge slot_words pool_words ops_stride\n"); return 2; }
  FILE* f = fopen(argv[1], "rb");
  if (!f) { fprintf(stderr, "cannot open %s\n", argv[1]); return 2; }
  int32_t np = 0;
  if (fread(&np, 4, 1, f) != 1) return 2;
  std::vector<std::vector<uint8_t>> q(np), t(np);
  std::vector<int> lq(np), lt(np), l1(np);
  int max_q = 0, max_t = 0;
  for (int k = 0; k < np; ++k) {
    int32_t l[2];
    if (fread(l, 4, 2, f) != 2) return 2;
    std::vector<uint8_t> a(l[0]), b(l[1]);
    if (l[0] && fread(a.data(), 1, l[0], f) != (size_t)l[0]) return 2;
    if (l[1] && fread(b.data(), 1, l[1], f) != (size_t)l[1]) return 2;
    const bool swap = l[1] < l[0];
    q[k] = swap ? b : a; t[k] = swap ? a : b;
    lq[k] = (int)q[k].size(); lt[k] = (int)t[k].size(); l1[k] = l[0];
    max_q = std::max(max_q, lq[k]); max_t = std::max(max_t, lt[k]);
  }
  fclose(f);
  const long long qs = std::max(1, (max_q + 31) / 32) + 2, ts = std::max(1, (max_t + 31) / 32) + 2;
  std::vector<uint64_t> qw((size_t)np * qs + 4, 0), tw((size_t)np * ts + 4, 0);
  for (int k = 0; k < np; ++k) { pack(q[k], &qw[(size_t)k * qs]); pack(t[k], &tw[(size_t)k * ts]); }
  const int W = 2;                                  // emulated warps
  const int ops_stride = atoi(argv[8]);
  std::vector<int> scores(np, -1), spans(4 * (size_t)np, -1), ops_count(np, -999), pending(np + 1), todo(np + 1);
  std::vector<uint32_t> ops((size_t)np * ops_stride + 1, 0);
  const long long slot_words = atoll(argv[6]);
  long long pool_words = atoll(argv[7]);
  pool_words = std::max(pool_words, (long_dir_words(max_t, max_q) + 1) / 2);   // as the host sizes it
  std::vector<uint64_t> slot((size_t)std::max(1LL, slot_words) * W), pool((size_t)std::max(1LL, pool_words));
  const long long row_stride = (std::max(max_t, 1) + 31) / 32 * 32;
  std::vector<int2> bnd((size_t)row_stride * W);
  std::vector<LongWarpSmem> sm(W);
  std::vector<uint32_t> stage((size_t)W * kLongStageLines * 32);
  unsigned long long pool_used = 0, cells = 0, next = 0;
  int npending = 0, err = 0;
  AlignBatchParams P{};
  P.q_words = qw.data(); P.t_words = tw.data(); P.q_len = lq.data(); P.t_len = lt.data(); P.len1 = l1.data();
  P.q_stride = qs; P.t_stride = ts; P.npairs = np;
  P.match = atoi(argv[2]); P.mismatch = atoi(argv[3]); P.gap_init = atoi(argv[4]); P.gap_ext = atoi(argv[5]);
  P.scores = scores.data(); P.spans = spans.data(); P.col = bnd.data(); P.row_stride = row_stride; P.next = &next;
  P.slot = slot.data(); P.slot_words = slot_words; P.pool = pool.data(); P.pool_words = pool_words; P.pool_used = &pool_used;
  P.todo = nullptr; P.ntodo = np; P.pending = pending.data(); P.npending = &npending;
  P.ops = ops.data(); P.ops_stride = ops_stride; P.ops_count = ops_count.data(); P.err = &err; P.cells = &cells;
  std::vector<WarpShared> ws(W);
  for (auto& x : ws) pthread_barrier_init(&x.bar, nullptr, 32);
  auto warps = [&](auto body) {
    std::vector<std::thread> th;
    for (int wi = 0; wi < W; ++wi)
      for (int l = 0; l < 32; ++l) th.emplace_back([&, wi, l]() { body(WarpCtx{l, &ws[wi]}, (long long)wi); });
    for (auto& x : th) x.join();
  };
  warps([&](const WarpCtx& w, long long wi) {
    long long c = 0;
    for (long long k = long_take(P, w); k < P.npairs; k = long_take(P, w)) c += long_span_pair(P, w, k, &bnd[wi * row_stride], &sm[wi]);
    align_atomic_add(P.cells, (unsigned long long)c);
  });
  int rounds = 0;
  for (;;) {
    ++rounds;
    next = 0;
    warps([&](const WarpCtx& w, long long wi) {
      long long c = 0;
      for (long long u = long_take(P, w); u < P.ntodo; u = long_take(P, w)) {
        const long long r = long_trace_pair(P, w, P.todo ? P.todo[u] : u, wi, &bnd[wi * row_stride], &sm[wi],
                                            &stage[(size_t)wi * kLongStageLines * 32]);
        c += r > 0 ? r : 0;
      }
      align_atomic_add(P.cells, (unsigned long long)c);
    });
    if (npending == 0) break;
    todo.assign(pending.begin(), pending.begin() + npending);
    P.todo = todo.data(); P.ntodo = npending;
    npending = 0; pool_used = 0;
  }
  for (int k = 0; k < np; ++k) {
    printf("%d %d %d %d %d %d", scores[k], spans[4 * k], spans[4 * k + 1], spans[4 * k + 2], spans[4 * k + 3], ops_count[k]);
    for (int u = 0; u < ops_count[k]; ++u) printf(" %u", ops[(size_t)k * ops_stride + u]);
    printf("\n");
  }
  printf("rounds %d err %d cells %llu\n", rounds, err, cells);
  return 0;
}
#else
int main() { return 0; }
#endif
