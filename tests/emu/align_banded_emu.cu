// align_banded_emu.cu -- runs the product's banded batch alignment bodies (csrc/swb_align_banded.cuh: band_span_pair,
// band_trace_pair) on CPU threads, two emulated warps of one pthread per lane, with the host driver's round structure
// (trace, then the pending pairs again with the pool emptied).  TEST TOOL ONLY.
//
// usage: align_banded_emu pairs.bin band_lo ma mi gi ge slot_words pool_words ops_stride
//   pairs.bin: int32 npairs, then per pair int32 len1, int32 len2, len1 bytes, len2 bytes (A, C, G, T only).
//   seq1 = columns, seq2 = rows, as a batch packed with keep_order = 1.
//   prints one line per pair: "score i_start j_start i_end j_end n_ops op op ..." (ops as count << 4 | op), then
//   "rounds R err E"
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <thread>
#include <algorithm>
#include "../../concurrentproject_b200/csrc/swb_align_banded.cuh"

using namespace swb;

#if !SWB_DEVICE_CODE

static void pack(const std::vector<uint8_t>& s, uint64_t* words) {
  for (size_t k = 0; k < s.size(); ++k) words[k >> 5] |= (uint64_t)((s[k] >> 1) & 3) << (2 * (k & 31));
}

int main(int argc, char** argv) {
  if (argc < 10) { fprintf(stderr, "usage: align_banded_emu pairs.bin band_lo ma mi gi ge slot_words pool_words ops_stride\n"); return 2; }
  FILE* f = fopen(argv[1], "rb");
  if (!f) { fprintf(stderr, "cannot open %s\n", argv[1]); return 2; }
  int32_t np = 0;
  if (fread(&np, 4, 1, f) != 1) return 2;
  std::vector<std::vector<uint8_t>> a(np), b(np);
  std::vector<int> la(np), lb(np);
  int max_a = 0, max_b = 0;
  for (int k = 0; k < np; ++k) {
    int32_t l[2];
    if (fread(l, 4, 2, f) != 2) return 2;
    a[k].resize(l[0]); b[k].resize(l[1]);
    if (l[0] && fread(a[k].data(), 1, l[0], f) != (size_t)l[0]) return 2;
    if (l[1] && fread(b[k].data(), 1, l[1], f) != (size_t)l[1]) return 2;
    la[k] = l[0]; lb[k] = l[1];
    max_a = std::max(max_a, la[k]); max_b = std::max(max_b, lb[k]);
  }
  fclose(f);
  const long long as = std::max(1, (max_a + 31) / 32) + 2, bs = std::max(1, (max_b + 31) / 32) + 2;   // keep_order strides
  std::vector<uint64_t> aw((size_t)np * as + 4, 0), bw((size_t)np * bs + 4, 0);
  for (int k = 0; k < np; ++k) { pack(a[k], &aw[(size_t)k * as]); pack(b[k], &bw[(size_t)k * bs]); }
  const int W = 2;                                  // emulated warps
  const int ops_stride = atoi(argv[9]);
  std::vector<int> scores(np, -1), spans(4 * (size_t)np, -1), ops_count(np, -999), pending(np + 1), todo(np + 1);
  std::vector<uint32_t> ops((size_t)np * ops_stride + 1, 0);
  const long long slot_words = atoll(argv[7]);
  long long pool_words = atoll(argv[8]);
  for (int k = 0; k < np; ++k) pool_words = std::max(pool_words, band_dir_words(la[k], lb[k]));   // as the host sizes it
  std::vector<uint32_t> slot((size_t)std::max(1LL, slot_words) * W), pool((size_t)std::max(1LL, pool_words));
  std::vector<uint32_t> stage((size_t)W * kBandStageLines * 32);
  unsigned long long pool_used = 0, cells = 0;
  int npending = 0, err = 0;
  AlignBandedParams P{};
  P.a_words = aw.data(); P.b_words = bw.data(); P.a_len = la.data(); P.b_len = lb.data();
  P.a_stride = as; P.b_stride = bs; P.npairs = np; P.band_lo = atoi(argv[2]);
  P.match = atoi(argv[3]); P.mismatch = atoi(argv[4]); P.gap_init = atoi(argv[5]); P.gap_ext = atoi(argv[6]);
  P.scores = scores.data(); P.spans = spans.data(); P.nwarps = W;
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
    for (long long k = wi; k < P.npairs; k += P.nwarps) c += band_span_pair(P, w, k);
    align_atomic_add(P.cells, (unsigned long long)c);
  });
  int rounds = 0;
  for (;;) {
    ++rounds;
    warps([&](const WarpCtx& w, long long wi) {
      long long c = 0;
      for (long long u = wi; u < P.ntodo; u += P.nwarps) {
        const long long r = band_trace_pair(P, w, P.todo ? P.todo[u] : u, wi, &stage[(size_t)wi * kBandStageLines * 32]);
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
