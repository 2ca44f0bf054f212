// wide_band_emu.cu -- runs the product's banded kernel bodies for bands wider than 64 diagonals on CPU threads, two
// emulated warps of one pthread per lane: the score body (csrc/swb_banded.cuh: banded_warpS<MODE, 8, W>) and the
// alignment bodies (csrc/swb_align_banded.cuh: band_span_pair<K>, band_trace_pair<K>, K = W / 64) with the host driver's
// round structure (trace, then the pending pairs again with the pool emptied).  TEST TOOL ONLY.
//
// usage: wide_band_emu score pairs.bin W MODE band_lo ma mi gi ge
//        wide_band_emu align pairs.bin W band_lo ma mi gi ge slot_words pool_words ops_stride
//   pairs.bin: int32 npairs, then per pair int32 len1, int32 len2, len1 bytes, len2 bytes (A, C, G, T only).
//   seq1 = columns, seq2 = rows, as a batch packed with keep_order = 1.
//   score prints "scores s s ...";  align prints one line per pair: "score i_start j_start i_end j_end n_ops op op ..."
//   (ops as count << 4 | op), then "rounds R err E cells C"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <thread>
#include <algorithm>
#include "../../concurrentproject_b200/csrc/swb_banded.cuh"
#include "../../concurrentproject_b200/csrc/swb_align_banded.cuh"

using namespace swb;

#if !SWB_DEVICE_CODE

static void pack(const std::vector<uint8_t>& s, uint64_t* words) {
  for (size_t k = 0; k < s.size(); ++k) words[k >> 5] |= (uint64_t)((s[k] >> 1) & 3) << (2 * (k & 31));
}

constexpr int NW = 2;   // emulated warps

static std::vector<WarpShared> make_warps() {
  std::vector<WarpShared> ws(NW);
  for (auto& x : ws) pthread_barrier_init(&x.bar, nullptr, 32);
  return ws;
}

template <typename F>
static void run_warps(std::vector<WarpShared>& ws, F body) {
  std::vector<std::thread> th;
  for (int wi = 0; wi < NW; ++wi)
    for (int l = 0; l < 32; ++l) th.emplace_back([&, wi, l]() { body(WarpCtx{l, &ws[wi]}, (long long)wi); });
  for (auto& x : th) x.join();
}

template <int MODE, int W>
static void score(const BandedParams& P) {
  auto ws = make_warps();
  std::vector<BandedWarpSmemS<8, W>> sm(NW);
  run_warps(ws, [&](const WarpCtx& w, long long wi) { banded_warpS<MODE, 8, W>(P, w, wi, NW, &sm[wi]); });
}

template <int K>
static int align(AlignBandedParams& P, std::vector<int>& todo) {
  auto ws = make_warps();
  std::vector<uint32_t> stage((size_t)NW * kBandStageLines * 32);
  run_warps(ws, [&](const WarpCtx& w, long long wi) {
    long long c = 0;
    for (long long k = wi; k < P.npairs; k += P.nwarps) c += band_span_pair<K>(P, w, k);
    align_atomic_add(P.cells, (unsigned long long)c);
  });
  int rounds = 0;
  for (;;) {
    ++rounds;
    run_warps(ws, [&](const WarpCtx& w, long long wi) {
      long long c = 0;
      for (long long u = wi; u < P.ntodo; u += P.nwarps) {
        const long long r = band_trace_pair<K>(P, w, P.todo ? P.todo[u] : u, wi, &stage[(size_t)wi * kBandStageLines * 32]);
        c += r > 0 ? r : 0;
      }
      align_atomic_add(P.cells, (unsigned long long)c);
    });
    if (*P.npending == 0) break;
    todo.assign(P.pending, P.pending + *P.npending);
    P.todo = todo.data(); P.ntodo = *P.npending;
    *P.npending = 0; *P.pool_used = 0;
  }
  return rounds;
}

int main(int argc, char** argv) {
  const bool is_score = argc == 10 && !strcmp(argv[1], "score"), is_align = argc == 12 && !strcmp(argv[1], "align");
  if (!is_score && !is_align) {
    fprintf(stderr, "usage: wide_band_emu score pairs.bin W MODE band_lo ma mi gi ge\n"
                    "       wide_band_emu align pairs.bin W band_lo ma mi gi ge slot_words pool_words ops_stride\n");
    return 2;
  }
  FILE* f = fopen(argv[2], "rb");
  if (!f) { fprintf(stderr, "cannot open %s\n", argv[2]); return 2; }
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
  const int W = atoi(argv[3]);
  std::vector<int> scores(np, -1);

  if (is_score) {
    const int mode = atoi(argv[4]);
    BandedParams P{};
    P.a_words = aw.data(); P.b_words = bw.data(); P.a_len = la.data(); P.b_len = lb.data(); P.a_stride = as; P.b_stride = bs;
    P.npairs = np; P.band_lo = atoi(argv[5]); P.scores = scores.data();
    P.match = atoi(argv[6]); P.mismatch = atoi(argv[7]); P.gap_init = atoi(argv[8]); P.gap_ext = atoi(argv[9]);
    switch (W * 2 + mode) {
      case 256: score<0, 128>(P); break;
      case 257: score<1, 128>(P); break;
      case 512: score<0, 256>(P); break;
      case 513: score<1, 256>(P); break;
      case 1024: score<0, 512>(P); break;
      case 1025: score<1, 512>(P); break;
      default: fprintf(stderr, "unsupported W / MODE\n"); return 2;
    }
    printf("scores");
    for (int k = 0; k < np; ++k) printf(" %d", scores[k]);
    printf("\n");
    return 0;
  }

  const int K = W / 64;
  const int ops_stride = atoi(argv[11]);
  std::vector<int> spans(4 * (size_t)np, -1), ops_count(np, -999), pending(np + 1), todo(np + 1);
  std::vector<uint32_t> ops((size_t)np * ops_stride + 1, 0);
  const long long slot_words = atoll(argv[9]);
  long long pool_words = atoll(argv[10]);
  for (int k = 0; k < np; ++k) pool_words = std::max(pool_words, K * band_dir_words(la[k], lb[k]));   // as the host sizes it
  std::vector<uint32_t> slot((size_t)std::max(1LL, slot_words) * NW), pool((size_t)std::max(1LL, pool_words));
  unsigned long long pool_used = 0, cells = 0;
  int npending = 0, err = 0;
  AlignBandedParams P{};
  P.a_words = aw.data(); P.b_words = bw.data(); P.a_len = la.data(); P.b_len = lb.data();
  P.a_stride = as; P.b_stride = bs; P.npairs = np; P.band_lo = atoi(argv[4]);
  P.match = atoi(argv[5]); P.mismatch = atoi(argv[6]); P.gap_init = atoi(argv[7]); P.gap_ext = atoi(argv[8]);
  P.scores = scores.data(); P.spans = spans.data(); P.nwarps = NW;
  P.slot = slot.data(); P.slot_words = slot_words; P.pool = pool.data(); P.pool_words = pool_words; P.pool_used = &pool_used;
  P.todo = nullptr; P.ntodo = np; P.pending = pending.data(); P.npending = &npending;
  P.ops = ops.data(); P.ops_stride = ops_stride; P.ops_count = ops_count.data(); P.err = &err; P.cells = &cells;
  int rounds = 0;
  switch (K) {
    case 2: rounds = align<2>(P, todo); break;
    case 4: rounds = align<4>(P, todo); break;
    case 8: rounds = align<8>(P, todo); break;
    default: fprintf(stderr, "unsupported W\n"); return 2;
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
