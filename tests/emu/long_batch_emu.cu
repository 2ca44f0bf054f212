// long_batch_emu.cu -- runs the product's multi-band batch kernel body (csrc/swb_batch.cuh, batch_warp with LONG) on CPU
// threads, one pthread per lane (see batch_emu.cu): two emulated warps take pairs from one counter.  TEST TOOL ONLY.
//
// usage: long_batch_emu pairs.bin R MODE [match mismatch gap_init gap_ext]
//   pairs.bin: int32 npairs, then per pair int32 len1, int32 len2, len1 bytes, len2 bytes; the shorter sequence of a pair is
//   striped (as launch_pack_batch does).  Prints "scores s0 s1 ...".
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <thread>
#include "../../concurrentproject_b200/csrc/swb_batch.cuh"

using namespace swb;

#if !SWB_DEVICE_CODE

static void pack(const std::vector<uint8_t>& s, uint64_t* words) {
  for (size_t k = 0; k < s.size(); ++k) words[k >> 5] |= (uint64_t)((s[k] >> 1) & 3) << (2 * (k & 31));
}

typedef void (*long_fn)(const BatchParams*, WarpShared*, int, long long, BatchWarpSmem*, uint32_t*, unsigned long long*);
template <int R, int MODE>
static void run_lane(const BatchParams* P, WarpShared* ws, int lane, long long wid, BatchWarpSmem* sm, uint32_t* bnd,
                     unsigned long long* next) {
  WarpCtx w{lane, ws};
  batch_warp<R, MODE, 32, true>(*P, w, wid, 2, sm, bnd, next);
}

int main(int argc, char** argv) {
  if (argc < 4) { fprintf(stderr, "usage: long_batch_emu pairs.bin R MODE [ma mi gi ge]\n"); return 2; }
  FILE* f = fopen(argv[1], "rb");
  if (!f) { fprintf(stderr, "cannot open %s\n", argv[1]); return 2; }
  const int R = atoi(argv[2]), mode = atoi(argv[3]);
  const int ma = argc > 4 ? atoi(argv[4]) : 1, mi = argc > 5 ? atoi(argv[5]) : -1, gi = argc > 6 ? atoi(argv[6]) : 1,
            ge = argc > 7 ? atoi(argv[7]) : 1;
  long_fn fn = nullptr;
  if (R == 2) fn = mode ? run_lane<2, 1> : run_lane<2, 0>;
  if (R == 4) fn = mode ? run_lane<4, 1> : run_lane<4, 0>;
  if (!fn) { fprintf(stderr, "unsupported R\n"); return 2; }
  int32_t np = 0;
  if (fread(&np, 4, 1, f) != 1) return 2;
  std::vector<std::vector<uint8_t>> s1(np), s2(np);
  int max_q = 0, max_t = 0;
  for (int k = 0; k < np; ++k) {
    int32_t l[2];
    if (fread(l, 4, 2, f) != 2) return 2;
    s1[k].resize(l[0]); s2[k].resize(l[1]);
    if (l[0] && fread(s1[k].data(), 1, l[0], f) != (size_t)l[0]) return 2;
    if (l[1] && fread(s2[k].data(), 1, l[1], f) != (size_t)l[1]) return 2;
    if (s1[k].size() > s2[k].size()) std::swap(s1[k], s2[k]);      // Q = the shorter one
    max_q = std::max(max_q, (int)s1[k].size()); max_t = std::max(max_t, (int)s2[k].size());
  }
  fclose(f);
  const long long qs = std::max(1, (max_q + 31) / 32), ts = std::max(1, (max_t + 31) / 32) + 2;
  std::vector<uint64_t> qw((size_t)np * qs + 4, 0), tw((size_t)np * ts + 4, 0);
  std::vector<int> ql(np), tl(np), scores(np, -1);
  for (int k = 0; k < np; ++k) { pack(s1[k], &qw[(size_t)k * qs]); pack(s2[k], &tw[(size_t)k * ts]); ql[k] = (int)s1[k].size(); tl[k] = (int)s2[k].size(); }
  BatchParams P{};
  P.q_words = qw.data(); P.t_words = tw.data(); P.q_len = ql.data(); P.t_len = tl.data(); P.q_stride = qs; P.t_stride = ts;
  P.npairs = np; P.scores = scores.data(); P.match = ma; P.mismatch = mi; P.gap_init = gi; P.gap_ext = ge;
  const int W = 2;
  const long long stride = (std::max(max_t, 1) + 31) / 32 * 32;
  std::vector<uint32_t> bnd((size_t)W * stride, 0xDEADBEEFu);   // stale words: the kernel must never read one it did not write
  unsigned long long next = 0;
  std::vector<WarpShared> ws(W);
  for (auto& x : ws) pthread_barrier_init(&x.bar, nullptr, 32);
  std::vector<BatchWarpSmem> sm(W);
  std::vector<std::thread> th;
  for (int w = 0; w < W; ++w)
    for (int l = 0; l < 32; ++l) th.emplace_back(fn, &P, &ws[w], l, (long long)w, &sm[w], bnd.data() + w * stride, &next);
  for (auto& x : th) x.join();
  printf("scores");
  for (int k = 0; k < np; ++k) printf(" %d", scores[k]);
  printf("\n");
  return 0;
}
#else
int main() { return 0; }
#endif
