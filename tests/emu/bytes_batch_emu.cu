// bytes_batch_emu.cu -- runs the product's batch bodies (csrc/swb_align_batch.cuh: align_score_pair, align_span_pair,
// align_trace_pair) on CPU threads in either symbol layout, one pthread per lane of one emulated warp, with the host
// driver's round structure (trace, then the pending pairs again with the pool emptied).  TEST TOOL ONLY.
//
// usage: bytes_batch_emu pairs.bin bits ma mi gi ge slot_words pool_words ops_stride
//   pairs.bin: int32 npairs, then per pair int32 len1, int32 len2, len1 bytes, len2 bytes.
//   bits 8: the byte layout of the byte packer (8 bytes per word, any byte); bits 2: the 2-bit layout (A, C, G, T only).
//   The shorter sequence of a pair is Q, as both packers do (swapped iff len1 > len2).
//   prints one line per pair: "score_only score i_start j_start i_end j_end n_ops op op ..." (ops as count << 4 | op),
//   then "rounds R err E"
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <thread>
#include <algorithm>
#include "../../concurrentproject_b200/csrc/swb_align_batch.cuh"

using namespace swb;

#if !SWB_DEVICE_CODE

static void pack(const std::vector<uint8_t>& s, uint64_t* words, int bits) {
  for (size_t k = 0; k < s.size(); ++k) {
    if (bits == 8) words[k >> 3] |= (uint64_t)s[k] << (8 * (k & 7));
    else words[k >> 5] |= (uint64_t)((s[k] >> 1) & 3) << (2 * (k & 31));
  }
}

template <int BITS>
static int run(AlignBatchParams& P, std::vector<int>& score_only, std::vector<int>& todo) {
  const int NT = (int)P.nthreads;
  {
    std::vector<std::thread> th;
    for (int l = 0; l < NT; ++l)
      th.emplace_back([&P, &score_only, l, NT]() {
        AlignBatchParams S = P;
        S.scores = score_only.data();
        for (long long k = l; k < P.npairs; k += NT) align_score_pair<BITS>(S, k, l);
      });
    for (auto& x : th) x.join();
  }
  {
    std::vector<std::thread> th;
    for (int l = 0; l < NT; ++l)
      th.emplace_back([&P, l, NT]() { for (long long k = l; k < P.npairs; k += NT) align_span_pair<BITS>(P, k, l); });
    for (auto& x : th) x.join();
  }
  int rounds = 0;
  for (;;) {
    ++rounds;
    std::vector<std::thread> th;
    for (int l = 0; l < NT; ++l)
      th.emplace_back([&P, l, NT]() { for (long long u = l; u < P.ntodo; u += NT) align_trace_pair<BITS>(P, P.todo ? P.todo[u] : u, l); });
    for (auto& x : th) x.join();
    if (*P.npending == 0) break;
    todo.assign(P.pending, P.pending + *P.npending);
    P.todo = todo.data(); P.ntodo = *P.npending;
    *P.npending = 0; *P.pool_used = 0;
  }
  return rounds;
}

int main(int argc, char** argv) {
  if (argc < 10) { fprintf(stderr, "usage: bytes_batch_emu pairs.bin bits ma mi gi ge slot_words pool_words ops_stride\n"); return 2; }
  FILE* f = fopen(argv[1], "rb");
  if (!f) { fprintf(stderr, "cannot open %s\n", argv[1]); return 2; }
  const int bits = atoi(argv[2]);
  if (bits != 2 && bits != 8) { fprintf(stderr, "bits must be 2 or 8\n"); return 2; }
  int32_t np = 0;
  if (fread(&np, 4, 1, f) != 1) return 2;
  std::vector<std::vector<uint8_t>> q(np), t(np);
  std::vector<int> len1(np), ql(np), tl(np);
  int max_q = 0, max_t = 0;
  for (int k = 0; k < np; ++k) {
    int32_t l[2];
    if (fread(l, 4, 2, f) != 2) return 2;
    std::vector<uint8_t> a(l[0]), b(l[1]);
    if (l[0] && fread(a.data(), 1, l[0], f) != (size_t)l[0]) return 2;
    if (l[1] && fread(b.data(), 1, l[1], f) != (size_t)l[1]) return 2;
    len1[k] = l[0];
    if (l[0] > l[1]) std::swap(a, b);
    q[k] = a; t[k] = b;
    ql[k] = (int)a.size(); tl[k] = (int)b.size();
    max_q = std::max(max_q, ql[k]); max_t = std::max(max_t, tl[k]);
  }
  fclose(f);
  // the strides of the host packers: byte_strides_for / batch_strides_for (swb200.cu)
  const int per = 64 / bits;
  const long long qs = std::max(1, (max_q + per - 1) / per), ts = std::max(1, (max_t + per - 1) / per) + (bits == 2 ? 2 : 0);
  std::vector<uint64_t> qw((size_t)np * qs + 1, 0), tw((size_t)np * ts + 1, 0);
  for (int k = 0; k < np; ++k) { pack(q[k], &qw[(size_t)k * qs], bits); pack(t[k], &tw[(size_t)k * ts], bits); }
  const int NT = 32;
  const int ops_stride = atoi(argv[9]);
  std::vector<int> scores(np, -1), score_only(np, -1), spans(4 * (size_t)np, -1), ops_count(np, -999), pending(np + 1), todo(np + 1);
  std::vector<uint32_t> ops((size_t)np * ops_stride + 1, 0);
  std::vector<int2> col((size_t)(max_q + 1) * NT);
  const long long slot_words = atoll(argv[7]);
  long long pool_words = atoll(argv[8]);
  for (int k = 0; k < np; ++k) pool_words = std::max(pool_words, align_dir_words(tl[k], ql[k]));   // as the host sizes it
  std::vector<uint64_t> slot((size_t)std::max(1LL, slot_words) * NT), pool((size_t)std::max(1LL, pool_words));
  unsigned long long pool_used = 0;
  int npending = 0, err = 0;
  AlignBatchParams P{};
  P.q_words = qw.data(); P.t_words = tw.data(); P.q_len = ql.data(); P.t_len = tl.data(); P.len1 = len1.data();
  P.q_stride = qs; P.t_stride = ts; P.npairs = np;
  P.match = atoi(argv[3]); P.mismatch = atoi(argv[4]); P.gap_init = atoi(argv[5]); P.gap_ext = atoi(argv[6]);
  P.scores = scores.data(); P.spans = spans.data(); P.col = col.data(); P.nthreads = NT;
  P.slot = slot.data(); P.slot_words = slot_words; P.pool = pool.data(); P.pool_words = pool_words; P.pool_used = &pool_used;
  P.todo = nullptr; P.ntodo = np; P.pending = pending.data(); P.npending = &npending;
  P.ops = ops.data(); P.ops_stride = ops_stride; P.ops_count = ops_count.data(); P.err = &err;
  const int rounds = bits == 8 ? run<8>(P, score_only, todo) : run<2>(P, score_only, todo);
  for (int k = 0; k < np; ++k) {
    printf("%d %d %d %d %d %d %d", score_only[k], scores[k], spans[4 * k], spans[4 * k + 1], spans[4 * k + 2], spans[4 * k + 3],
           ops_count[k]);
    for (int u = 0; u < ops_count[k]; ++u) printf(" %u", ops[(size_t)k * ops_stride + u]);
    printf("\n");
  }
  printf("rounds %d err %d\n", rounds, err);
  return 0;
}
#else
int main() { return 0; }
#endif
