/*
 * banded_span_oracle.c -- CPU checker for banded batch alignment (swb200_align_banded_batch).  TEST INFRASTRUCTURE ONLY:
 * built by tests/banded_oracle.py into a temporary directory; the shipped library never links it.
 *
 * oracle_gotoh_banded_span: score and span of the best local alignment all of whose cells lie in the band
 * band_lo <= j - i <= band_hi (i over seq2, j over seq1, 1-based):
 *   - score and end cell: main.cpp:57-63 on in-band cells only, out-of-band cells H = E = F = 0 (oracle_gotoh_banded),
 *     the end cell by oracle_gotoh_end's rule (smallest j, then smallest i);
 *   - start cell: the anchored recurrence (oracle_gotoh_anchored_end) over the reversed prefixes seq1[..j_end],
 *     seq2[..i_end] in the mirrored band (j_end - i_end) - band_hi .. (j_end - i_end) - band_lo, cells outside it
 *     unreachable; the first cell reaching the score by the same rule (largest j_start, then largest i_start).
 * Work and memory are O(band x length), so 10 kb pairs take milliseconds.  All zero for score 0.
 */
#include <stdlib.h>

typedef struct { int match, mismatch, gap_init, gap_ext; } banded_params;

static long long lmax(long long a, long long b) { return a > b ? a : b; }

static int better(long long h, int i, int j, long long best, int bi, int bj) {
  return h > best || (h == best && h > 0 && (j < bj || (j == bj && i < bi)));
}

/* pass 1: banded local end cell */
static int banded_end(const unsigned char* s1, const unsigned char* s2, int n, int m, int lo, int hi,
                      const banded_params* p, int* ie, int* je) {
  long long* H = (long long*)calloc((size_t)n + 2, sizeof(long long));
  long long* F = (long long*)calloc((size_t)n + 2, sizeof(long long));
  long long best = 0;
  int bi = 0, bj = 0;
  for (int i = 1; i <= m && H && F; ++i) {
    long jlo = (long)i + lo, jhi = (long)i + hi;
    if (jlo < 1) jlo = 1;
    if (jhi > n) jhi = n;
    if (jlo > jhi) continue;
    long long e = 0, hleft = 0, hdiag = jlo > 1 ? H[jlo - 1] : 0;
    for (long j = jlo; j <= jhi; ++j) {
      e = lmax(e - p->gap_ext, hleft - p->gap_init);
      const long long f = lmax(F[j] - p->gap_ext, H[j] - p->gap_init);
      long long h = hdiag + (s1[j - 1] == s2[i - 1] ? p->match : p->mismatch);
      h = lmax(lmax(h, e), lmax(f, 0));
      hdiag = H[j]; H[j] = h; F[j] = f; hleft = h;
      if (better(h, i, (int)j, best, bi, bj)) { best = h; bi = i; bj = (int)j; }
    }
  }
  free(H); free(F);
  *ie = bi; *je = bj;
  return (int)best;
}

/* pass 2: anchored recurrence from (0, 0) restricted to lo <= j - i <= hi (lo <= 0 <= hi); its maximum and cell */
static int banded_anchored(const unsigned char* s1, const unsigned char* s2, int n, int m, int lo, int hi,
                           const banded_params* p, int* ri, int* rj) {
  const long long NEG = -(1LL << 40);
  const int gi = p->gap_init, ge = p->gap_ext, gmin = gi < ge ? gi : ge;
  long long* H = (long long*)malloc(((size_t)n + 2) * sizeof(long long));
  long long* F = (long long*)malloc(((size_t)n + 2) * sizeof(long long));
  long long best = 0;
  int bi = 0, bj = 0;
  if (H && F) {
    for (int j = 0; j <= n + 1; ++j) { H[j] = (j <= n && j <= hi) ? (j == 0 ? 0 : -(gi + (long long)(j - 1) * gmin)) : NEG; F[j] = NEG; }
    for (int i = 1; i <= m; ++i) {
      long jlo = (long)i + lo, jhi = (long)i + hi;
      if (jlo < 0) jlo = 0;
      if (jhi > n) jhi = n;
      if (jlo > jhi) break;                       /* the band has left the rectangle for good */
      long long e = NEG, hleft = NEG, hdiag = jlo > 0 ? H[jlo - 1] : NEG;
      for (long j = jlo; j <= jhi; ++j) {
        if (j == 0) {                              /* column 0: the border */
          hdiag = H[0];
          H[0] = -(gi + (long long)(i - 1) * gmin); F[0] = NEG; hleft = H[0];
          continue;
        }
        e = lmax(e - ge, hleft - gi);
        const long long f = lmax(F[j] - ge, H[j] - gi);   /* (i-1, j): NEG where it was outside the band */
        long long h = hdiag + (s1[j - 1] == s2[i - 1] ? p->match : p->mismatch);
        h = lmax(h, lmax(e, f));
        hdiag = H[j]; H[j] = h; F[j] = f; hleft = h;
        if (better(h, i, (int)j, best, bi, bj)) { best = h; bi = i; bj = (int)j; }
      }
      /* (i, jhi + 1) lies right of the band: no earlier row wrote that entry, so the next row reads it as NEG */
    }
  }
  free(H); free(F);
  *ri = bi; *rj = bj;
  return (int)best;
}

int oracle_gotoh_banded_span(const unsigned char* seq1, const unsigned char* seq2, int n, int m, int band_lo, int band_hi,
                             const banded_params* p, int* i_start, int* j_start, int* i_end, int* j_end) {
  *i_start = *j_start = *i_end = *j_end = 0;
  if (n < 0 || m < 0 || band_lo > band_hi) return -1;
  int ie = 0, je = 0;
  const int s = banded_end(seq1, seq2, n, m, band_lo, band_hi, p, &ie, &je);
  if (s <= 0) return s;
  unsigned char* r1 = (unsigned char*)malloc((size_t)je + 1);
  unsigned char* r2 = (unsigned char*)malloc((size_t)ie + 1);
  if (!r1 || !r2) { free(r1); free(r2); return -1; }
  for (int k = 0; k < je; ++k) r1[k] = seq1[je - 1 - k];
  for (int k = 0; k < ie; ++k) r2[k] = seq2[ie - 1 - k];
  int ri = 0, rj = 0;
  const int s2 = banded_anchored(r1, r2, je, ie, (je - ie) - band_hi, (je - ie) - band_lo, p, &ri, &rj);
  free(r1); free(r2);
  if (s2 != s) return -2;                          /* cannot happen: the best alignment ends at (i_end, j_end) */
  *i_start = ie - ri + 1; *j_start = je - rj + 1; *i_end = ie; *j_end = je;
  return s;
}
