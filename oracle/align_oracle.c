/*
 * align_oracle.c — CPU restatement (plain C) of the edit-operation alignment
 * of espnet_data/preprocess/align.py (hyp_alignment.json).
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product path may call this file:
 * it is the checker of tests/test_align_host.py, tests/test_gpu_align.py and
 * the "port" arm of tools/bench_align.py.  Built on first use by
 * oracle/align_oracle.py (gcc -O2, into a per-user cache directory).
 */
#include <stdint.h>
#include <stdlib.h>

/* ---------------------------------------------------------------------------
 * Edit-operation alignment: espnet_data/preprocess/align.py
 * (levenshtein_distance_alignment, hyp_alignment.json), restated from the
 * contract of DESIGN.md §3.10 on the full (na+1) x (nb+1) table.  Backtrace
 * from (na, nb): the first predecessor attaining D[i][j] in the order
 * diagonal (U/S), up (I: reference symbol unmatched), left (D: hypothesis
 * symbol unmatched).  Ops are ASCII letters in forward order; counts are
 * (U, S, I, D).  Returns the number of ops.
 * ------------------------------------------------------------------------- */
int32_t oracle_align(const int32_t* a, int32_t na, const int32_t* b, int32_t nb, uint8_t* ops, int32_t* counts) {
  const int64_t w = (int64_t)nb + 1;
  int32_t* D = (int32_t*)malloc(sizeof(int32_t) * (size_t)((int64_t)(na + 1) * w));
  for (int32_t j = 0; j <= nb; ++j) D[j] = j;
  for (int32_t i = 1; i <= na; ++i) {
    D[i * w] = i;
    for (int32_t j = 1; j <= nb; ++j) {
      int32_t sub = D[(i - 1) * w + j - 1] + (a[i - 1] != b[j - 1]);
      int32_t up = D[(i - 1) * w + j] + 1;
      int32_t left = D[i * w + j - 1] + 1;
      int32_t v = sub < up ? sub : up;
      D[i * w + j] = v < left ? v : left;
    }
  }
  int32_t n = 0, i = na, j = nb;
  uint8_t* rev = (uint8_t*)malloc((size_t)na + (size_t)nb + 1);
  counts[0] = counts[1] = counts[2] = counts[3] = 0;
  while (i > 0 || j > 0) {
    int32_t d = D[i * w + j], c;
    if (i > 0 && j > 0 && D[(i - 1) * w + j - 1] + (a[i - 1] != b[j - 1]) == d) c = a[i - 1] != b[j - 1];
    else if (i > 0 && D[(i - 1) * w + j] + 1 == d) c = 2;
    else c = 3;
    rev[n++] = "USID"[c];
    counts[c] += 1;
    if (c != 3) --i;
    if (c != 2) --j;
  }
  for (int32_t k = 0; k < n; ++k) ops[k] = rev[n - 1 - k];
  free(rev);
  free(D);
  return n;
}

/* pair i: ref[pair_ref[i]] vs hyp i; ops of pair i at ops_off[i] (slot of na + nb bytes). */
void oracle_align_batch(const int32_t* ref_cp, const int64_t* ref_off, const int32_t* hyp_cp,
                        const int64_t* hyp_off, const int32_t* pair_ref, int32_t n_pairs,
                        const int64_t* ops_off, uint8_t* out_ops, int32_t* out_n_ops, int32_t* out_counts) {
  for (int32_t p = 0; p < n_pairs; ++p) {
    int32_t r = pair_ref[p];
    out_n_ops[p] = oracle_align(ref_cp + ref_off[r], (int32_t)(ref_off[r + 1] - ref_off[r]),
                                hyp_cp + hyp_off[p], (int32_t)(hyp_off[p + 1] - hyp_off[p]),
                                out_ops + ops_off[p], out_counts + 4 * (int64_t)p);
  }
}
