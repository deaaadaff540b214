/*
 * mcmc_main.c -- the `mcmc` command line over the C ABI (host code stays in C).
 *
 * Drop-in for the reference binary's contract (C_Implementation/mcmc.c:102-210, called by
 * script.py:44-45 as `./mcmc <chain_index> < dataset.txt` with GSL_RNG_SEED in the environment):
 *   - argv[1] = chain index -> files go to Chains/chain_XX/ (two digits, like mcmc.c:148-178)
 *   - stdin   = dataset in the reference's .txt format
 *   - 1000 burn-in + 1000 sampling calls of 10 sweeps, one thinned sample per call
 *   - writes chain_data.csv, exp_data.csv, taxa.csv, sites.csv, hard_sites.csv
 *   - stderr echoes "GSL_RNG_SEED=<n>" like gsl_rng_env_setup(); exit 0 / 1
 * Differences, all deliberate: the random stream is the structured Philox stream keyed by
 * (GSL_RNG_SEED, chain index) instead of GSL's MT19937; Chains/chain_XX/ is created when missing
 * (the reference dereferences a NULL FILE*); `mcmc` without arguments prints usage instead of
 * crashing at atoi(NULL) (mcmc.c:153).
 *
 * Batch mode (replaces script.py's Pool over 100 processes by one call over all the chains, on one GPU or
 * sharded over the GPUs of the box -- ser_multi_*):
 *   mcmc --chains N [--gpus G] [--first I] [--burn B] [--samples S] [--seed X] [--dataset file]
 *        [--chains-dir DIR] [--select K] [--po file.csv] [--device D] [--manycd 0|1] [--replay-selected --window W]
 *        [--checkpoint FILE [--checkpoint-every C] [--resume] [--stop-after C]] [--diagnostics FILE] [--rank-diagnostics FILE]
 *        [--marginals PREFIX] [--taxon-pairs PREFIX] [--cd-marginals FILE] [--diversity PREFIX]
 * --replay-selected (with --select) runs select-then-replay: the chains keep no sample history (SER_STORE_NONE, so no
 * Chains/ files) and the pair-order counts of the K chosen chains come from their replay: the same output lines and po.csv
 * as the one-shot step, with device memory for K chains' window instead of every chain's history.
 * Every --select output (po.csv under --replay-selected, and the outputs of the six flags below) comes from one replay of the chosen
 * chains, alone on --device (ser_run_create_chains), which exits 1 unless each reproduces its first run's E[-logL] bit for
 * bit.  That replay keeps every sample (SER_STORE_FULL) when --diagnostics or --rank-diagnostics is given, and otherwise
 * runs through a window of W samples (--window, default 64) while what the outputs read accumulates (ser_run_accumulate);
 * the summaries are the same bits from either store.
 * --checkpoint FILE writes every chain's state to FILE at the end of the sweeps (ser_multi_save_checkpoint), and every C calls
 * with --checkpoint-every C (the advance runs in segments of at most C calls; splitting a launch changes no chain).  --resume
 * loads FILE when it exists in place of the random start and runs the calls of the --burn B --samples S schedule that are left
 * (it refuses a file that has advanced past B + S calls, or whose sample count is not max(0, calls - B)).  --stop-after C
 * advances at most C calls in this invocation, writes FILE and exits 0 with one line saying where it stopped, before any
 * summary or Chains/ file: a long run split into slices gives the same output as the run done in one piece.
 * --diagnostics FILE (with --select) writes the per-quantity split-R-hat and effective sample sizes of the chosen chains to FILE and
 * prints one summary line.
 * --rank-diagnostics FILE (with --select) writes the rank-normalised R-hat, bulk- and tail-ESS pooled over the chosen chains
 * (ser_run_rank_diagnostics) to FILE "quantity,rhat,rhat_bulk,rhat_fold,ess_bulk,ess_tail,ess_mean,q05,q95", with one summary line:
 * the largest R-hat, the smallest bulk- and tail-ESS, and how many quantities have R-hat > 1.01 or a bulk- or tail-ESS below 100 per chain.
 * --marginals PREFIX (with --select) pools the position and a / b histograms of the chosen chains and writes PREFIX.sites.csv
 * "site,hard,mean,q025,median,q975,mode,p_mode" (file order, 0-based positions) and PREFIX.taxa.csv
 * "taxon,a_mean,a_q025,a_median,a_q975,b_mean,b_q025,b_median,b_q975", and prints one summary line.
 * --taxon-pairs PREFIX (with --select) pools the taxon pair relations of the chosen chains (ser_run_taxon_pairs) and writes
 * PREFIX.first.csv, PREFIX.last.csv, PREFIX.precedes.csv and PREFIX.coexist.csv: dense M x M probability matrices (row m, column n,
 * taxa in file order; po.csv's format) of P(a_m < a_n), P(b_m < b_n), P(b_m <= a_n) and P(the ranges of m and n share a position), and
 * prints one summary line.
 * --cd-marginals FILE (with --select) pools the error-rate marginals of the chosen chains (ser_run_cd_marginals) and writes FILE
 * "taxon,c_mean,c_q025,c_median,c_q975,d_mean,d_q025,d_median,d_q975": one row per taxon (file order) on a --manycd 1 run, one row
 * "all" otherwise; the means are the posterior means of the probabilities exp(c), exp(d), q025 is the lower edge of the 2.5 % quantile's
 * bin, q975 the upper edge of the 97.5 % quantile's bin and the median the log-midpoint of its bin, all as probabilities.  It prints one
 * summary line: the rows with the highest mean d (most missed occurrences) and the highest mean c (most spurious ones).
 * --diversity PREFIX (with --select) pools the diversity curves of the chosen chains (ser_run_diversity) and writes PREFIX.positions.csv
 * "position,rich_mean,rich_q025,rich_median,rich_q975,orig_mean,orig_q025,orig_median,orig_q975,ext_mean,ext_q025,ext_median,ext_q975"
 * (range-through richness, originations and extinctions at every position of the sequence) and PREFIX.sites.csv
 * "site,hard,rich_mean,rich_q025,rich_median,rich_q975" (the richness at the position each site holds; file order, 0-based), the
 * quantiles as numbers of taxa, and prints one summary line: the peak mean richness, its position and its 95 % interval.
 * Replay mode: SER_TAPE_IN=<file of raw doubles> mcmc <idx> < dataset.txt
 */
#include <errno.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>

#include "../../include/seriation_b200.h"

static void die(const char *what)
{
  fprintf(stderr, "mcmc: %s: %s\n", what, ser_last_error());
  exit(1);
}

static void *xmalloc(size_t bytes)
{
  void *p = malloc(bytes);
  if (!p) { fprintf(stderr, "mcmc: out of memory\n"); exit(1); }
  return p;
}

static FILE *open_out(const char *path)
{
  FILE *f = fopen(path, "w");
  if (!f) { fprintf(stderr, "mcmc: cannot open %s\n", path); exit(1); }
  return f;
}

static void close_out(FILE *f, const char *path)
{
  if (fclose(f)) { fprintf(stderr, "mcmc: cannot write %s\n", path); exit(1); }
}

static void usage(const char *argv0)
{
  fprintf(stderr,
          "usage: %s <chain_index> < dataset.txt          (reference-compatible single chain)\n"
          "       %s [manycd Tburnin T] < dataset.txt      (manycd 1: per-taxon c, d; chain 0)\n"
          "       %s --chains N [--gpus G] [--first I] [--burn B] [--samples S] [--seed X] [--dataset F]\n"
          "              [--chains-dir DIR] [--select K] [--po out.csv] [--device D] [--manycd 0|1]\n"
          "              [--replay-selected --window W]   (with --select: keep no sample history, replay the chosen chains)\n"
          "              [--checkpoint FILE [--checkpoint-every C] [--resume] [--stop-after C]]\n"
          "                  (save every chain to FILE at the end and every C calls; --resume continues FILE's run; --stop-after C\n"
          "                   advances at most C calls, saves and exits)\n"
          "              [--diagnostics FILE]   (with --select: split-R-hat and ESS of the chosen chains to FILE)\n"
          "              [--rank-diagnostics FILE]   (with --select: rank-normalised R-hat, bulk- and tail-ESS pooled over the\n"
          "                                           chosen chains to FILE)\n"
          "              [--marginals PREFIX]   (with --select: position and a / b credible intervals of the chosen chains to\n"
          "                                      PREFIX.sites.csv and PREFIX.taxa.csv; the replay uses --window W)\n"
          "              [--taxon-pairs PREFIX]   (with --select: first / last appearance order, superposition and coexistence\n"
          "                                        of every pair of taxa to PREFIX.{first,last,precedes,coexist}.csv; --window W)\n"
          "              [--cd-marginals FILE]   (with --select: posterior means and credible intervals of the error rates c, d\n"
          "                                       per taxon (--manycd 1) or of the scalar pair to FILE; --window W)\n"
          "              [--diversity PREFIX]   (with --select: richness, originations and extinctions per position and richness\n"
          "                                      per site of the chosen chains to PREFIX.positions.csv and PREFIX.sites.csv; --window W)\n",
          argv0, argv0, argv0);
  exit(1);
}

static const char *quantity_name(int q, char *buf, size_t len)
{
  if (q < 3) return q == 0 ? "-logL" : q == 1 ? "c" : "d";
  snprintf(buf, len, "site_%d", q - 3);
  return buf;
}

/* NaN when either is NaN, as numpy.maximum / numpy.minimum */
static double max_nan(double a, double b) { return isnan(a) || isnan(b) ? NAN : a > b ? a : b; }
static double min_nan(double a, double b) { return isnan(a) || isnan(b) ? NAN : a < b ? a : b; }

/* --rank-diagnostics: the pooled rank-normalised diagnostics of the chosen chains of `sub` to `path` and one summary line */
static void write_rank_diagnostics(ser_run *sub, const int32_t *chosen, int32_t k, int32_t N, const char *path)
{
  const int Q = 3 + N;
  double *out = xmalloc(sizeof(double) * (size_t)Q * SER_RDIAG_FIELDS);
  double r_max = NAN, bulk_min = NAN, tail_min = NAN;
  int q, q_r = -1, q_b = -1, q_t = -1, flagged = 0;
  char b1[32], b2[32], b3[32];
  FILE *f;
  if (ser_run_rank_diagnostics(sub, chosen, k, SER_DIAG_SCALARS | SER_DIAG_SITES, out)) die("ser_run_rank_diagnostics");
  f = open_out(path);
  fprintf(f, "quantity,rhat,rhat_bulk,rhat_fold,ess_bulk,ess_tail,ess_mean,q05,q95\n");
  for (q = 0; q < Q; q++) {
    const double *o = out + (size_t)q * SER_RDIAG_FIELDS;
    const double rhat = max_nan(o[0], o[1]), tail = min_nan(o[4], o[5]);
    fprintf(f, "%s,%.17g,%.17g,%.17g,%.17g,%.17g,%.17g,%.17g,%.17g\n", quantity_name(q, b1, sizeof(b1)), rhat, o[0], o[1], o[2], tail, o[3],
            o[6], o[7]);
    if (!isnan(rhat) && (q_r < 0 || rhat > r_max)) { r_max = rhat; q_r = q; }
    if (!isnan(o[2]) && (q_b < 0 || o[2] < bulk_min)) { bulk_min = o[2]; q_b = q; }
    if (!isnan(tail) && (q_t < 0 || tail < tail_min)) { tail_min = tail; q_t = q; }
    flagged += rhat > 1.01 || o[2] < 100.0 * k || tail < 100.0 * k;
  }
  close_out(f, path);
  printf("rank diagnostics: %d chains  R-hat max %.4f (%s)  bulk-ESS min %.1f (%s)  tail-ESS min %.1f (%s)  "
         "%d of %d quantities with R-hat > 1.01 or ESS < %d\n", k, r_max, q_r < 0 ? "none" : quantity_name(q_r, b1, sizeof(b1)), bulk_min,
         q_b < 0 ? "none" : quantity_name(q_b, b2, sizeof(b2)), tail_min, q_t < 0 ? "none" : quantity_name(q_t, b3, sizeof(b3)), flagged, Q,
         100 * k);
  free(out);
}

/* --diagnostics: the split-R-hat and ESS of the chosen chains of `sub` to `path` as CSV, and one summary line */
static void write_diagnostics(ser_run *sub, const int32_t *chosen, int32_t k, int32_t N, const char *path)
{
  const int Q = 3 + N;
  double *stats = xmalloc(sizeof(double) * (size_t)k * Q * 4), *halves = xmalloc(sizeof(double) * (size_t)k * Q * 4);
  double *rhat = xmalloc(sizeof(double) * (size_t)Q);
  int32_t *n = xmalloc(sizeof(int32_t) * (size_t)k);
  int q, c, s_max = -1, s_min = -1, constant = 0;
  double r_max = NAN, ess_min_site = NAN, ess_min[3];
  char name[32];
  FILE *f;
  if (ser_run_diagnostics(sub, chosen, k, SER_DIAG_SCALARS | SER_DIAG_SITES, 0, stats, halves, n)) die("ser_run_diagnostics");
  if (ser_split_rhat(halves, n, k, Q, rhat)) die("ser_split_rhat");
  f = open_out(path);
  fprintf(f, "quantity,mean,rhat,ess_min,ess_sum\n");
  for (q = 0; q < Q; q++) {
    double mean = 0.0, emin = NAN, esum = NAN;
    for (c = 0; c < k; c++) {
      const double *st = stats + ((size_t)c * Q + q) * 4;
      mean += st[0];
      if (isnan(st[2])) continue;
      emin = isnan(emin) || st[2] < emin ? st[2] : emin;
      esum = isnan(esum) ? st[2] : esum + st[2];
    }
    mean /= k;
    fprintf(f, "%s,%.17g,%.17g,%.17g,%.17g\n", quantity_name(q, name, sizeof(name)), mean, rhat[q], emin, esum);
    if (q < 3) ess_min[q] = emin;
    else {
      if (isnan(emin)) constant++; /* constant in every chosen chain */
      if (!isnan(rhat[q]) && (s_max < 0 || rhat[q] > r_max)) { r_max = rhat[q]; s_max = q - 3; }
      if (!isnan(emin) && (s_min < 0 || emin < ess_min_site)) { ess_min_site = emin; s_min = q - 3; }
    }
  }
  close_out(f, path);
  for (q = 0; q < 3; q++) constant += isnan(ess_min[q]);
  printf("diagnostics: R-hat -logL %.4f  c %.4f  d %.4f  sites max %.4f (site %d)  ESS -logL min %.1f  sites min %.1f (site %d)  "
         "constant %d\n", rhat[0], rhat[1], rhat[2], r_max, s_max, ess_min[0], ess_min_site, s_min, constant);
  free(stats); free(halves); free(rhat); free(n);
}

/* mean, 2.5 / 50 / 97.5 % quantiles, mode and P(mode) of one row of pooled counts */
struct marginal {
  double mean, p_mode;
  int32_t q[3], mode;
};
static void summarise(const int32_t *h, int32_t bins, struct marginal *out)
{
  static const double probs[3] = {0.025, 0.5, 0.975};
  int64_t total = 0, num = 0;
  int32_t j;
  out->mode = 0;
  for (j = 0; j < bins; j++) {
    total += h[j];
    num += (int64_t)j * h[j];
    if (h[j] > h[out->mode]) out->mode = j;
  }
  out->mean = (double)num / (double)total;
  out->p_mode = (double)h[out->mode] / (double)total;
  if (ser_hist_quantiles(h, 1, bins, probs, 3, out->q)) die("ser_hist_quantiles");
}

static int cmp_double(const void *x, const void *y)
{
  const double a = *(const double *)x, b = *(const double *)y;
  return a < b ? -1 : a > b;
}

/* median width q97.5 - q2.5 of n marginals (sorts w) */
static double median_width(const struct marginal *m, int32_t n, double *w)
{
  int32_t i;
  for (i = 0; i < n; i++) w[i] = m[i].q[2] - m[i].q[0];
  qsort(w, (size_t)n, sizeof(double), cmp_double);
  return n % 2 ? w[n / 2] : 0.5 * (w[n / 2 - 1] + w[n / 2]);
}

/* --taxon-pairs: the taxon pair relations of the chosen chains of `sub` pooled over the chains to PREFIX.<name>.csv as probability
 * matrices, and one summary line */
static void write_taxon_pairs(ser_run *sub, const int32_t *chosen, int32_t k, int32_t M, const char *prefix)
{
  static const char *names[4] = {"first", "last", "precedes", "coexist"};
  const size_t MM = (size_t)M * M;
  int32_t *tp[4], *n = xmalloc(sizeof(int32_t) * (size_t)k), tot = 0;
  long long hi = 0, lo = 0;
  char path[4096];
  int q, c;
  size_t j;
  FILE *f;
  for (q = 0; q < 4; q++) tp[q] = xmalloc(sizeof(int32_t) * k * MM);
  if (ser_run_taxon_pairs(sub, chosen, k, tp[0], tp[1], tp[2], tp[3], n)) die("ser_run_taxon_pairs");
  for (c = 0; c < k; c++) tot += n[c];
  for (q = 0; q < 4; q++) {
    snprintf(path, sizeof(path), "%s.%s.csv", prefix, names[q]);
    f = open_out(path);
    for (j = 0; j < MM; j++) {
      int64_t sum = 0;
      double p;
      for (c = 0; c < k; c++) sum += tp[q][c * MM + j];
      p = (double)sum / (double)tot;
      fprintf(f, "%.6f%c", p, (j + 1) % (size_t)M ? ',' : '\n');
      if (q == 3 && j / M < j % M) { hi += p >= 0.95; lo += p <= 0.05; }
    }
    close_out(f, path);
  }
  printf("taxon pairs: %d chains  %d samples  of %lld pairs of taxa %lld coexist with P >= 0.95 and %lld with P <= 0.05\n", k, tot,
         (long long)M * (M - 1) / 2, hi, lo);
  for (q = 0; q < 4; q++) free(tp[q]);
  free(n);
}

/* --cd-marginals: the error-rate marginals of the chosen chains of `sub` pooled over the chains (sums chain by chain in the order of
 * `chosen`) to `path`, and one summary line */
static void write_cd_marginals(ser_run *sub, const int32_t *chosen, int32_t k, int32_t R, const char *path)
{
  static const double probs[3] = {0.025, 0.5, 0.975};
  const double lo[2] = {SER_MINC, SER_MIND}, hi[2] = {SER_MAXC, SER_MAXD};
  const size_t RB = (size_t)R * SER_CD_BINS;
  double *sum[2], *mean[2], best[2] = {-1.0, -1.0};
  int32_t *hist[2], *q[2], *n = xmalloc(sizeof(int32_t) * (size_t)k), tot = 0, arg[2] = {0, 0}, h, c, r, i;
  size_t j;
  char name[2][32];
  FILE *f;
  for (h = 0; h < 2; h++) {
    sum[h] = xmalloc(sizeof(double) * (size_t)k * R);
    mean[h] = xmalloc(sizeof(double) * (size_t)R);
    hist[h] = xmalloc(sizeof(int32_t) * k * RB);
    q[h] = xmalloc(sizeof(int32_t) * (size_t)R * 3);
  }
  if (ser_run_cd_marginals(sub, chosen, k, sum[0], sum[1], hist[0], hist[1], n)) die("ser_run_cd_marginals");
  for (c = 0; c < k; c++) tot += n[c];
  for (h = 0; h < 2; h++) {
    for (r = 0; r < R; r++) {
      double s = 0.0;
      for (c = 0; c < k; c++) s += sum[h][(size_t)c * R + r];
      mean[h][r] = s / (double)tot;
      if (mean[h][r] > best[h]) { best[h] = mean[h][r]; arg[h] = r; }
    }
    for (c = 1; c < k; c++) /* pool the chains' counts into chain 0's slab */
      for (j = 0; j < RB; j++) hist[h][j] += hist[h][c * RB + j];
    if (ser_hist_quantiles(hist[h], R, SER_CD_BINS, probs, 3, q[h])) die("ser_hist_quantiles");
  }
  f = open_out(path);
  fprintf(f, "taxon,c_mean,c_q025,c_median,c_q975,d_mean,d_q025,d_median,d_q975\n");
  for (r = 0; r < R; r++) {
    if (R > 1) fprintf(f, "%d", r);
    else fprintf(f, "all");
    for (h = 0; h < 2; h++) {
      const double w = (hi[h] - lo[h]) / SER_CD_BINS;
      const int32_t *qr = q[h] + (size_t)r * 3;
      fprintf(f, ",%.6g,%.6g,%.6g,%.6g", mean[h][r], exp(lo[h] + qr[0] * w), exp(0.5 * ((lo[h] + qr[1] * w) + (lo[h] + (qr[1] + 1) * w))),
              exp(lo[h] + (qr[2] + 1) * w));
    }
    fprintf(f, "\n");
  }
  close_out(f, path);
  for (i = 0; i < 2; i++) {
    if (R > 1) snprintf(name[i], sizeof(name[i]), "taxon %d", arg[1 - i]);
    else snprintf(name[i], sizeof(name[i]), "all");
  }
  printf("cd marginals: %d chains  %d samples  highest mean d %.6g (%s)  highest mean c %.6g (%s)\n", k, tot, best[1], name[0], best[0],
         name[1]);
  for (h = 0; h < 2; h++) { free(sum[h]); free(mean[h]); free(hist[h]); free(q[h]); }
  free(n);
}

/* --marginals: the position and a / b histograms of the chosen chains of `sub` pooled over the chains to PREFIX.sites.csv and
 * PREFIX.taxa.csv, and one summary line */
static void write_marginals(ser_run *sub, const ser_dataset *ds, const int32_t *chosen, int32_t k, const char *prefix)
{
  int32_t N, M, nh, i, c, tot = 0;
  size_t j;
  char path[4096];
  FILE *f;
  ser_dataset_dims(ds, &N, &M, &nh);
  const size_t NN = (size_t)N * N, MB = (size_t)M * (N + 1);
  int32_t *pos = xmalloc(sizeof(int32_t) * k * NN), *ah = xmalloc(sizeof(int32_t) * k * MB), *bh = xmalloc(sizeof(int32_t) * k * MB);
  int32_t *n = xmalloc(sizeof(int32_t) * (size_t)k);
  double *w = xmalloc(sizeof(double) * (size_t)(N > M ? N : M));
  struct marginal *ms = xmalloc(sizeof(struct marginal) * (size_t)N);
  struct marginal *ma = xmalloc(sizeof(struct marginal) * (size_t)M), *mb = xmalloc(sizeof(struct marginal) * (size_t)M);
  uint8_t *hard = xmalloc((size_t)N);
  if (ser_run_marginals(sub, chosen, k, pos, ah, bh, n)) die("ser_run_marginals");
  for (c = 1; c < k; c++) { /* pool the chains' counts into chain 0's slabs */
    for (j = 0; j < NN; j++) pos[j] += pos[c * NN + j];
    for (j = 0; j < MB; j++) { ah[j] += ah[c * MB + j]; bh[j] += bh[c * MB + j]; }
  }
  for (c = 0; c < k; c++) tot += n[c];
  for (i = 0; i < N; i++) summarise(pos + (size_t)i * N, N, &ms[i]);
  for (i = 0; i < M; i++) { summarise(ah + (size_t)i * (N + 1), N + 1, &ma[i]); summarise(bh + (size_t)i * (N + 1), N + 1, &mb[i]); }
  ser_dataset_get(ds, NULL, hard);
  snprintf(path, sizeof(path), "%s.sites.csv", prefix);
  f = open_out(path);
  fprintf(f, "site,hard,mean,q025,median,q975,mode,p_mode\n");
  for (i = 0; i < N; i++)
    fprintf(f, "%d,%d,%.6f,%d,%d,%d,%d,%.6f\n", i, hard[i] != 0, ms[i].mean, ms[i].q[0], ms[i].q[1], ms[i].q[2], ms[i].mode, ms[i].p_mode);
  close_out(f, path);
  snprintf(path, sizeof(path), "%s.taxa.csv", prefix);
  f = open_out(path);
  fprintf(f, "taxon,a_mean,a_q025,a_median,a_q975,b_mean,b_q025,b_median,b_q975\n");
  for (i = 0; i < M; i++)
    fprintf(f, "%d,%.6f,%d,%d,%d,%.6f,%d,%d,%d\n", i, ma[i].mean, ma[i].q[0], ma[i].q[1], ma[i].q[2], mb[i].mean, mb[i].q[0], mb[i].q[1],
            mb[i].q[2]);
  close_out(f, path);
  printf("marginals: %d chains  %d samples  median width of the 95%% intervals: sites %.1f  a %.1f  b %.1f positions\n", k, tot,
         median_width(ms, N, w), median_width(ma, M, w), median_width(mb, M, w));
  free(pos); free(ah); free(bh); free(n); free(w); free(ms); free(ma); free(mb); free(hard);
}

/* --diversity: the diversity curves of the chosen chains of `sub` pooled over the chains to PREFIX.positions.csv and PREFIX.sites.csv,
 * and one summary line */
static void write_diversity(ser_run *sub, const ser_dataset *ds, const int32_t *chosen, int32_t k, const char *prefix)
{
  int32_t N, M, nh, i, c, q, tot = 0, peak = 0;
  size_t j;
  char path[4096];
  FILE *f;
  ser_dataset_dims(ds, &N, &M, &nh);
  const size_t cells = (size_t)N * (M + 1);
  int32_t *h[4], *n = xmalloc(sizeof(int32_t) * (size_t)k);
  struct marginal *m[4];
  uint8_t *hard = xmalloc((size_t)N);
  for (q = 0; q < 4; q++) {
    h[q] = xmalloc(sizeof(int32_t) * k * cells);
    m[q] = xmalloc(sizeof(struct marginal) * (size_t)N);
  }
  if (ser_run_diversity(sub, chosen, k, h[0], h[1], h[2], h[3], n)) die("ser_run_diversity");
  for (c = 0; c < k; c++) tot += n[c];
  for (q = 0; q < 4; q++) {
    for (c = 1; c < k; c++) /* pool the chains' counts into chain 0's slab */
      for (j = 0; j < cells; j++) h[q][j] += h[q][c * cells + j];
    for (i = 0; i < N; i++) summarise(h[q] + (size_t)i * (M + 1), M + 1, &m[q][i]);
  }
  snprintf(path, sizeof(path), "%s.positions.csv", prefix);
  f = open_out(path);
  fprintf(f, "position,rich_mean,rich_q025,rich_median,rich_q975,orig_mean,orig_q025,orig_median,orig_q975,ext_mean,ext_q025,ext_median,"
             "ext_q975\n");
  for (i = 0; i < N; i++) {
    fprintf(f, "%d", i);
    for (q = 0; q < 3; q++) fprintf(f, ",%.6f,%d,%d,%d", m[q][i].mean, m[q][i].q[0], m[q][i].q[1], m[q][i].q[2]);
    fprintf(f, "\n");
    if (m[0][i].mean > m[0][peak].mean) peak = i;
  }
  close_out(f, path);
  ser_dataset_get(ds, NULL, hard);
  snprintf(path, sizeof(path), "%s.sites.csv", prefix);
  f = open_out(path);
  fprintf(f, "site,hard,rich_mean,rich_q025,rich_median,rich_q975\n");
  for (i = 0; i < N; i++) fprintf(f, "%d,%d,%.6f,%d,%d,%d\n", i, hard[i] != 0, m[3][i].mean, m[3][i].q[0], m[3][i].q[1], m[3][i].q[2]);
  close_out(f, path);
  printf("diversity: %d chains  %d samples  peak mean richness %.6f taxa at position %d (95%% interval %d-%d)\n", k, tot, m[0][peak].mean,
         peak, m[0][peak].q[0], m[0][peak].q[2]);
  for (q = 0; q < 4; q++) { free(h[q]); free(m[q]); }
  free(n); free(hard);
}

/* The chosen chains re-simulated alone, once for every --select output: bit-identical to their first run, whose E[-logL] per global
 * id - first is e[] (any difference exits 1).  acc = 0 keeps every sample (SER_STORE_FULL, max_samples = samples), so every getter
 * reads the store; otherwise the SER_ACC_* parts in acc accumulate through a window of W samples, in SER_STORE_PI when acc is
 * SER_ACC_PO alone (pair order reads pi only) and SER_STORE_FULL else.  The caller destroys the run. */
static ser_run *replay_chosen(const ser_dataset *ds, const ser_run_config *cfg, const int32_t *chosen, int32_t k, const double *e, int first,
                              int burn, int samples, int window, int acc)
{
  ser_run_config c2 = *cfg;
  ser_run *sub = NULL;
  double *e2 = xmalloc(sizeof(double) * (size_t)k);
  int32_t ns = 0, i;
  c2.n_chains = k;
  c2.chain_offset = 0;
  c2.store = acc == SER_ACC_PO ? SER_STORE_PI : SER_STORE_FULL;
  c2.max_samples = acc ? window : samples;
  if (ser_run_create_chains(ds, &c2, chosen, k, &sub)) die("ser_run_create_chains");
  if (ser_run_init(sub)) die("ser_run_init");
  if (acc && ser_run_accumulate(sub, acc)) die("ser_run_accumulate");
  if (ser_run_advance_both(sub, burn, samples) || ser_run_sync(sub)) die("replay of the chosen chains");
  if (ser_run_chain_stats(sub, e2, NULL, NULL, &ns)) die("ser_run_chain_stats");
  for (i = 0; i < k; i++)
    if (memcmp(&e2[i], &e[chosen[i] - first], sizeof(double))) {
      fprintf(stderr, "mcmc: the replayed chain %d does not reproduce its first run (E[-logL] %.17g vs %.17g)\n", chosen[i], e2[i],
              e[chosen[i] - first]);
      exit(1);
    }
  free(e2);
  return sub;
}

static double *read_tape(const char *path, uint64_t *len)
{
  FILE *f = fopen(path, "rb");
  long sz;
  double *buf;
  if (!f) { fprintf(stderr, "mcmc: cannot open tape %s\n", path); exit(1); }
  fseek(f, 0, SEEK_END);
  sz = ftell(f);
  fseek(f, 0, SEEK_SET);
  buf = (double *)malloc((size_t)sz + 8);
  if (!buf || fread(buf, 1, (size_t)sz, f) != (size_t)sz) { fprintf(stderr, "mcmc: cannot read tape %s\n", path); exit(1); }
  fclose(f);
  *len = (uint64_t)sz / sizeof(double);
  return buf;
}

int main(int argc, char **argv)
{
  int n_chains = 1, first = 0, burn = 1000, samples = 1000, select_k = 0, device = 0, batch = 0, manycd = 0, gpus = 1, i;
  int replay_selected = 0, window = 64, resume = 0, ckpt_every = 0, stop_after = -1;
  int64_t done = 0, total;
  unsigned long seed = 0;
  const char *dataset = NULL, *chains_dir = "Chains", *po_path = NULL, *tape_path = getenv("SER_TAPE_IN"), *ckpt_path = NULL;
  const char *diag_path = NULL, *marg_prefix = NULL, *rdiag_path = NULL, *pairs_prefix = NULL, *cd_path = NULL, *div_prefix = NULL;
  const char *env_seed = getenv("GSL_RNG_SEED");
  ser_dataset *ds = NULL;
  ser_run *run = NULL;   /* single-chain replay */
  ser_multi *multi = NULL; /* everything else: the chains of the call over `gpus` devices */
  ser_run_config cfg;
  int32_t N, M, nh, bad = 0, devs[8];

  if (env_seed) {
    seed = strtoul(env_seed, NULL, 0);
    fprintf(stderr, "GSL_RNG_SEED=%lu\n", seed);
  }
  if (argc == 1) usage(argv[0]);
  if (argv[1][0] == '-' && argv[1][1] == '-') {
    batch = 1;
    for (i = 1; i < argc; i++) {
      const char *a = argv[i], *v = (i + 1 < argc) ? argv[i + 1] : NULL;
      if (!strcmp(a, "--replay-selected")) { replay_selected = 1; continue; }
      if (!strcmp(a, "--resume")) { resume = 1; continue; }
      if (!v) usage(argv[0]);
      if (!strcmp(a, "--chains")) n_chains = atoi(v);
      else if (!strcmp(a, "--gpus")) gpus = atoi(v);
      else if (!strcmp(a, "--first")) first = atoi(v);
      else if (!strcmp(a, "--burn")) burn = atoi(v);
      else if (!strcmp(a, "--samples")) samples = atoi(v);
      else if (!strcmp(a, "--seed")) seed = strtoul(v, NULL, 0);
      else if (!strcmp(a, "--dataset")) dataset = v;
      else if (!strcmp(a, "--chains-dir")) chains_dir = v;
      else if (!strcmp(a, "--select")) select_k = atoi(v);
      else if (!strcmp(a, "--po")) po_path = v;
      else if (!strcmp(a, "--device")) device = atoi(v);
      else if (!strcmp(a, "--manycd")) manycd = atoi(v) != 0;
      else if (!strcmp(a, "--window")) window = atoi(v);
      else if (!strcmp(a, "--checkpoint")) ckpt_path = v;
      else if (!strcmp(a, "--diagnostics")) diag_path = v;
      else if (!strcmp(a, "--rank-diagnostics")) rdiag_path = v;
      else if (!strcmp(a, "--marginals")) marg_prefix = v;
      else if (!strcmp(a, "--taxon-pairs")) pairs_prefix = v;
      else if (!strcmp(a, "--cd-marginals")) cd_path = v;
      else if (!strcmp(a, "--diversity")) div_prefix = v;
      else if (!strcmp(a, "--checkpoint-every")) { if ((ckpt_every = atoi(v)) < 1) usage(argv[0]); }
      else if (!strcmp(a, "--stop-after")) { if ((stop_after = atoi(v)) < 0) usage(argv[0]); }
      else usage(argv[0]);
      i++;
    }
    if (n_chains < 1 || burn < 0 || samples < 0 || gpus < 1 || gpus > 8 || n_chains < gpus) usage(argv[0]);
    if (replay_selected && (select_k < 1 || window < 1)) usage(argv[0]);
    if ((diag_path || rdiag_path) && select_k < 1) usage(argv[0]);
    if ((marg_prefix || pairs_prefix || cd_path || div_prefix) && (select_k < 1 || window < 1)) usage(argv[0]);
    if (!ckpt_path && (ckpt_every || stop_after >= 0 || resume)) usage(argv[0]); /* these act on the --checkpoint file */
  } else if (argc == 2) {
    char *end = NULL;
    const long idx = strtol(argv[1], &end, 10); /* mcmc.c:115,153 */
    if (end == argv[1] || *end || idx < 0 || idx > 99) {
      /* the reference builds "Chains/chain_XX" from two digits (mcmc.c:148-178); an index outside 0..99 has no
       * directory there -- refuse it up front instead of simulating 20 000 sweeps and writing nothing */
      fprintf(stderr, "mcmc: chain index '%s' must be an integer in 0..99 (Chains/chain_XX)\n", argv[1]);
      return 1;
    }
    first = (int)idx;
  } else if (argc == 4) {
    if (!(sscanf(argv[1], "%d", &manycd) == 1 && sscanf(argv[2], "%d", &burn) == 1 && burn >= 0 &&
          sscanf(argv[3], "%d", &samples) == 1 && samples >= 0))
      usage(argv[0]);
    manycd = manycd != 0; /* mcmc_readmodel tests it as a flag (mcmc.c:363) */
  } else {
    usage(argv[0]);
  }

  if (ser_dataset_read_txt(dataset, &ds)) { fprintf(stderr, "%s\n", ser_last_error()); return 1; } /* mcmc_readmodel's messages */
  ser_dataset_dims(ds, &N, &M, &nh);

  memset(&cfg, 0, sizeof(cfg));
  cfg.struct_size = (uint32_t)sizeof(cfg);
  cfg.n_chains = n_chains;
  cfg.chain_offset = first;
  cfg.sweeps_per_call = 10;
  cfg.mode = tape_path ? SER_MODE_REPLAY : SER_MODE_FREE;
  cfg.seed = (uint32_t)seed;
  cfg.store = replay_selected ? SER_STORE_NONE : (n_chains <= 100) ? SER_STORE_FULL : SER_STORE_PI;
  cfg.max_samples = samples;
  cfg.device = device;
  cfg.manycd = manycd;
  for (i = 0; i < 8; i++) devs[i] = device + i;

  if (tape_path && ckpt_path) { fprintf(stderr, "mcmc: --checkpoint drives the free-running batch mode, not SER_TAPE_IN\n"); return 1; }
  total = (int64_t)burn + samples;
  if (tape_path) { /* replay of one recorded chain (validation against the reference) */
    uint64_t offs[2] = {0, 0};
    double *tape;
    if (n_chains != 1 || gpus != 1) { fprintf(stderr, "mcmc: SER_TAPE_IN drives exactly one chain\n"); return 1; }
    if (ser_run_create(ds, &cfg, &run)) die("ser_run_create");
    tape = read_tape(tape_path, &offs[1]);
    if (ser_run_set_tapes(run, tape, offs)) die("ser_run_set_tapes");
    free(tape);
    if (ser_run_init(run)) die("ser_run_init");
    if (ser_run_advance_both(run, burn, samples)) die("sweeps"); /* mcmc.c:140-143, :180-185 */
    if (ser_run_sync(run)) die("ser_run_sync");
    if (ser_run_check(run, &bad)) { fprintf(stderr, "main: error. (%s)\n", ser_last_error()); return 1; } /* mcmc.c:199-204 */
  } else {
    struct stat sb;
    int64_t end;
    if (ser_multi_create(ds, &cfg, gpus, devs, &multi)) die("ser_multi_create");
    if (resume && stat(ckpt_path, &sb) == 0) {
      int32_t ns = 0;
      if (ser_checkpoint_info(ckpt_path, NULL, NULL, NULL, &done, &ns, NULL, NULL, NULL)) die("ser_checkpoint_info");
      if (done > total || ns != (done > burn ? done - burn : 0)) {
        fprintf(stderr, "mcmc: %s holds %lld calls and %d samples: not a point of the --burn %d --samples %d schedule\n", ckpt_path,
                (long long)done, ns, burn, samples);
        return 1;
      }
      if (ser_multi_load_checkpoint(multi, ckpt_path)) die("ser_multi_load_checkpoint");
    } else if (ser_multi_init(multi)) {
      die("ser_multi_init");
    }
    end = (stop_after >= 0 && done + stop_after < total) ? done + stop_after : total;
    while (done < end) { /* mcmc.c:140-143, :180-185, in segments of at most --checkpoint-every calls */
      const int64_t seg = (ckpt_every > 0 && end - done > ckpt_every) ? ckpt_every : end - done;
      const int64_t b = done < burn ? (seg < burn - done ? seg : burn - done) : 0;
      if (ser_multi_advance(multi, (int32_t)b, (int32_t)(seg - b))) die("sweeps");
      done += seg;
      if (ckpt_every > 0 && done < end && ser_multi_save_checkpoint(multi, ckpt_path)) die("ser_multi_save_checkpoint");
    }
    if (ckpt_path && ser_multi_save_checkpoint(multi, ckpt_path)) die("ser_multi_save_checkpoint");
    if (done < total) {
      printf("stopped after call %lld of %lld; %s holds every chain; run again with --checkpoint %s --resume to continue\n", (long long)done,
             (long long)total, ckpt_path, ckpt_path);
      ser_multi_destroy(multi);
      ser_dataset_free(ds);
      return 0;
    }
    if (ser_multi_sync(multi)) die("ser_multi_sync");
    if (ser_multi_check(multi, &bad)) { fprintf(stderr, "main: error. (%s)\n", ser_last_error()); return 1; }
  }

  /* Chains/chain_XX/ for the chains whose index has a two-digit directory */
  if (cfg.store == SER_STORE_FULL) {
    int skipped = 0;
    mkdir(chains_dir, 0777);
    for (i = 0; i < n_chains; i++) {
      char dir[1024];
      const int idx = first + i;
      ser_run *owner = run;
      int32_t local = i;
      if (idx < 0 || idx > 99) { skipped++; continue; } /* the reference's directory name has two digits (mcmc.c:148-178) */
      if (multi && ser_multi_locate(multi, idx, &owner, &local)) die("ser_multi_locate");
      snprintf(dir, sizeof(dir), "%s/chain_%02d", chains_dir, idx);
      if (mkdir(dir, 0777) && errno != EEXIST) { fprintf(stderr, "mcmc: cannot create %s\n", dir); return 1; }
      if (ser_write_chain_files(owner, local, dir)) die("ser_write_chain_files");
    }
    if (skipped) fprintf(stderr, "mcmc: %d chain(s) outside the index range 0..99 have no Chains/chain_XX directory and were not written\n", skipped);
  } else if (batch && !select_k) {
    fprintf(stderr, "mcmc: %d chains is more than the 100 the reference's file layout holds: no chain files are written; "
                    "use --select K [--po FILE] for the cross-chain summaries\n", n_chains);
  }

  if (batch && multi) {
    double *e = (double *)malloc(sizeof(double) * (size_t)n_chains), *ec = (double *)malloc(sizeof(double) * (size_t)n_chains);
    double *ed = (double *)malloc(sizeof(double) * (size_t)n_chains), ms = 0.0;
    int32_t ns = 0, peer = 0;
    if (!e || !ec || !ed) { fprintf(stderr, "mcmc: out of memory\n"); return 1; }
    if (ser_multi_chain_stats(multi, e, ec, ed, &ns)) die("ser_multi_chain_stats");
    ser_multi_elapsed_ms(multi, &ms, 0);
    ser_multi_layout(multi, NULL, NULL, &peer);
    printf("chains %d  gpus %d%s  sites %d  taxa %d  hard %d  sweeps/chain %d  gpu_ms %.1f  sweeps/s %.0f\n", n_chains, gpus,
           gpus > 1 ? (peer ? " (peer stores)" : " (nccl)") : "", N, M, nh, (burn + samples) * 10, ms,
           ms > 0 ? (double)n_chains * (burn + samples) * 10 / (ms * 1e-3) : 0.0);
    if (select_k > 0) {
      int32_t *chosen = (int32_t *)malloc(sizeof(int32_t) * (size_t)select_k), nchosen = 0;
      int32_t *counts = po_path ? (int32_t *)calloc((size_t)select_k * N * N, sizeof(int32_t)) : NULL;
      double mn, sd;
      if (!chosen || (po_path && !counts)) { fprintf(stderr, "mcmc: out of memory\n"); return 1; }
      if (!replay_selected) {
        /* E[-logL] -> selection -> pair-order counts in one step on the device(s) (script.py:70-99, :155-189) */
        if (ser_multi_cross_chain(multi, select_k, chosen, &nchosen, &mn, &sd, counts)) die("ser_multi_cross_chain");
      } else {
        /* selection on the host; the chosen chains' pair-order counts come from their replay below */
        if (ser_select_chains(e, n_chains, select_k, chosen, &nchosen, &mn, &sd)) die("ser_select_chains");
        for (i = 0; i < nchosen; i++) chosen[i] += first; /* index in e -> global id */
      }
      printf("selection: min E[-logL] %.6f  sigma %.6f  chosen", mn, sd);
      for (i = 0; i < nchosen; i++) printf(" %d", chosen[i]);
      printf("\n");
      if (nchosen > 0) {
        double sc = 0.0, sdd = 0.0;
        for (i = 0; i < nchosen; i++) { sc += ec[chosen[i] - first]; sdd += ed[chosen[i] - first]; }
        printf("E[c] %.6f  E[d] %.6f over the chosen chains\n", sc / nchosen, sdd / nchosen);
      }
      if (nchosen > 0 && (diag_path || rdiag_path || marg_prefix || pairs_prefix || cd_path || div_prefix || (replay_selected && po_path))) {
        /* one replay for every output: every sample kept for the diagnostics, else a window accumulating what the outputs read */
        const int acc = (diag_path || rdiag_path) ? 0
                        : (replay_selected && po_path ? SER_ACC_PO : 0) | (marg_prefix ? SER_ACC_POS | SER_ACC_RANGE : 0) |
                          (pairs_prefix ? SER_ACC_TAXA : 0) | (cd_path ? SER_ACC_CD : 0) | (div_prefix ? SER_ACC_DIV : 0);
        ser_run *sub = replay_chosen(ds, &cfg, chosen, nchosen, e, first, burn, samples, window, acc);
        if (replay_selected && po_path && ser_run_po_counts(sub, chosen, nchosen, counts)) die("ser_run_po_counts");
        if (rdiag_path) write_rank_diagnostics(sub, chosen, nchosen, N, rdiag_path);
        if (diag_path) write_diagnostics(sub, chosen, nchosen, N, diag_path);
        if (pairs_prefix) write_taxon_pairs(sub, chosen, nchosen, M, pairs_prefix);
        if (cd_path) write_cd_marginals(sub, chosen, nchosen, manycd ? M : 1, cd_path);
        if (marg_prefix) write_marginals(sub, ds, chosen, nchosen, marg_prefix);
        if (div_prefix) write_diversity(sub, ds, chosen, nchosen, div_prefix);
        ser_run_destroy(sub);
      }
      if (po_path && nchosen > 0) {
        double *po = (double *)malloc(sizeof(double) * (size_t)N * N);
        FILE *f;
        int r, c;
        if (!po) { fprintf(stderr, "mcmc: out of memory\n"); return 1; }
        if (ser_po_finalize(counts, nchosen, N, select_k, 1, po)) die("ser_po_finalize");
        if (!(f = fopen(po_path, "w"))) { fprintf(stderr, "mcmc: cannot open %s\n", po_path); return 1; }
        for (r = 0; r < N; r++)
          for (c = 0; c < N; c++) fprintf(f, "%.6f%c", po[(size_t)r * N + c], c + 1 < N ? ',' : '\n');
        fclose(f);
        free(po);
      }
      free(chosen); free(counts);
    }
    free(e); free(ec); free(ed);
  }
  ser_run_destroy(run);
  ser_multi_destroy(multi);
  ser_dataset_free(ds);
  return 0;
}
