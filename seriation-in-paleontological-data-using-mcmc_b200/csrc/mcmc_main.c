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
 *        [--checkpoint FILE [--checkpoint-every C] [--resume] [--stop-after C]] [--diagnostics FILE] [--marginals PREFIX]
 * --replay-selected (with --select) runs select-then-replay: the chains keep no sample history (SER_STORE_NONE, so no
 * Chains/ files), the K chosen chains are re-simulated alone on --device (ser_run_create_chains, bit-identical) while
 * their pair-order counts accumulate through a window of W samples (ser_run_accumulate, default 64): the same output
 * lines and po.csv as the one-shot step, with device memory for K chains' window instead of every chain's history.
 * --checkpoint FILE writes every chain's state to FILE at the end of the sweeps (ser_multi_save_checkpoint), and every C calls
 * with --checkpoint-every C (the advance runs in segments of at most C calls; splitting a launch changes no chain).  --resume
 * loads FILE when it exists in place of the random start and runs the calls of the --burn B --samples S schedule that are left
 * (it refuses a file that has advanced past B + S calls, or whose sample count is not max(0, calls - B)).  --stop-after C
 * advances at most C calls in this invocation, writes FILE and exits 0 with one line saying where it stopped, before any
 * summary or Chains/ file: a long run split into slices gives the same output as the run done in one piece.
 * --diagnostics FILE (with --select) re-simulates the chosen chains alone keeping every sample (SER_STORE_FULL, bit-identical to
 * their first run, which is checked), writes per-quantity split-R-hat and effective sample sizes to FILE and prints one summary
 * line; under --replay-selected --po the same run supplies the pair-order counts.
 * --marginals PREFIX (with --select) re-simulates the chosen chains alone through a window of W samples (--window, default 64) while
 * their position and a / b histograms accumulate (bit-identical to their first run, which is checked), pools the counts over the
 * chains and writes PREFIX.sites.csv "site,hard,mean,q025,median,q975,mode,p_mode" (file order, 0-based positions) and
 * PREFIX.taxa.csv "taxon,a_mean,a_q025,a_median,a_q975,b_mean,b_q025,b_median,b_q975", and prints one summary line; under
 * --replay-selected --po (without --diagnostics) the same run supplies the pair-order counts, so the chains are replayed once.
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
          "              [--marginals PREFIX]   (with --select: position and a / b credible intervals of the chosen chains to\n"
          "                                      PREFIX.sites.csv and PREFIX.taxa.csv; the replay uses --window W)\n",
          argv0, argv0, argv0);
  exit(1);
}

/* --diagnostics: the chosen chains re-simulated alone with every sample kept (bit-identical to their first run, whose E[-logL]
 * per global id - first is e[]; any difference exits 1), their split-R-hat and ESS written to `path` as CSV and summarised in one
 * line.  `counts` (NULL: not wanted) receives their pair-order counts from the same run. */
static void replay_diagnostics(const ser_dataset *ds, const ser_run_config *cfg, const int32_t *chosen, int32_t k, const double *e, int first,
                               int burn, int samples, int32_t *counts, const char *path)
{
  ser_run_config c2 = *cfg;
  ser_run *sub = NULL;
  int32_t N, M, nh, ns = 0, i, q, c;
  double *e2, *stats, *halves, *rhat;
  int32_t *n;
  FILE *f;
  int s_max = -1, s_min = -1, constant = 0;
  double r_max = NAN, ess_min_site = NAN, ess_min[3];
  ser_dataset_dims(ds, &N, &M, &nh);
  const int Q = 3 + N;
  c2.n_chains = k;
  c2.chain_offset = 0;
  c2.store = SER_STORE_FULL;
  c2.max_samples = samples;
  e2 = (double *)malloc(sizeof(double) * (size_t)k);
  stats = (double *)malloc(sizeof(double) * (size_t)k * Q * 4);
  halves = (double *)malloc(sizeof(double) * (size_t)k * Q * 4);
  rhat = (double *)malloc(sizeof(double) * (size_t)Q);
  n = (int32_t *)malloc(sizeof(int32_t) * (size_t)k);
  if (!e2 || !stats || !halves || !rhat || !n) { fprintf(stderr, "mcmc: out of memory\n"); exit(1); }
  if (ser_run_create_chains(ds, &c2, chosen, k, &sub)) die("ser_run_create_chains");
  if (ser_run_init(sub) || ser_run_advance_both(sub, burn, samples) || ser_run_sync(sub)) die("replay of the chosen chains");
  if (ser_run_chain_stats(sub, e2, NULL, NULL, &ns)) die("ser_run_chain_stats");
  for (i = 0; i < k; i++)
    if (memcmp(&e2[i], &e[chosen[i] - first], sizeof(double))) {
      fprintf(stderr, "mcmc: the replayed chain %d does not reproduce its first run (E[-logL] %.17g vs %.17g)\n", chosen[i], e2[i],
              e[chosen[i] - first]);
      exit(1);
    }
  if (counts && ser_run_po_counts(sub, chosen, k, counts)) die("ser_run_po_counts");
  if (ser_run_diagnostics(sub, chosen, k, SER_DIAG_SCALARS | SER_DIAG_SITES, 0, stats, halves, n)) die("ser_run_diagnostics");
  if (ser_split_rhat(halves, n, k, Q, rhat)) die("ser_split_rhat");
  ser_run_destroy(sub);
  if (!(f = fopen(path, "w"))) { fprintf(stderr, "mcmc: cannot open %s\n", path); exit(1); }
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
    if (q < 3) fprintf(f, "%s,", q == 0 ? "-logL" : q == 1 ? "c" : "d");
    else fprintf(f, "site_%d,", q - 3);
    fprintf(f, "%.17g,%.17g,%.17g,%.17g\n", mean, rhat[q], emin, esum);
    if (q < 3) ess_min[q] = emin;
    else {
      if (isnan(emin)) constant++; /* constant in every chosen chain */
      if (!isnan(rhat[q]) && (s_max < 0 || rhat[q] > r_max)) { r_max = rhat[q]; s_max = q - 3; }
      if (!isnan(emin) && (s_min < 0 || emin < ess_min_site)) { ess_min_site = emin; s_min = q - 3; }
    }
  }
  if (fclose(f)) { fprintf(stderr, "mcmc: cannot write %s\n", path); exit(1); }
  for (q = 0; q < 3; q++) constant += isnan(ess_min[q]);
  printf("diagnostics: R-hat -logL %.4f  c %.4f  d %.4f  sites max %.4f (site %d)  ESS -logL min %.1f  sites min %.1f (site %d)  "
         "constant %d\n", rhat[0], rhat[1], rhat[2], r_max, s_max, ess_min[0], ess_min_site, s_min, constant);
  free(e2); free(stats); free(halves); free(rhat); free(n);
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

/* --marginals: the chosen chains re-simulated alone through a window of W samples while their position and a / b histograms accumulate
 * (bit-identical to their first run, whose E[-logL] per global id - first is e[]; any difference exits 1), the counts pooled over the
 * chains, PREFIX.sites.csv and PREFIX.taxa.csv written and one summary line printed.  `counts` (NULL: not wanted) receives their
 * pair-order counts from the same run. */
static void replay_marginals(const ser_dataset *ds, const ser_run_config *cfg, const int32_t *chosen, int32_t k, const double *e, int first,
                             int burn, int samples, int window, int32_t *counts, const char *prefix)
{
  ser_run_config c2 = *cfg;
  ser_run *sub = NULL;
  int32_t N, M, nh, ns = 0, i, c, tot = 0;
  size_t j;
  char path[4096];
  FILE *f;
  ser_dataset_dims(ds, &N, &M, &nh);
  const size_t NN = (size_t)N * N, MB = (size_t)M * (N + 1);
  int32_t *pos = (int32_t *)malloc(sizeof(int32_t) * k * NN), *ah = (int32_t *)malloc(sizeof(int32_t) * k * MB);
  int32_t *bh = (int32_t *)malloc(sizeof(int32_t) * k * MB), *n = (int32_t *)malloc(sizeof(int32_t) * (size_t)k);
  double *e2 = (double *)malloc(sizeof(double) * (size_t)k), *w = (double *)malloc(sizeof(double) * (size_t)(N > M ? N : M));
  struct marginal *ms = (struct marginal *)malloc(sizeof(struct marginal) * (size_t)N);
  struct marginal *ma = (struct marginal *)malloc(sizeof(struct marginal) * (size_t)M), *mb = (struct marginal *)malloc(sizeof(struct marginal) * (size_t)M);
  uint8_t *hard = (uint8_t *)malloc((size_t)N);
  if (!pos || !ah || !bh || !n || !e2 || !w || !ms || !ma || !mb || !hard) { fprintf(stderr, "mcmc: out of memory\n"); exit(1); }
  c2.n_chains = k;
  c2.chain_offset = 0;
  c2.store = SER_STORE_FULL;
  c2.max_samples = window;
  if (ser_run_create_chains(ds, &c2, chosen, k, &sub)) die("ser_run_create_chains");
  if (ser_run_init(sub) || ser_run_accumulate(sub, SER_ACC_POS | SER_ACC_RANGE | (counts ? SER_ACC_PO : 0))) die("ser_run_accumulate");
  if (ser_run_advance_both(sub, burn, samples) || ser_run_sync(sub)) die("replay of the chosen chains");
  if (ser_run_chain_stats(sub, e2, NULL, NULL, &ns)) die("ser_run_chain_stats");
  for (i = 0; i < k; i++)
    if (memcmp(&e2[i], &e[chosen[i] - first], sizeof(double))) {
      fprintf(stderr, "mcmc: the replayed chain %d does not reproduce its first run (E[-logL] %.17g vs %.17g)\n", chosen[i], e2[i],
              e[chosen[i] - first]);
      exit(1);
    }
  if (counts && ser_run_po_counts(sub, chosen, k, counts)) die("ser_run_po_counts");
  if (ser_run_marginals(sub, chosen, k, pos, ah, bh, n)) die("ser_run_marginals");
  ser_run_destroy(sub);
  for (c = 1; c < k; c++) { /* pool the chains' counts into chain 0's slabs */
    for (j = 0; j < NN; j++) pos[j] += pos[c * NN + j];
    for (j = 0; j < MB; j++) { ah[j] += ah[c * MB + j]; bh[j] += bh[c * MB + j]; }
  }
  for (c = 0; c < k; c++) tot += n[c];
  for (i = 0; i < N; i++) summarise(pos + (size_t)i * N, N, &ms[i]);
  for (i = 0; i < M; i++) { summarise(ah + (size_t)i * (N + 1), N + 1, &ma[i]); summarise(bh + (size_t)i * (N + 1), N + 1, &mb[i]); }
  ser_dataset_get(ds, NULL, hard);
  snprintf(path, sizeof(path), "%s.sites.csv", prefix);
  if (!(f = fopen(path, "w"))) { fprintf(stderr, "mcmc: cannot open %s\n", path); exit(1); }
  fprintf(f, "site,hard,mean,q025,median,q975,mode,p_mode\n");
  for (i = 0; i < N; i++)
    fprintf(f, "%d,%d,%.6f,%d,%d,%d,%d,%.6f\n", i, hard[i] != 0, ms[i].mean, ms[i].q[0], ms[i].q[1], ms[i].q[2], ms[i].mode, ms[i].p_mode);
  if (fclose(f)) { fprintf(stderr, "mcmc: cannot write %s\n", path); exit(1); }
  snprintf(path, sizeof(path), "%s.taxa.csv", prefix);
  if (!(f = fopen(path, "w"))) { fprintf(stderr, "mcmc: cannot open %s\n", path); exit(1); }
  fprintf(f, "taxon,a_mean,a_q025,a_median,a_q975,b_mean,b_q025,b_median,b_q975\n");
  for (i = 0; i < M; i++)
    fprintf(f, "%d,%.6f,%d,%d,%d,%.6f,%d,%d,%d\n", i, ma[i].mean, ma[i].q[0], ma[i].q[1], ma[i].q[2], mb[i].mean, mb[i].q[0], mb[i].q[1],
            mb[i].q[2]);
  if (fclose(f)) { fprintf(stderr, "mcmc: cannot write %s\n", path); exit(1); }
  printf("marginals: %d chains  %d samples  median width of the 95%% intervals: sites %.1f  a %.1f  b %.1f positions\n", k, tot,
         median_width(ms, N, w), median_width(ma, M, w), median_width(mb, M, w));
  free(pos); free(ah); free(bh); free(n); free(e2); free(w); free(ms); free(ma); free(mb); free(hard);
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
  const char *diag_path = NULL, *marg_prefix = NULL;
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
      else if (!strcmp(a, "--marginals")) marg_prefix = v;
      else if (!strcmp(a, "--checkpoint-every")) { if ((ckpt_every = atoi(v)) < 1) usage(argv[0]); }
      else if (!strcmp(a, "--stop-after")) { if ((stop_after = atoi(v)) < 0) usage(argv[0]); }
      else usage(argv[0]);
      i++;
    }
    if (n_chains < 1 || burn < 0 || samples < 0 || gpus < 1 || gpus > 8 || n_chains < gpus) usage(argv[0]);
    if (replay_selected && (select_k < 1 || window < 1)) usage(argv[0]);
    if (diag_path && select_k < 1) usage(argv[0]);
    if (marg_prefix && (select_k < 1 || window < 1)) usage(argv[0]);
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
        /* selection on the host, then the chosen chains again, alone, with the pair-order counts accumulating */
        if (ser_select_chains(e, n_chains, select_k, chosen, &nchosen, &mn, &sd)) die("ser_select_chains");
        for (i = 0; i < nchosen; i++) chosen[i] += first; /* index in e -> global id */
        if (counts && nchosen > 0 && !diag_path && !marg_prefix) {
          ser_run_config c2 = cfg;
          ser_run *sub = NULL;
          c2.n_chains = nchosen;
          c2.chain_offset = 0;
          c2.store = SER_STORE_PI;
          c2.max_samples = window;
          if (ser_run_create_chains(ds, &c2, chosen, nchosen, &sub)) die("ser_run_create_chains");
          if (ser_run_init(sub) || ser_run_accumulate(sub, SER_ACC_PO)) die("ser_run_accumulate");
          if (ser_run_advance_both(sub, burn, samples) || ser_run_po_counts(sub, chosen, nchosen, counts)) die("replay of the chosen chains");
          ser_run_destroy(sub);
        }
      }
      printf("selection: min E[-logL] %.6f  sigma %.6f  chosen", mn, sd);
      for (i = 0; i < nchosen; i++) printf(" %d", chosen[i]);
      printf("\n");
      if (nchosen > 0) {
        double sc = 0.0, sdd = 0.0;
        for (i = 0; i < nchosen; i++) { sc += ec[chosen[i] - first]; sdd += ed[chosen[i] - first]; }
        printf("E[c] %.6f  E[d] %.6f over the chosen chains\n", sc / nchosen, sdd / nchosen);
      }
      if (diag_path && nchosen > 0)
        replay_diagnostics(ds, &cfg, chosen, nchosen, e, first, burn, samples, replay_selected ? counts : NULL, diag_path);
      if (marg_prefix && nchosen > 0)
        replay_marginals(ds, &cfg, chosen, nchosen, e, first, burn, samples, window, (replay_selected && !diag_path) ? counts : NULL,
                         marg_prefix);
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
