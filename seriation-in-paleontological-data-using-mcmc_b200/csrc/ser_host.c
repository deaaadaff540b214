/*
 * ser_host.c -- host side of the C ABI that needs no CUDA: dataset readers (.txt / .genus /
 * .sites), the synthetic-matrix generator, host chain selection, pair-order finalisation and
 * the reference-compatible Chains/chain_XX/ writers.
 *
 * Reference behaviour restated (file:line under /root/reference):
 *   ser_dataset_read_stream   mcmc_readmodel            C_Implementation/mcmc.c:339-401
 *   ser_select_chains         choose_chains             script.py:70-99
 *   ser_po_finalize           compute_pair_order_matrix script.py:155-175
 *   ser_write_chain_files     mcmc_save_chain / print_exp_data / mcmc_save
 *                                                       mcmc.c:69-92, :60-67, :261-294
 */
#define _GNU_SOURCE
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "ser_internal.h"

static __thread char g_err[512] = "";

void ser_set_error(const char *fmt, ...)
{
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char *ser_last_error(void) { return g_err; }
const char *ser_version(void) { return "seriation_b200 0.1 (sm_100a)"; }

/* ------------------------------------------------------------------ datasets */
static ser_dataset *ds_alloc(int32_t N, int32_t M)
{
  ser_dataset *ds = (ser_dataset *)calloc(1, sizeof(*ds));
  if (!ds) return NULL;
  ds->N = N; ds->M = M;
  ds->X = (uint8_t *)calloc((size_t)N * M, 1);
  ds->hard = (uint8_t *)calloc((size_t)N, 1);
  if (!ds->X || !ds->hard) { free(ds->X); free(ds->hard); free(ds); return NULL; }
  return ds;
}

int ser_dataset_from_bits(int32_t N, int32_t M, const uint8_t *X, const uint8_t *hard, ser_dataset **out)
{
  if (!X || !out || N <= 0 || M <= 0) { ser_set_error("ser_dataset_from_bits: bad argument"); return SER_E_ARG; }
  ser_dataset *ds = ds_alloc(N, M);
  if (!ds) { ser_set_error("out of memory"); return SER_E_ARG; }
  for (size_t i = 0; i < (size_t)N * M; i++) ds->X[i] = X[i] ? 1 : 0;
  for (int32_t n = 0; n < N; n++) { ds->hard[n] = (hard && hard[n]) ? 1 : 0; ds->nh += ds->hard[n]; }
  *out = ds;
  return SER_OK;
}

/* mcmc_readmodel's grammar: header "N M"; per row the first M '0'/'1' characters whatever
 * separates them (a short row leaves the rest 0, as the calloc'ed matrix does at mcmc.c:366);
 * a '*' anywhere after them marks a hard site.  Unlike the reference, lines are not cut at
 * MAXS = 2000 characters (mcmc.h:25), so wide matrices parse correctly. */
int ser_dataset_read_stream(FILE *f, ser_dataset **out)
{
  char *line = NULL;
  size_t cap = 0;
  int n, m;
  if (!f || !out) { ser_set_error("ser_dataset_read_stream: null argument"); return SER_E_ARG; }
  if (getline(&line, &cap, f) < 0) { free(line); ser_set_error("mcmc_readmodel: read error."); return SER_E_PARSE; }
  if (sscanf(line, "%d %d", &n, &m) != 2 || n <= 0 || m <= 0) {
    free(line);
    ser_set_error("mcmc_readmodel: read error at header.");
    return SER_E_PARSE;
  }
  ser_dataset *ds = ds_alloc(n, m);
  if (!ds) { free(line); ser_set_error("out of memory"); return SER_E_ARG; }
  for (int i = 0; i < n; i++) {
    if (getline(&line, &cap, f) < 0) {
      free(line); ser_dataset_free(ds);
      ser_set_error("mcmc_readmodel: read error.");
      return SER_E_PARSE;
    }
    const char *s = line;
    size_t k = 0;
    for (int j = 0; j < m; j++) {
      while (s[k] != '0' && s[k] != '1' && s[k] != '\0') k++;
      if (s[k] == '\0') break;
      ds->X[(size_t)i * m + j] = (uint8_t)(s[k] == '1');
      k++;
    }
    while (s[k] != '*' && s[k] != '\0') k++;
    if (s[k] == '*') { ds->hard[i] = 1; ds->nh++; }
  }
  free(line);
  *out = ds;
  return SER_OK;
}

int ser_dataset_read_txt(const char *path, ser_dataset **out)
{
  if (!path) return ser_dataset_read_stream(stdin, out);
  FILE *f = fopen(path, "r");
  if (!f) { ser_set_error("cannot open %s", path); return SER_E_IO; }
  int rc = ser_dataset_read_stream(f, out);
  fclose(f);
  return rc;
}

int ser_dataset_dims(const ser_dataset *ds, int32_t *N, int32_t *M, int32_t *nh)
{
  if (!ds) return SER_E_ARG;
  if (N) *N = ds->N;
  if (M) *M = ds->M;
  if (nh) *nh = ds->nh;
  return SER_OK;
}

int ser_dataset_get(const ser_dataset *ds, uint8_t *X, uint8_t *hard)
{
  if (!ds) return SER_E_ARG;
  if (X) memcpy(X, ds->X, (size_t)ds->N * ds->M);
  if (hard) memcpy(hard, ds->hard, (size_t)ds->N);
  return SER_OK;
}

static void free_names(char **v, int32_t n)
{
  if (!v) return;
  for (int32_t i = 0; i < n; i++) free(v[i]);
  free(v);
}

void ser_dataset_free(ser_dataset *ds)
{
  if (!ds) return;
  free(ds->X); free(ds->hard);
  free_names(ds->taxon_names, ds->M);
  free_names(ds->site_names, ds->N);
  free(ds->site_mn); free(ds->site_age); free(ds->site_star);
  free(ds);
}

static void rstrip(char *s)
{
  size_t n = strlen(s);
  while (n && (s[n - 1] == '\n' || s[n - 1] == '\r' || s[n - 1] == ' ' || s[n - 1] == '\t')) s[--n] = '\0';
}

/* .genus: one taxon name per line (trailing blank).  .sites: "Name [MN_unit,age_Ma]" and an
 * optional " *" for hard sites.  No reference code reads these files; the format is pinned by
 * Dataset/g*.genus / g*.sites themselves. */
int ser_dataset_read_names(ser_dataset *ds, const char *genus_path, const char *sites_path)
{
  char *line = NULL;
  size_t cap = 0;
  if (!ds) return SER_E_ARG;
  if (genus_path) {
    FILE *f = fopen(genus_path, "r");
    if (!f) { ser_set_error("cannot open %s", genus_path); return SER_E_IO; }
    char **names = (char **)calloc((size_t)ds->M, sizeof(char *));
    int32_t m = 0;
    while (getline(&line, &cap, f) >= 0) {
      rstrip(line);
      if (!*line) continue;
      if (m < ds->M) names[m] = strdup(line);
      m++;
    }
    fclose(f);
    if (m != ds->M) {
      free_names(names, ds->M); free(line);
      ser_set_error("%s: %d taxon names for M=%d", genus_path, m, ds->M);
      return SER_E_PARSE;
    }
    free_names(ds->taxon_names, ds->M);
    ds->taxon_names = names;
  }
  if (sites_path) {
    FILE *f = fopen(sites_path, "r");
    if (!f) { free(line); ser_set_error("cannot open %s", sites_path); return SER_E_IO; }
    char **names = (char **)calloc((size_t)ds->N, sizeof(char *));
    int32_t *mn = (int32_t *)calloc((size_t)ds->N, sizeof(int32_t));
    double *age = (double *)calloc((size_t)ds->N, sizeof(double));
    uint8_t *star = (uint8_t *)calloc((size_t)ds->N, 1);
    int32_t n = 0, bad = 0;
    while (getline(&line, &cap, f) >= 0) {
      rstrip(line);
      if (!*line) continue;
      if (n < ds->N) {
        char *br = strrchr(line, '[');
        int unit = 0;
        double a = 0.0;
        if (!br || sscanf(br, "[%d,%lf]", &unit, &a) != 2) bad = 1;
        else {
          char *close = strchr(br, ']');
          star[n] = (uint8_t)(close && strchr(close, '*') != NULL);
          *br = '\0';
          rstrip(line);
          names[n] = strdup(line);
          mn[n] = unit; age[n] = a;
        }
      }
      n++;
    }
    fclose(f);
    if (bad || n != ds->N) {
      free_names(names, ds->N); free(mn); free(age); free(star); free(line);
      ser_set_error("%s: %s (%d site lines for N=%d)", sites_path, bad ? "malformed line" : "count mismatch", n, ds->N);
      return SER_E_PARSE;
    }
    free_names(ds->site_names, ds->N); free(ds->site_mn); free(ds->site_age); free(ds->site_star);
    ds->site_names = names; ds->site_mn = mn; ds->site_age = age; ds->site_star = star;
  }
  free(line);
  return SER_OK;
}

const char *ser_dataset_taxon_name(const ser_dataset *ds, int32_t m)
{
  return (ds && ds->taxon_names && m >= 0 && m < ds->M) ? ds->taxon_names[m] : NULL;
}
const char *ser_dataset_site_name(const ser_dataset *ds, int32_t n)
{
  return (ds && ds->site_names && n >= 0 && n < ds->N) ? ds->site_names[n] : NULL;
}
int ser_dataset_site_age(const ser_dataset *ds, int32_t n, int32_t *mn_unit, double *age_ma, int32_t *hard)
{
  if (!ds || !ds->site_names || n < 0 || n >= ds->N) { ser_set_error("no site labels loaded"); return SER_E_STATE; }
  if (mn_unit) *mn_unit = ds->site_mn[n];
  if (age_ma) *age_ma = ds->site_age[n];
  if (hard) *hard = ds->site_star[n];
  return SER_OK;
}

/* SplitMix64 */
static uint64_t sm64(uint64_t *s)
{
  uint64_t z = (*s += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
static uint32_t sm_below(uint64_t *s, uint32_t n) { return (uint32_t)(((sm64(s) >> 32) * (uint64_t)n) >> 32); }
static double sm_unit(uint64_t *s) { return (double)(sm64(s) >> 11) * (1.0 / 9007199254740992.0); }

/* Synthetic occurrence matrix (SURVEY.md 8d config 5): truth order = identity; each taxon lives
 * on a span of l ~ U{lmin..lmax} sites, present w.p. 0.5 inside and 0.01 outside; all-zero rows
 * and columns get one forced presence; n_hard hard sites evenly spaced in truth order; the file
 * order is a shuffle that keeps the hard sites in their true relative order. */
int ser_dataset_synthetic(int32_t N, int32_t M, int32_t n_hard, uint64_t seed, ser_dataset **out)
{
  if (!out || N < 2 || M < 1 || n_hard < 0 || n_hard > N) { ser_set_error("ser_dataset_synthetic: bad argument"); return SER_E_ARG; }
  uint64_t st = seed ? seed : 0x5EB1A710ull;
  uint8_t *T = (uint8_t *)calloc((size_t)N * M, 1); /* truth order */
  uint8_t *th = (uint8_t *)calloc((size_t)N, 1);
  int32_t *order = (int32_t *)malloc((size_t)N * sizeof(int32_t));
  int32_t lmin = N / 64 > 2 ? N / 64 : 2, lmax = N / 4 > lmin ? N / 4 : lmin + 1;
  if (lmax > N) lmax = N;
  if (lmin > lmax) lmin = lmax;
  for (int32_t m = 0; m < M; m++) {
    const int32_t l = lmin + (int32_t)sm_below(&st, (uint32_t)(lmax - lmin + 1));
    const int32_t a = (int32_t)sm_below(&st, (uint32_t)(N - l + 1)), b = a + l;
    int any = 0;
    for (int32_t n = 0; n < N; n++) {
      const double pr = (n >= a && n < b) ? 0.5 : 0.01;
      const int v = sm_unit(&st) < pr;
      T[(size_t)n * M + m] = (uint8_t)v;
      any |= v;
    }
    if (!any) T[(size_t)(a + l / 2) * M + m] = 1;
  }
  for (int32_t n = 0; n < N; n++) {
    int any = 0;
    for (int32_t m = 0; m < M; m++) any |= T[(size_t)n * M + m];
    if (!any) T[(size_t)n * M + sm_below(&st, (uint32_t)M)] = 1;
  }
  for (int32_t k = 0; k < n_hard; k++) th[(int32_t)(((int64_t)(2 * k + 1) * N) / (2 * n_hard))] = 1;
  /* shuffle rows, then put the hard rows back into increasing truth order on their slots */
  for (int32_t n = 0; n < N; n++) order[n] = n;
  for (int32_t i = N - 1; i > 0; i--) {
    const int32_t j = (int32_t)sm_below(&st, (uint32_t)(i + 1));
    const int32_t t = order[i]; order[i] = order[j]; order[j] = t;
  }
  {
    int32_t next_hard = 0;
    for (int32_t slot = 0; slot < N; slot++) {
      if (!th[order[slot]]) continue;
      while (!th[next_hard]) next_hard++;
      order[slot] = next_hard++;
    }
  }
  ser_dataset *ds = ds_alloc(N, M);
  if (!ds) { free(T); free(th); free(order); ser_set_error("out of memory"); return SER_E_ARG; }
  for (int32_t slot = 0; slot < N; slot++) {
    memcpy(ds->X + (size_t)slot * M, T + (size_t)order[slot] * M, (size_t)M);
    ds->hard[slot] = th[order[slot]];
    ds->nh += ds->hard[slot];
  }
  free(T); free(th); free(order);
  *out = ds;
  return SER_OK;
}

/* ------------------------------------------------------------------ cross-chain (host) */
/* choose_chains, script.py:70-99: population std (np.std, ddof = 0) over ALL chains, strict
 * inequalities, the k smallest, ids ascending. */
int ser_select_chains(const double *e, int32_t n, int32_t k, int32_t *chosen, int32_t *n_chosen, double *min_out,
                      double *sigma_out)
{
  if (!e || !chosen || !n_chosen || n < 1 || k < 0) { ser_set_error("ser_select_chains: bad argument"); return SER_E_ARG; }
  double mn = e[0], mean = 0.0, var = 0.0;
  for (int32_t i = 0; i < n; i++) { if (e[i] < mn) mn = e[i]; mean += e[i]; }
  mean /= n;
  for (int32_t i = 0; i < n; i++) var += (e[i] - mean) * (e[i] - mean);
  const double sigma = sqrt(var / n);
  int32_t found = 0, last_i = -1;
  double last_v = -HUGE_VAL;
  for (int32_t r = 0; r < k; r++) {
    int32_t bi = -1;
    for (int32_t i = 0; i < n; i++) {
      if (!(e[i] > mn - sigma && e[i] < mn + sigma)) continue;
      if (e[i] < last_v || (e[i] == last_v && i <= last_i)) continue;
      if (bi < 0 || e[i] < e[bi]) bi = i;
    }
    if (bi < 0) break;
    chosen[found++] = bi;
    last_v = e[bi]; last_i = bi;
  }
  for (int32_t x = 1; x < found; x++) {
    const int32_t key = chosen[x];
    int32_t y = x - 1;
    while (y >= 0 && chosen[y] > key) { chosen[y + 1] = chosen[y]; y--; }
    chosen[y + 1] = key;
  }
  *n_chosen = found;
  if (min_out) *min_out = mn;
  if (sigma_out) *sigma_out = sigma;
  return SER_OK;
}

/* compute_pair_order_matrix, script.py:155-175.  counts[c] already holds the per-chain sums of
 * generate_po_matrix (:178-189).  faithful != 0 keeps the reference's carry-over: the per-chain
 * accumulator is not reset, so chain c starts from chain c-1's matrix already divided by 1000. */
int ser_po_finalize(const int32_t *counts, int32_t k, int32_t N, int32_t chains_selected, int32_t faithful, double *po)
{
  if (!counts || !po || k < 1 || N < 1 || chains_selected < 1) { ser_set_error("ser_po_finalize: bad argument"); return SER_E_ARG; }
  const size_t nn = (size_t)N * N;
  double *carry = (double *)calloc(nn, sizeof(double));
  if (!carry) { ser_set_error("out of memory"); return SER_E_ARG; }
  for (size_t i = 0; i < nn; i++) po[i] = 0.0;
  for (int32_t c = 0; c < k; c++) {
    const int32_t *cnt = counts + (size_t)c * nn;
    for (size_t i = 0; i < nn; i++) {
      const double acc = ((faithful ? carry[i] : 0.0) + (double)cnt[i]) / 1000;
      po[i] += acc;
      carry[i] = acc;
    }
  }
  for (size_t i = 0; i < nn; i++) po[i] /= chains_selected;
  free(carry);
  return SER_OK;
}

/* split-R-hat (BDA3 section 11.4) from the half-sequences ser_run_diagnostics reports: halves [k][Q][4] = mean1, var1, mean2, var2 */
/* inverse-CDF quantiles of integer histograms (ser_run_marginals' rows): the comparison is made in double, p * total against the
 * running count, as numpy's searchsorted(cumsum(h), p * total) makes it */
int ser_hist_quantiles(const int32_t *hist, int32_t rows, int32_t bins, const double *probs, int32_t n_probs, int32_t *out)
{
  if (!hist || !probs || !out || rows < 1 || bins < 1 || n_probs < 1) {
    ser_set_error("ser_hist_quantiles: bad argument (rows = %d, bins = %d, n_probs = %d)", rows, bins, n_probs);
    return SER_E_ARG;
  }
  for (int32_t q = 0; q < n_probs; q++)
    if (!(probs[q] > 0.0 && probs[q] <= 1.0)) { ser_set_error("ser_hist_quantiles: probability %g is not in (0, 1]", probs[q]); return SER_E_ARG; }
  for (int32_t r = 0; r < rows; r++) {
    const int32_t *h = hist + (size_t)r * bins;
    int64_t total = 0;
    for (int32_t j = 0; j < bins; j++) total += h[j];
    for (int32_t q = 0; q < n_probs; q++) {
      int32_t b = -1;
      if (total > 0) {
        const double target = probs[q] * (double)total;
        int64_t cum = 0;
        for (b = 0; b < bins - 1; b++) {
          cum += h[b];
          if ((double)cum >= target) break;
        }
      }
      out[(size_t)r * n_probs + q] = b;
    }
  }
  return SER_OK;
}

int ser_split_rhat(const double *halves, const int32_t *n_samples, int32_t k, int32_t Q, double *rhat)
{
  if (!halves || !n_samples || !rhat || k < 1 || Q < 1) { ser_set_error("ser_split_rhat: bad argument (k = %d, Q = %d)", k, Q); return SER_E_ARG; }
  for (int32_t c = 1; c < k; c++)
    if (n_samples[c] != n_samples[0]) {
      ser_set_error("ser_split_rhat: the chains hold different numbers of samples (%d vs %d)", n_samples[0], n_samples[c]);
      return SER_E_ARG;
    }
  if (n_samples[0] < 4) { ser_set_error("ser_split_rhat: %d samples per chain (at least 4 are needed)", n_samples[0]); return SER_E_ARG; }
  const double n = (double)(n_samples[0] / 2), m = 2.0 * k;
  for (int32_t q = 0; q < Q; q++) {
    double W = 0.0, mean = 0.0, B = 0.0;
    for (int32_t c = 0; c < k; c++) {
      const double *h = halves + ((size_t)c * Q + q) * 4;
      W += h[1] + h[3];
      mean += h[0] + h[2];
    }
    W /= m;
    mean /= m;
    for (int32_t c = 0; c < k; c++) {
      const double *h = halves + ((size_t)c * Q + q) * 4;
      B += (h[0] - mean) * (h[0] - mean) + (h[2] - mean) * (h[2] - mean);
    }
    B /= m - 1.0; /* B / n */
    rhat[q] = W > 0.0 ? sqrt(((n - 1.0) / n * W + B) / W) : NAN;
  }
  return SER_OK;
}

/* ------------------------------------------------------------------ Chains/chain_XX writers */
int ser_write_chain_files(ser_run *run, int32_t chain, const char *dir)
{
  int32_t N, M, nh, nc, ns = 0;
  char path[1024];
  if (!run || !dir) { ser_set_error("ser_write_chain_files: null argument"); return SER_E_ARG; }
  ser_run_dims(run, &N, &M, &nh, &nc);
  int rc = ser_run_fetch_samples(run, chain, NULL, NULL, NULL, NULL, NULL, NULL, &ns);
  if (rc) return rc;
  int32_t *a = (int32_t *)malloc((size_t)(ns ? ns : 1) * M * 4), *b = (int32_t *)malloc((size_t)(ns ? ns : 1) * M * 4);
  int32_t *pi = (int32_t *)malloc((size_t)(ns ? ns : 1) * N * 4);
  double *c = (double *)malloc((size_t)(ns ? ns : 1) * 8), *d = (double *)malloc((size_t)(ns ? ns : 1) * 8);
  double *ll = (double *)malloc((size_t)(ns ? ns : 1) * 8);
  int32_t *fa = (int32_t *)malloc((size_t)M * 4), *fb = (int32_t *)malloc((size_t)M * 4), *fpi = (int32_t *)malloc((size_t)N * 4);
  double cdl[3], sums[3];
  /* manycd: per-taxon c, d of every sample and of the final state */
  const int many = ser_run_is_manycd(run);
  double *call = NULL, *dall = NULL, *fc = NULL, *fd = NULL;
  FILE *f = NULL;
  if (!a || !b || !pi || !c || !d || !ll || !fa || !fb || !fpi) { ser_set_error("ser_write_chain_files: out of memory"); rc = SER_E_ARG; goto done; }
  rc = ser_run_fetch_samples(run, chain, a, b, pi, c, d, ll, &ns);
  if (!rc && many) {
    call = (double *)malloc((size_t)(ns ? ns : 1) * M * 8); dall = (double *)malloc((size_t)(ns ? ns : 1) * M * 8);
    fc = (double *)malloc((size_t)M * 8); fd = (double *)malloc((size_t)M * 8);
    if (!call || !dall || !fc || !fd) { ser_set_error("ser_write_chain_files: out of memory"); rc = SER_E_ARG; goto done; }
    rc = ser_run_fetch_cd_samples(run, chain, call, dall, NULL);
    if (!rc) rc = ser_run_get_cd(run, chain, fc, fd);
  }
  if (!rc) rc = ser_run_get_state(run, chain, fa, fb, fpi, NULL, NULL, NULL, NULL, NULL, NULL, cdl, NULL);
  if (!rc) rc = ser_run_chain_sums(run, chain, sums, NULL);
  if (rc) goto done;

  /* chain_data.csv: one line per thinned sample (mcmc_save_chain, mcmc.c:69-92) */
  snprintf(path, sizeof(path), "%s/chain_data.csv", dir);
  if (!(f = fopen(path, "w"))) { ser_set_error("cannot open %s", path); rc = SER_E_IO; goto done; }
  for (int32_t s = 0; s < ns; s++) {
    const double ec = exp(c[s]), ed = exp(d[s]);
    for (int32_t i = 0; i < M; i++) fprintf(f, "%d ", a[(size_t)s * M + i]);
    fprintf(f, ",");
    for (int32_t i = 0; i < M; i++) fprintf(f, "%d ", b[(size_t)s * M + i]);
    fprintf(f, ",");
    for (int32_t i = 0; i < N; i++) fprintf(f, "%d ", pi[(size_t)s * N + i]);
    fprintf(f, ",");
    for (int32_t i = 0; i < M; i++) fprintf(f, "%.14f ", many ? exp(call[(size_t)s * M + i]) : ec);
    fprintf(f, ",");
    for (int32_t i = 0; i < M; i++) fprintf(f, "%.14f ", many ? exp(dall[(size_t)s * M + i]) : ed);
    fprintf(f, ",%.14f\n", ll[s]);
  }
  fclose(f);

  /* exp_data.csv: sums divided by the literal 1000 (print_exp_data, mcmc.c:60-67) */
  snprintf(path, sizeof(path), "%s/exp_data.csv", dir);
  if (!(f = fopen(path, "w"))) { ser_set_error("cannot open %s", path); rc = SER_E_IO; goto done; }
  fprintf(f, "exp_loglik,exp_c,exp_d\n");
  fprintf(f, "%.14f,%.14f,%.14f", sums[0] / 1000, sums[1] / 1000, sums[2] / 1000);
  fclose(f);

  /* taxa.csv / sites.csv / hard_sites.csv: final state (mcmc_save, mcmc.c:261-294) */
  snprintf(path, sizeof(path), "%s/taxa.csv", dir);
  if (!(f = fopen(path, "w"))) { ser_set_error("cannot open %s", path); rc = SER_E_IO; goto done; }
  fprintf(f, "a,b,c,d\n");
  for (int32_t i = 0; i < M; i++)
    fprintf(f, "%d,%d,%.14f,%.14f\n", fa[i], fb[i], exp(many ? fc[i] : cdl[0]), exp(many ? fd[i] : cdl[1]));
  fclose(f);
  snprintf(path, sizeof(path), "%s/sites.csv", dir);
  if (!(f = fopen(path, "w"))) { ser_set_error("cannot open %s", path); rc = SER_E_IO; goto done; }
  fprintf(f, "sites\n");
  for (int32_t i = 0; i < N; i++) fprintf(f, "%d\n", fpi[i]);
  fclose(f);
  snprintf(path, sizeof(path), "%s/hard_sites.csv", dir);
  if (!(f = fopen(path, "w"))) { ser_set_error("cannot open %s", path); rc = SER_E_IO; goto done; }
  fprintf(f, "i,pi_i\n");
  {
    const uint8_t *hard = ser_run_hard_flags(run);
    for (int32_t i = 0; i < N; i++) if (hard[i]) fprintf(f, "%d,%d\n", i, fpi[i]);
  }
  fclose(f);
done:
  free(a); free(b); free(pi); free(c); free(d); free(ll); free(fa); free(fb); free(fpi);
  free(call); free(dall); free(fc); free(fd);
  return rc;
}

/* labelled final state: names from the .genus / .sites files next to the sampler's a, b, pi */
int ser_write_labelled_files(ser_run *run, int32_t chain, const ser_dataset *ds, const char *dir)
{
  int32_t N, M, nh, nc;
  char path[1024];
  FILE *f;
  if (!run || !ds || !dir) { ser_set_error("ser_write_labelled_files: null argument"); return SER_E_ARG; }
  ser_run_dims(run, &N, &M, &nh, &nc);
  if (ds->N != N || ds->M != M) { ser_set_error("ser_write_labelled_files: dataset does not match the run"); return SER_E_ARG; }
  if (!ds->taxon_names || !ds->site_names) { ser_set_error("ser_write_labelled_files: no labels loaded (ser_dataset_read_names)"); return SER_E_STATE; }
  int32_t *a = (int32_t *)malloc((size_t)M * 4), *b = (int32_t *)malloc((size_t)M * 4), *pi = (int32_t *)malloc((size_t)N * 4);
  if (!a || !b || !pi) { free(a); free(b); free(pi); ser_set_error("ser_write_labelled_files: out of memory"); return SER_E_ARG; }
  int rc = ser_run_get_state(run, chain, a, b, pi, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL);
  if (!rc) {
    snprintf(path, sizeof(path), "%s/taxa_named.csv", dir);
    if (!(f = fopen(path, "w"))) { ser_set_error("cannot open %s", path); rc = SER_E_IO; }
    else {
      fprintf(f, "taxon,a,b\n");
      for (int32_t m = 0; m < M; m++) fprintf(f, "%s,%d,%d\n", ds->taxon_names[m], a[m], b[m]);
      fclose(f);
    }
  }
  if (!rc) {
    snprintf(path, sizeof(path), "%s/sites_named.csv", dir);
    if (!(f = fopen(path, "w"))) { ser_set_error("cannot open %s", path); rc = SER_E_IO; }
    else {
      fprintf(f, "site,mn_unit,age_ma,hard,pi\n");
      for (int32_t n = 0; n < N; n++)
        fprintf(f, "%s,%d,%g,%d,%d\n", ds->site_names[n], ds->site_mn[n], ds->site_age[n], (int)ds->hard[n], pi[n]);
      fclose(f);
    }
  }
  free(a); free(b); free(pi);
  return rc;
}

/* ------------------------------------------------------------------ CORR_MN against the .sites ages
 * Docs/Report.pdf Table 1 reports the correlation of the sampled site order with the MN chronology; the
 * reference's compute_exp_ages (script.py:129-152) uses the FILE order as a stand-in for it (the files list the
 * sites oldest first).  Here the .sites columns are used: the mean over the stored samples of
 * pearsonr(pi_t, x) for x = MN unit and x = -age.  pi_t is a permutation of 0..N-1 (mean (N-1)/2, variance
 * (N^2-1)/12), so the mean over samples follows exactly from sum_t pi_t(i), which the posterior kernel reduces
 * on the device:  mean_t r_t = sum_i (x_i - xbar) (pi_sum_i / T - (N-1)/2) / (N sd_pi sd_x). */
int ser_run_site_age_corr(ser_run *run, const ser_dataset *ds, const int32_t *chosen, int32_t k, double *corr_age, double *corr_mn,
                          int32_t *n_sites_used)
{
  int32_t N, M, nh, nc, T = 0;
  if (!run || !ds || !chosen || k < 1) { ser_set_error("ser_run_site_age_corr: bad argument"); return SER_E_ARG; }
  ser_run_dims(run, &N, &M, &nh, &nc);
  if (ds->N != N) { ser_set_error("ser_run_site_age_corr: dataset does not match the run"); return SER_E_ARG; }
  if (!ds->site_age || !ds->site_mn) { ser_set_error("ser_run_site_age_corr: no site ages loaded (ser_dataset_read_names with a .sites file)"); return SER_E_STATE; }
  for (int32_t n = 0; n < N; n++)
    if (!(ds->site_age[n] > 0.0)) { ser_set_error("ser_run_site_age_corr: site %d has no age", n); return SER_E_STATE; }
  int64_t *corr = (int64_t *)calloc((size_t)k, sizeof(int64_t));
  int32_t *pis = (int32_t *)calloc((size_t)k * N, sizeof(int32_t));
  if (!corr || !pis) { free(corr); free(pis); ser_set_error("ser_run_site_age_corr: out of memory"); return SER_E_ARG; }
  int rc = ser_run_posterior_sums(run, chosen, k, corr, pis, NULL, NULL, &T);
  if (!rc && T < 1) { ser_set_error("ser_run_site_age_corr: no stored samples"); rc = SER_E_STATE; }
  if (!rc) {
    double mean_age = 0.0, mean_mn = 0.0, var_age = 0.0, var_mn = 0.0, sum_age = 0.0, sum_mn = 0.0;
    const double mean_pi = ((double)N - 1.0) / 2.0, sd_pi = sqrt(((double)N * N - 1.0) / 12.0);
    int owned = 0;
    for (int32_t n = 0; n < N; n++) { mean_age += ds->site_age[n]; mean_mn += ds->site_mn[n]; }
    mean_age /= N; mean_mn /= N;
    for (int32_t n = 0; n < N; n++) {
      var_age += (ds->site_age[n] - mean_age) * (ds->site_age[n] - mean_age);
      var_mn += (ds->site_mn[n] - mean_mn) * (ds->site_mn[n] - mean_mn);
    }
    var_age /= N; var_mn /= N;
    for (int32_t c = 0; c < k; c++) {
      if (ser_run_local_chain(run, chosen[c]) < 0) continue; /* owned by another rank, or -1 */
      owned++;
      for (int32_t n = 0; n < N; n++) {
        const double dp = (double)pis[(size_t)c * N + n] / T - mean_pi;
        sum_age += (ds->site_age[n] - mean_age) * dp;
        sum_mn += (ds->site_mn[n] - mean_mn) * dp;
      }
    }
    if (!owned) { ser_set_error("ser_run_site_age_corr: none of the chosen chains lives on this run"); rc = SER_E_ARG; }
    else {
      if (corr_age) *corr_age = var_age > 0.0 ? -sum_age / owned / (N * sd_pi * sqrt(var_age)) : 0.0; /* older = earlier */
      if (corr_mn) *corr_mn = var_mn > 0.0 ? sum_mn / owned / (N * sd_pi * sqrt(var_mn)) : 0.0;
      if (n_sites_used) *n_sites_used = N;
    }
  }
  free(corr); free(pis);
  return rc;
}
